"""GPU parity of the cell + head (forward, loss, every parameter gradient) against the CPU oracle,
through the drop-in nn.Module surface (which calls the C-ABI).  Tolerance: 1e-5 normwise relative
in fp32 mode (BASELINE.json north_star)."""
import numpy as np
import pytest
import torch

from parity_util import W, build_cuda, is_dead, oracle_step, profiled, relerr, to_dev

pytestmark = pytest.mark.gpu
TOL = 1e-5


def _cases():
    c = []
    for adv in (False, True):
        c.append((W.tiny_workload("TemporalGCN", N=19, T=3, H=32, O=2, R=0, B=2, seed=21, adversarial=adv), 2))
        c.append((W.tiny_workload("RegionalTemporalGCN", N=23, T=4, H=32, O=3, R=3, B=2, seed=22, adversarial=adv), 2))
    c.append((W.tiny_workload("RegionalTemporalGCN", N=70, T=5, H=64, O=1, R=5, B=3, seed=23, k_intra=4), 3))
    c.append((W.tiny_workload("TemporalGCN", N=150, T=12, H=72, O=12, R=0, B=1, seed=24, k_intra=5), 1))
    c.append((W.make_workload(1), 1))      # TPIMS, reference defaults H=256 R=5
    c.append((W.make_workload(2), 2))      # METR-LA shape, sub-batch
    c.append((W.make_workload(3), 1))      # PEMS-BAY shape, H=256 R=12, sub-batch
    # fewer than 32 rows B*N*T, run at tf32x3 (_precision): the GEMM-by-GEMM cell of cell_g.cu with less than one TMA box
    # of rows, through the merged four-segment weight-gradient launch (H = 256) and the single-segment one (H = 32)
    c.append((W.tiny_workload("RegionalTemporalGCN", N=7, T=2, H=256, O=2, R=2, B=2, seed=25), 2))
    c.append((W.tiny_workload("TemporalGCN", N=5, T=3, H=32, O=2, R=0, B=2, seed=26), 2))
    return c


def _precision(w, B):
    return "tf32x3" if B * w.N * w.T < 32 else "fp32"


def _compare(w, B, cuda_out, cuda_hid, cuda_loss, cuda_grads, ref):
    assert relerr(cuda_hid, ref["hid"]) <= TOL, "out_hidden"
    assert relerr(cuda_out, ref["out"]) <= TOL, "out"
    if cuda_loss is not None:
        assert abs(float(cuda_loss) - ref["loss"]) <= TOL * abs(ref["loss"]), "loss"
    worst = 0.0
    for k, g in ref["grads"].items():
        if is_dead(w.model, k):
            assert cuda_grads.get(k) is None or float(cuda_grads[k].abs().max()) == 0.0, f"dead param {k} got a gradient"
            continue
        e = relerr(cuda_grads[k], g)
        worst = max(worst, e)
        assert e <= TOL, f"grad {k}: {e:.3e}"
    return worst


@pytest.mark.parametrize("w,B", _cases(), ids=lambda v: v.name if hasattr(v, "name") else str(v))
def test_autograd_path_matches_oracle(w, B):
    ref = oracle_step(w, B)
    prec = _precision(w, B)
    m = build_cuda(w, ref["state"], precision=prec)
    x, y = w.inputs(B)
    x, y = x.cuda(), y.cuda()
    out, hid = m(x, *to_dev(w.graph_args(), "cuda"))
    loss = ((out - y) ** 2).mean(dim=(1, 2)).sum()      # sum_b mean_b  (run.py:180 per snapshot)
    loss.backward()
    grads = {k: p.grad for k, p in m.named_parameters()}
    _compare(w, B, out, hid, loss, grads, ref)


@pytest.mark.parametrize("w,B", _cases()[:5] + _cases()[6:8] + _cases()[9:], ids=lambda v: v.name if hasattr(v, "name") else str(v))
def test_fused_step_matches_oracle(w, B):
    ref = oracle_step(w, B)
    prec = _precision(w, B)
    m = build_cuda(w, ref["state"], precision=prec)
    x, y = w.inputs(B)
    (loss, out, hid), names = profiled(lambda: m.fused_step(x.cuda(), y.cuda(), *to_dev(w.graph_args(), "cuda")))
    if prec == "tf32x3":
        for k in ("k_gemm_nt_tma_ts", "k_gemm_tn_tma"):
            assert k in names, (k, sorted(names))
    grads = {k: p.grad for k, p in m.named_parameters()}
    _compare(w, B, out, hid, loss, grads, ref)
    # a second call accumulates (run.py:190: grads accumulate over snapshots until optimizer.step)
    m.fused_step(x.cuda(), y.cuda(), *to_dev(w.graph_args(), "cuda"))
    for k, g in ref["grads"].items():
        if not is_dead(w.model, k):
            assert relerr(m.get_parameter(k).grad, 2 * g) <= TOL


def test_reference_single_snapshot_signature():
    """x [N,F,T] (no batch dim) with the 12 positional tensors of run.py:178."""
    w = W.make_workload(1)
    ref = oracle_step(w, 1)
    m = build_cuda(w, ref["state"])
    x, y = w.inputs(1)
    out, hid = m(x[0].cuda(), *to_dev(w.graph_args(), "cuda"))
    assert out.shape == (w.N, w.O) and hid.shape == (w.N, w.H)
    assert relerr(out, ref["out"][0]) <= TOL


def test_tgcn_cell_standalone():
    """models.utils.TGCN.forward(X, edge_index, edge_weight, H) incl. H=None and dL/dH."""
    from oracle import regt_oracle as O
    from models.utils import TGCN
    w = W.tiny_workload("TemporalGCN", N=40, T=1, H=32, O=1, R=0, B=1, seed=31, adversarial=True)
    torch.manual_seed(3)
    ref = O.TGCN(8, 32).double()
    W.init_params_synthetic(ref, 77)
    m = TGCN(8, 32)
    m.load_state_dict({k: v.float() for k, v in ref.state_dict().items()}, strict=True)
    m = m.cuda()
    X = torch.rand(w.N, 8, generator=torch.Generator().manual_seed(1))
    Hs = torch.rand(w.N, 32, generator=torch.Generator().manual_seed(2)) - 0.5
    for Hin in (None, Hs):
        Hd = None if Hin is None else Hin.double().requires_grad_()
        o_ref = ref(X.double(), w.edge_index, w.edge_attr.double(), Hd)
        Hc = None if Hin is None else Hin.cuda().requires_grad_()
        o = m(X.cuda(), w.edge_index.cuda(), w.edge_attr.cuda(), Hc)
        assert relerr(o, o_ref) <= TOL
        ref.zero_grad(); m.zero_grad()
        o_ref.square().sum().backward()
        o.square().sum().backward()
        for (k, p), (_, q) in zip(m.named_parameters(), ref.named_parameters()):
            assert relerr(p.grad, q.grad) <= TOL, k
        if Hin is not None:
            assert relerr(Hc.grad, Hd.grad) <= TOL


def test_bad_baseblock_raises_like_reference():
    from models.utils import TGCN
    with pytest.raises(NotImplementedError):
        TGCN(8, 16, baseblock="foo")


def test_batch_additivity_full_size_config2():
    """size-independent property at BASELINE config 2 full size (B=64): the batched fused step equals
    the sum of two half-batch steps (gradient accumulation is linear in the snapshots), and the
    forward is invariant to permuting the batch."""
    w = W.make_workload(2)
    ref_state = oracle_step(w, 1)["state"]
    x, y = w.inputs(w.B)
    x, y = x.cuda(), y.cuda()
    g = to_dev(w.graph_args(), "cuda")
    m1 = build_cuda(w, ref_state)
    l1, out1, _ = m1.fused_step(x, y, *g)
    m2 = build_cuda(w, ref_state)
    la, _, _ = m2.fused_step(x[:32].contiguous(), y[:32].contiguous(), *g)
    lb, _, _ = m2.fused_step(x[32:].contiguous(), y[32:].contiguous(), *g)
    assert abs(float(l1) - float(la) - float(lb)) <= 1e-5 * abs(float(l1))
    for (k, p), (_, q) in zip(m1.named_parameters(), m2.named_parameters()):
        if p.grad is not None:
            assert relerr(p.grad, q.grad) <= 2e-5, k
    perm = torch.randperm(w.B, generator=torch.Generator().manual_seed(0)).cuda()
    with torch.no_grad():
        out_p, _ = m1(x[perm].contiguous(), *g)
    assert torch.equal(out_p, out1[perm])


@pytest.mark.parametrize("precision,tol", [("fp32", 1e-5), ("tf32x3", 1e-5)])
def test_config1_matches_committed_golden(precision, tol):
    """BASELINE configs[0] (the reference's own CPU-runnable case: TPIMS graph, R=5, H=256) against the COMMITTED oracle
    vectors (tests/golden/cfg1_oracle_fp64.npz, made by make_cfg1_golden.py): no live oracle in the loop, so a drift of the
    oracle and of the kernels in the same direction cannot hide."""
    import os
    from parity_util import build_oracle
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cfg1_oracle_fp64.npz"))
    w = W.make_workload(1)
    state = build_oracle(w).state_dict()            # the seeded synthetic parameters the golden run used
    m = build_cuda(w, state, precision=precision)
    x, y = w.inputs(1)
    loss, out, hid = m.fused_step(x.cuda(), y.cuda(), *to_dev(w.graph_args(), "cuda"))
    assert relerr(out, torch.from_numpy(gold["out"])) <= tol
    assert relerr(hid, torch.from_numpy(gold["hid"])) <= tol
    assert abs(float(loss) - float(gold["loss"])) <= tol * abs(float(gold["loss"]))
    from parity_util import attention_limit, oracle_step
    att_lim, _ = attention_limit(w, 1, oracle_step(w, 1), tol)      # SURVEY 8(c): 1e-5 or within 4x of the fp32 twin
    for k, p in m.named_parameters():
        if is_dead(w.model, k) or ("gmax:" + k) not in gold:
            continue
        g = p.grad.double().reshape(-1).cpu()
        gmax = float(gold["gmax:" + k])
        lim = att_lim if k.endswith("_attention") else tol
        assert float((g[:32] - torch.from_numpy(gold["ghead:" + k])).abs().max()) <= lim * gmax, k
        assert float(g.abs().max()) <= (1.0 + 10 * lim) * gmax + 1e-30, k      # and nothing larger than the oracle's largest entry
