"""precision bf16 at hidden widths other than the fused cell's 64: the GEMM-by-GEMM cell of cell_g.cu on the single-pass
bf16 GEMMs of gemm_tma.cu (k_gemm_nt_bf16, k_gemm_tn_bf16), with the FFMA head kernels.

1. the GEMM test hooks against an fp64 matmul of the bf16-rounded operands (what the tensor core is asked to compute):
   ragged M / N / K tails, resident and streamed weights, the row contraction with several segments and the plane B2;
2. the models against the fp64 oracle at the stated bf16 bounds (2e-2 activations and loss, 5e-2 gradients, 0.15 for
   the period-attention gradient) at H = 128 and 256: RegionalTemporalGCN on a plain and on an adversarial multi-segment
   graph, TemporalGCN, models.utils.TGCN with H given (dH included), through autograd and through fused_step with
   micro-batches; config 1 against the committed fp64 vectors;
3. forward-only (no_grad) against the training forward, two runs, a NaN-poisoned workspace and a CUDA-graph replay: bit
   for bit;
4. a sum of region-shard steps against the full step.

Every model test asserts that the bf16 GEMMs ran and that neither the 3xTF32 GEMMs nor the fused bf16 cell did."""
import os

import numpy as np
import pytest
import torch

from parity_util import W, build_cuda, build_oracle, is_dead, oracle_step, profiled, relerr, to_dev
from test_gpu_step_edges import _grads, _run_on_workspace, _zero_grads

pytestmark = pytest.mark.gpu
ATOL, GTOL, ATT_TOL = 2e-2, 5e-2, 0.15       # stated bf16 tolerances against the oracle
BF16_GEMMS = ("k_pack_bf16", "k_gemm_nt_bf16", "k_gemm_tn_bf16")
FORBIDDEN = ("k_split_hilo", "k_gemm_nt_tma_ts", "k_gemm_tn_tma", "k_gemm_kt")


def _st():
    return torch.cuda.current_stream().cuda_stream


def _bf(t):
    return t.to(torch.bfloat16).double()


def _ran_bf16_gemms(names, backward=True):
    for k in (BF16_GEMMS if backward else BF16_GEMMS[:2]):
        assert k in names, (k, sorted(names))
    bad = [n for n in names if n in FORBIDDEN or (n.startswith("k_cell_") and n.endswith("_tc"))]
    assert not bad, f"other cell kernels ran: {bad}"


def _model_node(t):
    """the autograd node of the library's model function behind ``t`` (``t`` may be a view of its output, as
    ``models.utils.TGCN`` returns ``out[0]``)."""
    todo, seen = [t.grad_fn], set()
    while todo:
        node = todo.pop()
        if node is None or node in seen:
            continue
        if type(node).__name__.startswith("_ModelFn"):
            return node
        seen.add(node)
        todo.extend(f for f, _ in node.next_functions)
    raise AssertionError("no model node behind the tensor")


def _backward_names(node_of, loss):
    """``loss.backward()``; returns the names of the kernels the model node behind ``node_of`` launched.  Autograd runs
    that node on its own thread and the recorder is per thread, so hooks on the node switch it on and off there."""
    from regt_b200 import _lib
    lib = _lib.load()
    names = set()

    def pre(grad_outputs):
        lib.regt_profile(1, torch.cuda.current_stream().cuda_stream)

    def post(grad_inputs, grad_outputs):
        torch.cuda.synchronize()
        names.update(n for n, _ in _lib.profile_read())
        lib.regt_profile(0, None)

    node = _model_node(node_of)
    hooks = [node.register_prehook(pre), node.register_hook(post)]
    try:
        loss.backward()
        torch.cuda.synchronize()
    finally:
        for h in hooks:
            h.remove()
    return names


# ------------------------------------------------------------------------------------------------------------------
# 1. GEMM hooks
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,N,K,pad", [(128, 128, 64, 0), (300, 256, 128, 0), (1000, 64, 256, 8), (640, 512, 64, 4), (129, 16, 96, 0),
                                       (4096, 128, 136, 0), (50000, 128, 128, 0), (20011, 64, 64, 0), (30000, 256, 256, 0),
                                       (77, 512, 64, 4), (1, 128, 128, 0), (5000, 128, 384, 0), (3000, 128, 512, 0),
                                       (999, 96, 40, 4)])
def test_gemm_nt_bf16(M, N, K, pad):
    """resident weights (N <= 128, K <= 384), streamed weights, ragged M / N / K (a chunk whose second 32-wide box lies
    wholly past K is not loaded), many tiles per CTA, fewer rows than one 128-row tile."""
    from regt_b200 import _lib
    lib = _lib.load()
    g = torch.Generator().manual_seed(M + N + K)
    A = (torch.rand(M, K + pad, generator=g) - 0.5).cuda()
    Bt = (torch.rand(N, K + pad, generator=g) - 0.5).cuda()
    C = torch.full((M, N + pad), float("nan"), device="cuda")
    scratch = torch.empty(2 * ((N + 127) // 128 * 128) * ((K + 31) // 32 * 32), device="cuda")   # the tf32 hook's size
    rc = lib.regt_debug_gemm_nt_bf16(A.data_ptr(), K + pad, Bt.data_ptr(), K + pad, C.data_ptr(), N + pad, M, N, K,
                                     scratch.data_ptr(), _st())
    _lib.check(rc, "regt_debug_gemm_nt_bf16")
    ref = _bf(A[:, :K]) @ _bf(Bt[:, :K]).t()
    assert relerr(C[:, :N], ref) <= 1e-5
    if pad:
        assert torch.isnan(C[:, N:]).all()


@pytest.mark.parametrize("M,K,N,splits", [(256, 128, 128, 1), (1000, 256, 64, 4), (5000, 512, 128, 7), (70, 64, 32, 3),
                                          (4097, 128, 288, 5), (777, 64, 0, 2), (40000, 128, 128, 37), (1000, 256, 128, 4),
                                          (3000, 128, 256, 3), (20, 64, 32, 1), (20000, 1024, 256, 10), (65, 96, 96, 1)])
def test_gemm_tn_bf16(M, K, N, splits):
    """the row contraction against B and, in the same pass, the 32-column plane B2; splits of 64-row chunks, many
    accumulator drains (40000 / 37 rows = 17 chunks per split), an M below one chunk (TMA zero-fills the box)."""
    from regt_b200 import _lib
    lib = _lib.load()
    g = torch.Generator().manual_seed(M + N + K)
    A = (torch.rand(M, K + 4, generator=g) - 0.5).cuda()
    B = (torch.rand(M, max(N, 4) + 8, generator=g) - 0.5).cuda()
    B2 = (torch.rand(M, 32, generator=g) - 0.5).cuda()
    Cp = torch.full((splits, K, max(N, 1)), float("nan"), device="cuda")
    Cp2 = torch.full((splits, K, 32), float("nan"), device="cuda")
    rc = lib.regt_debug_gemm_tn_bf16(A.data_ptr(), K + 4, B.data_ptr() if N else None, max(N, 4) + 8, Cp.data_ptr() if N else None, M,
                                     K, N, splits, B2.data_ptr(), 32, Cp2.data_ptr(), _st())
    _lib.check(rc, "regt_debug_gemm_tn_bf16")
    if N:
        assert relerr(Cp.double().sum(0), _bf(A[:, :K]).t() @ _bf(B[:, :N])) <= 1e-5
    assert relerr(Cp2.double().sum(0), _bf(A[:, :K]).t() @ _bf(B2)) <= 1e-5


@pytest.mark.parametrize("M,H,splits", [(3000, 128, 5), (20000, 256, 10), (40000, 128, 37), (20, 128, 1)])
def test_gemm_tn_bf16_multi_segment(M, H, splits):
    """the cell backward's single launch: D [M, 4H] against h (z | r blocks), h*R (h~ block) and the feature plane."""
    from regt_b200 import _lib
    lib = _lib.load()
    g = torch.Generator().manual_seed(M + H)
    D = (torch.rand(M, 4 * H, generator=g) - 0.5).cuda()
    h = (torch.rand(M, H, generator=g) - 0.5).cuda()
    hR = (torch.rand(M, H, generator=g) - 0.5).cuda()
    F = (torch.rand(M, 32, generator=g) - 0.5).cuda()
    C0 = torch.full((splits, 2 * H, H), float("nan"), device="cuda")
    C1 = torch.full((splits, H, H), float("nan"), device="cuda")
    C2 = torch.full((splits, 4 * H, 32), float("nan"), device="cuda")
    rc = lib.regt_debug_gemm_tn_multi_bf16(D.data_ptr(), 4 * H, M, H, h.data_ptr(), hR.data_ptr(), C0.data_ptr(), C1.data_ptr(),
                                           splits, F.data_ptr(), C2.data_ptr(), _st())
    _lib.check(rc, "regt_debug_gemm_tn_multi_bf16")
    Dd = _bf(D)
    assert relerr(C0.double().sum(0), Dd[:, :2 * H].t() @ _bf(h)) <= 1e-5
    assert relerr(C1.double().sum(0), Dd[:, 2 * H:3 * H].t() @ _bf(hR)) <= 1e-5
    assert relerr(C2.double().sum(0), Dd.t() @ _bf(F)) <= 1e-5


# ------------------------------------------------------------------------------------------------------------------
# 2. models against the oracle
# ------------------------------------------------------------------------------------------------------------------
def _check(w, ref, loss, out, hid, grads, tag):
    errs = {"out_hidden": relerr(hid, ref["hid"])}
    if out is not None:
        errs["out"] = relerr(out, ref["out"])
    if loss is not None:
        errs["loss"] = abs(float(loss) - ref["loss"]) / abs(ref["loss"])
    for k, e in errs.items():
        assert e <= ATOL, f"{tag}: {k} {e:.3e} > {ATOL}"
    worst = 0.0
    for k, g in ref["grads"].items():
        if is_dead(w.model, k):
            continue
        if g is None:
            assert grads[k] is None or float(grads[k].abs().max()) == 0.0, f"{tag}: grad {k} should be zero"
            continue
        e = relerr(grads[k], g)
        bound = ATT_TOL if k.endswith("_attention") else GTOL
        assert e <= bound, f"{tag}: grad {k} {e:.3e} > {bound}"
        worst = max(worst, e) if not k.endswith("_attention") else worst
    print(f"{tag}: " + ", ".join(f"{k} {e:.2e}" for k, e in errs.items()) + f", worst grad {worst:.2e}")


_WORKLOADS = {
    "regional_h128": lambda: (W.tiny_workload("RegionalTemporalGCN", N=300, T=4, H=128, O=4, R=5, B=3, seed=61, k_intra=4), 3),
    # a node in two regional lists (two segments), self-loops, duplicates, an isolated node
    "regional_adv_h128": lambda: (W.tiny_workload("RegionalTemporalGCN", N=60, T=6, H=128, O=3, R=3, B=3, seed=62, adversarial=True), 3),
    "regional_h256": lambda: (W.tiny_workload("RegionalTemporalGCN", N=90, T=3, H=256, O=2, R=4, B=3, seed=63, k_intra=4), 3),
    "regional_adv_h256": lambda: (W.tiny_workload("RegionalTemporalGCN", N=40, T=3, H=256, O=2, R=3, B=3, seed=64, adversarial=True), 3),
    "a3tgcn_h128": lambda: (W.tiny_workload("TemporalGCN", N=200, T=5, H=128, O=6, R=0, B=3, seed=65, adversarial=True), 3),
    "a3tgcn_h256": lambda: (W.tiny_workload("TemporalGCN", N=150, T=4, H=256, O=3, R=0, B=3, seed=66), 3),
}
_ORACLES = {}


def _oracle(key):
    if key not in _ORACLES:
        w, B = _WORKLOADS[key]()
        _ORACLES[key] = (w, B, oracle_step(w, B))
    return _ORACLES[key]


@pytest.mark.parametrize("key", list(_WORKLOADS))
def test_autograd_matches_oracle(key):
    w, B, ref = _oracle(key)
    m = build_cuda(w, ref["state"], precision="bf16")
    x, y = w.inputs(B)
    x, y = x.cuda(), y.cuda()
    g = to_dev(w.graph_args(), "cuda")
    (out, hid), names = profiled(lambda: m(x, *g))
    _ran_bf16_gemms(names, backward=False)
    loss = ((out - y) ** 2).mean(dim=(1, 2)).sum()
    _ran_bf16_gemms(_backward_names(hid, loss) | names)
    _check(w, ref, loss, out, hid, {k: p.grad for k, p in m.named_parameters()}, f"{key}/autograd")


@pytest.mark.parametrize("mb", [None, 2], ids=["whole", "mb2"])
@pytest.mark.parametrize("key", list(_WORKLOADS))
def test_fused_step_matches_oracle(key, mb):
    """micro_batch 2 of B = 3: two steps of the kernels, the second ragged and accumulating into .grad and the loss."""
    w, B, ref = _oracle(key)
    m = build_cuda(w, ref["state"], precision="bf16")
    x, y = w.inputs(B)
    (loss, out, hid), names = profiled(lambda: m.fused_step(x.cuda(), y.cuda(), *to_dev(w.graph_args(), "cuda"), micro_batch=mb or B))
    _ran_bf16_gemms(names)
    _check(w, ref, loss, out, hid, _grads(m), f"{key}/fused mb={mb}")


@pytest.mark.parametrize("H", [128, 256])
def test_tgcn_cell_with_state_matches_oracle(H):
    """models.utils.TGCN(precision="bf16") with the state H given: H' and the gradients wrt the parameters and H."""
    from models.utils import TGCN
    from oracle import regt_oracle as O
    w = W.tiny_workload("TemporalGCN", N=300, T=1, H=H, O=1, R=0, B=1, seed=67, adversarial=True)
    gen = torch.Generator().manual_seed(7)
    X = torch.rand(w.N, 8, generator=gen)
    H0 = torch.rand(w.N, H, generator=gen) - 0.5
    c = torch.rand(w.N, H, generator=gen) - 0.5
    torch.manual_seed(0)
    om = O.TGCN(8, H).double()
    W.init_params_synthetic(om, 1234)
    Hr = H0.double().requires_grad_(True)
    ref_out = om(X.double(), w.edge_index, w.edge_attr.double(), Hr)
    (c.double() * ref_out).sum().backward()
    m = TGCN(8, H, precision="bf16")
    m.load_state_dict({k: v.float() for k, v in om.state_dict().items()}, strict=True)
    m = m.cuda()
    Hd = H0.cuda().requires_grad_(True)

    out, names = profiled(lambda: m(X.cuda(), w.edge_index.cuda(), w.edge_attr.cuda(), Hd))
    _ran_bf16_gemms(_backward_names(out, (c.cuda() * out).sum()) | names)
    out = out.detach()
    assert relerr(out, ref_out) <= ATOL, relerr(out, ref_out)
    pairs = [(p.grad, q.grad, k) for (k, p), (_, q) in zip(m.named_parameters(), om.named_parameters())] + [(Hd.grad, Hr.grad, "H")]
    for got, want, k in pairs:
        assert got.shape == want.shape and relerr(got, want) <= GTOL, f"grad {k} {relerr(got, want):.3e}"


def test_config1_matches_committed_golden():
    """BASELINE configs[0] (TPIMS graph, R = 5, H = 256, the reference's width) in bf16 against the committed fp64 vectors."""
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cfg1_oracle_fp64.npz"))
    w = W.make_workload(1)
    m = build_cuda(w, build_oracle(w).state_dict(), precision="bf16")
    x, y = w.inputs(1)
    (loss, out, hid), names = profiled(lambda: m.fused_step(x.cuda(), y.cuda(), *to_dev(w.graph_args(), "cuda")))
    _ran_bf16_gemms(names)
    assert relerr(out, torch.from_numpy(gold["out"])) <= ATOL
    assert relerr(hid, torch.from_numpy(gold["hid"])) <= ATOL
    assert abs(float(loss) - float(gold["loss"])) <= ATOL * abs(float(gold["loss"]))
    for k, p in m.named_parameters():
        if is_dead(w.model, k) or ("gmax:" + k) not in gold:
            continue
        gr = p.grad.double().reshape(-1).cpu()
        gmax = float(gold["gmax:" + k])
        lim = ATT_TOL if k.endswith("_attention") else GTOL
        assert float((gr[:32] - torch.from_numpy(gold["ghead:" + k])).abs().max()) <= lim * gmax, k
        assert float(gr.abs().max()) <= (1.0 + lim) * gmax + 1e-30, k


# ------------------------------------------------------------------------------------------------------------------
# 3. forward-only mode and reproducibility
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("key", ["regional_adv_h128", "a3tgcn_h256"])
def test_forward_only_equals_training_forward(key):
    w, B = _WORKLOADS[key]()
    m = build_cuda(w, build_oracle(w).state_dict(), precision="bf16")
    x, _ = w.inputs(B)
    x = x.cuda()
    g = to_dev(w.graph_args(), "cuda")
    out, hid = m(x, *g)
    assert out.requires_grad
    with torch.no_grad():
        (out0, hid0), names = profiled(lambda: m(x, *g))
    _ran_bf16_gemms(names, backward=False)
    assert torch.equal(out0, out.detach()) and torch.equal(hid0, hid.detach())


@pytest.mark.parametrize("path", ["fused", "autograd", "inference"])
@pytest.mark.parametrize("key", ["regional_adv_h128", "a3tgcn_h256"])
def test_two_runs_and_poisoned_workspace_are_bit_identical(key, path, monkeypatch):
    """the same step on a NaN-filled workspace and, twice, on a zeroed one: finite and bit-identical outputs and
    gradients (no kernel reads a byte it did not write first; nothing depends on timing)."""
    monkeypatch.delenv("REGT_UNFUSED", raising=False)
    w, B = _WORKLOADS[key]()
    runs = [_run_on_workspace(w, B, "bf16", path, poison) for poison in (True, False, False)]
    _ran_bf16_gemms(runs[0][2], backward=path != "inference")
    (l0, o0, h0), g0, _ = runs[0]
    assert torch.isfinite(o0).all() and torch.isfinite(h0).all()
    for (l1, o1, h1), g1, _ in runs[1:]:
        assert torch.equal(o0, o1) and torch.equal(h0, h1)
        assert (l0 is None) == (l1 is None) and (l0 is None or torch.equal(l0, l1))
        for k, t in g0.items():
            assert (t is None) == (g1[k] is None) and (t is None or torch.equal(t, g1[k])), k


def test_graph_replay_equals_eager():
    """fused_step(micro_batch=2) captured in a CUDA graph as bench.py runs it: a replay equals an eager step bit for bit."""
    w, B = _WORKLOADS["regional_h256"]()
    m = build_cuda(w, build_oracle(w).state_dict(), precision="bf16")
    x, y = w.inputs(B)
    xs, ys = x.cuda(), y.cuda()
    g = to_dev(w.graph_args(), "cuda")

    def step():
        return m.fused_step(xs, ys, *g, micro_batch=2)
    _, names = profiled(step)
    _ran_bf16_gemms(names)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        _zero_grads(m)
        step()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        res = step()
    _zero_grads(m)
    eager = [t.clone() for t in step()]
    ge = {k: v.clone() for k, v in _grads(m).items() if v is not None}
    _zero_grads(m)
    graph.replay()
    torch.cuda.synchronize()
    for a, b in zip(res, eager):
        assert torch.equal(a, b)
    for k, v in _grads(m).items():
        if v is not None:
            assert torch.equal(v, ge[k]), k


# ------------------------------------------------------------------------------------------------------------------
# 4. region shards
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [2, 3])
def test_sum_of_region_shards_matches_full_step(world):
    """each rank's step over its owned rows and halo (x_rows > N) on the bf16 GEMMs; outputs scattered back, losses and
    gradients summed, against the unsharded bf16 step: the same per-row arithmetic, cross-row sums in another order."""
    from regt_b200 import shard as S
    w = W.tiny_workload("RegionalTemporalGCN", N=300, T=4, H=128, O=3, R=5, B=2, seed=68, k_intra=4, n_cross=30)
    B = 2
    state = build_oracle(w).state_dict()
    x, y = w.inputs(B)
    x, y = x.cuda(), y.cuda()
    full = build_cuda(w, state, precision="bf16")
    (loss_f, out_f, hid_f), names = profiled(lambda: full.fused_step(x, y, *to_dev(w.graph_args(), "cuda")))
    _ran_bf16_gemms(names)
    ei, reis, reas = w.edge_index.cuda(), [e.cuda() for e in w.reg_edge_index], [a.cuda() for a in w.reg_edge_attr]
    loss_sum, grad_sum = 0.0, {}
    out_s = torch.zeros(B, w.N, w.O, device="cuda")
    hid_s = torch.zeros(B, w.N, w.H, device="cuda")
    halo = 0
    for rank in range(world):
        m = build_cuda(w, state, precision="bf16")
        sm = S.RegionShardedModel(m, ei, reis, reas, rank, world)
        halo += sm.shard.n_halo
        (loss, out, hid), names = profiled(lambda: sm.fused_step(x, y, sync=False))
        _ran_bf16_gemms(names)
        loss_sum += float(loss)
        S.scatter_rows(out, sm.own, out_s)
        S.scatter_rows(hid, sm.own, hid_s)
        for k, p in m.named_parameters():
            if p.grad is not None:
                grad_sum[k] = p.grad.double().cpu() + grad_sum.get(k, 0.0)
    assert halo > 0
    assert relerr(out_s, out_f) <= 1e-4 and relerr(hid_s, hid_f) <= 1e-4
    assert abs(loss_sum - float(loss_f)) <= 1e-4 * abs(float(loss_f))
    for k, p in full.named_parameters():
        if is_dead(w.model, k) or p.grad is None:
            continue
        assert relerr(grad_sum[k], p.grad) <= 1e-4, f"grad {k}: {relerr(grad_sum[k], p.grad):.3e}"
