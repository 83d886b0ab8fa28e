"""The fused step's MAE and masked losses (``fused_step(loss=, null_value=)``) on every head kernel a fused step can run,
and the masked evaluation metrics.

For each head path (k_head_fwd, k_head_fused, the tf32x3 head's k_hf_mid, the bf16 k_head_tc; shapes from the route table)
x {mse, mae} x {no mask, ~20 % of the targets 0 with null_value=0.0, ~20 % NaN with null_value=nan}: loss, out and every
parameter gradient against the fp64 oracle (oracle/masked_loss.py) at the precision's bound -- 1e-5 for fp32 / tf32x3
(gradients: or 4x the fp32 twin's own error), DESIGN section 3's bf16 bounds -- and, on the fp32 paths, against the
autograd path with the same torch loss at 1e-5.  Then the edges: a mask that finds nothing missing gives the unmasked step
bit for bit; an all-missing snapshot adds 0 and no NaN; micro-batches and region shards add up to the whole step; a
CUDA-graph replay and a NaN-poisoned workspace give the same bits; the epoch loop and evaluate() with a mask."""
import functools

import numpy as np
import pytest
import torch

from parity_util import W, build_cuda, build_oracle, is_dead, profiled, relerr, to_dev

pytestmark = pytest.mark.gpu
NAN = float("nan")
TOL, ATT_TOL = 1e-5, 1e-4
BF16_A, BF16_G, BF16_ATT, BF16_ATT_MAE = 2e-2, 5e-2, 0.15, 0.25

# path -> (workload, B, precision, head kernel); 3 * 150 rows: 128-row tiles and 64-row blocks span two snapshots
_PATHS = {
    "rows": (lambda: W.tiny_workload("RegionalTemporalGCN", N=150, T=3, H=128, O=12, R=4, B=3, seed=21), 3, "fp32", "k_head_fwd"),
    "fused_ffma": (lambda: W.tiny_workload("RegionalTemporalGCN", N=150, T=3, H=64, O=12, R=4, B=3, seed=22), 3, "fp32",
                   "k_head_fused"),
    # N * O % 4 == 0: a micro-batch's slice of y starts on 16 bytes
    "tf32x3": (lambda: W.tiny_workload("RegionalTemporalGCN", N=152, T=3, H=64, O=5, R=4, B=3, seed=23), 3, "tf32x3", "k_hf_mid"),
    # the bf16 edge tests' shape: 12 periods keep the attention gradient (a softmax-Jacobian difference) within its bound
    "bf16": (lambda: W.tiny_workload("TemporalGCN", N=150, T=12, H=64, O=12, R=0, B=3, seed=7, k_intra=5), 3, "bf16", "k_head_tc"),
}
_NULL = {"none": None, "zero": 0.0, "nan": NAN}


def _targets(y, mask, seed=5):
    y = y.clone()
    if mask != "none":
        drop = torch.rand(y.shape, generator=torch.Generator().manual_seed(seed)) < 0.2
        y[drop] = 0.0 if mask == "zero" else NAN
    return y


@functools.lru_cache(maxsize=None)
def _workload(path):
    return _PATHS[path][0]()


@functools.lru_cache(maxsize=None)
def _oracle(path, loss, mask):
    """fp64 masked step, per-gradient bounds from the fp32 twin, and the inputs."""
    from oracle.masked_loss import masked_batched_step
    w, B = _workload(path), _PATHS[path][1]
    x, y = w.inputs(B)
    y = _targets(y, mask)
    res = {}
    for dt in (torch.float64, torch.float32):
        m = build_oracle(w, dt)
        state = {k: v.clone() for k, v in m.state_dict().items()}
        o, h, l = masked_batched_step(m, x.to(dt), y.to(dt), w.graph_args(), loss, _NULL[mask])
        res[dt] = dict(out=o, hid=h, loss=l, grads={k: p.grad for k, p in m.named_parameters()}, state=state)
    ref, twin = res[torch.float64], res[torch.float32]
    lims = {k: max(TOL, 4.0 * relerr(twin["grads"][k], g)) for k, g in ref["grads"].items() if g is not None}
    return w, B, x, y, ref, lims


def _grads(m):
    return {k: (None if p.grad is None else p.grad.detach().clone()) for k, p in m.named_parameters()}


def _step(path, state, x, y, loss, null, **kw):
    w, prec = _workload(path), _PATHS[path][2]
    m = build_cuda(w, state, precision=prec)
    g = to_dev(w.graph_args(), "cuda")
    (l, out, hid), names = profiled(lambda: m.fused_step(x.cuda(), y.cuda(), *g, loss=loss, null_value=null, **kw))
    return m, (l, out, hid), _grads(m), names


@pytest.mark.parametrize("mask", list(_NULL))
@pytest.mark.parametrize("loss", ["mse", "mae"])
@pytest.mark.parametrize("path", list(_PATHS))
def test_head_path_matches_oracle(path, loss, mask):
    w, B, x, y, ref, lims = _oracle(path, loss, mask)
    prec, kern = _PATHS[path][2], _PATHS[path][3]
    m, (l, out, hid), grads, names = _step(path, ref["state"], x, y, loss, _NULL[mask])
    assert kern in names, (kern, sorted(names))
    assert ("k_loss_count" in names) == (mask != "none"), sorted(names)
    tag = f"{path}/{loss}/{mask}"
    assert np.isfinite(float(l)), tag
    a_tol = BF16_A if prec == "bf16" else TOL
    assert relerr(out, ref["out"]) <= a_tol, f"{tag}: out {relerr(out, ref['out']):.3e}"
    assert relerr(hid, ref["hid"]) <= a_tol, f"{tag}: out_hidden {relerr(hid, ref['hid']):.3e}"
    assert abs(float(l) - ref["loss"]) <= a_tol * abs(ref["loss"]), f"{tag}: loss {float(l)} vs {ref['loss']}"
    for k, g in ref["grads"].items():
        if is_dead(w.model, k) or g is None:
            continue
        assert torch.isfinite(grads[k]).all(), f"{tag}: grad {k} not finite"
        if prec == "bf16":
            # under the MAE an output within bf16's rounding of its target takes the other sign of the gradient than in
            # fp64; the period-attention gradient, a difference of nearly equal sums, shows that most (0.19 measured)
            bound = (BF16_ATT_MAE if loss == "mae" else BF16_ATT) if k.endswith("_attention") else BF16_G
        else:
            bound = max(lims[k], ATT_TOL) if (k.endswith("_attention") and prec == "tf32x3") else lims[k]
        e = relerr(grads[k], g)
        assert e <= bound, f"{tag}: grad {k} {e:.3e} > {bound:.3e}"
    if prec != "fp32":
        return
    # the autograd path with the same torch loss, on the same kernels' precision
    from oracle.masked_loss import masked_loss
    m2 = build_cuda(w, ref["state"], precision=prec)
    out2, _ = m2(x.cuda(), *to_dev(w.graph_args(), "cuda"))
    l2 = masked_loss(out2, y.cuda(), loss, _NULL[mask])
    l2.backward()
    l2 = l2.detach()
    assert abs(float(l) - float(l2)) <= TOL * abs(float(l2)), f"{tag}: loss vs autograd {float(l)} {float(l2)}"
    assert relerr(out, out2) <= TOL
    for k, p in m2.named_parameters():
        if p.grad is not None and not is_dead(w.model, k):
            assert relerr(grads[k], p.grad) <= TOL, f"{tag}: grad {k} vs autograd {relerr(grads[k], p.grad):.3e}"


@pytest.mark.parametrize("path", list(_PATHS))
def test_mask_without_missing_targets_is_the_unmasked_step_bit_for_bit(path):
    w, B = _workload(path), _PATHS[path][1]
    x, y = w.inputs(B)
    y = y.abs() + 0.5                                  # no target equals the null value
    state = build_oracle(w).state_dict()
    _, (l0, o0, h0), g0, _ = _step(path, state, x, y, "mse", None)
    _, (l1, o1, h1), g1, names = _step(path, state, x, y, "mse", 0.0)
    assert "k_loss_count" in names
    assert torch.equal(l0, l1) and torch.equal(o0, o1) and torch.equal(h0, h1), (float(l0), float(l1))
    for k in g0:
        assert (g0[k] is None and g1[k] is None) or torch.equal(g0[k], g1[k]), k


@pytest.mark.parametrize("loss", ["mse", "mae"])
@pytest.mark.parametrize("path", list(_PATHS))
def test_all_missing_snapshot_adds_nothing(path, loss):
    """snapshot 1 entirely missing (NaN and the null value mixed): the step equals the step of snapshots 0 and 2 alone."""
    w, B = _workload(path), _PATHS[path][1]
    x, y = w.inputs(B)
    y = _targets(y, "zero")
    y[1] = 0.0
    y[1, ::7] = NAN
    state = build_oracle(w).state_dict()
    _, (l, out, hid), g, _ = _step(path, state, x, y, loss, 0.0)
    keep = torch.tensor([0, 2])
    _, (lr, outr, _), gr, _ = _step(path, state, x[keep], y[keep], loss, 0.0)
    a_tol, g_tol = (BF16_A, BF16_G) if _PATHS[path][2] == "bf16" else (TOL, TOL)
    assert np.isfinite(float(l)) and torch.isfinite(out).all() and torch.isfinite(hid).all()
    assert abs(float(l) - float(lr)) <= a_tol * abs(float(lr)), (float(l), float(lr))
    assert relerr(out[keep], outr) <= a_tol
    for k in g:
        if g[k] is not None and not is_dead(w.model, k):
            assert torch.isfinite(g[k]).all(), k
            bound = (BF16_ATT if a_tol > TOL else ATT_TOL) if k.endswith("_attention") else g_tol
            assert relerr(g[k], gr[k]) <= bound, (k, relerr(g[k], gr[k]))


@pytest.mark.parametrize("path", ["tf32x3", "bf16"])
def test_micro_batches_add_up(path):
    """micro_batch=1 runs one step per snapshot with the library counting each one; the loss is the sum of the single
    snapshot steps exactly, and loss and gradients meet the whole-batch step."""
    w, B = _workload(path), _PATHS[path][1]
    x, y = w.inputs(B)
    y = _targets(y, "zero")
    state = build_oracle(w).state_dict()
    _, (lw, ow, _), gw, _ = _step(path, state, x, y, "mae", 0.0)
    _, (lm, om, _), gm, _ = _step(path, state, x, y, "mae", 0.0, micro_batch=1)
    singles = [_step(path, state, x[b:b + 1], y[b:b + 1], "mae", 0.0)[1][0] for b in range(B)]
    total = singles[0]
    for s in singles[1:]:
        total = total + s
    assert torch.equal(lm, total)
    tol = BF16_A if path == "bf16" else TOL
    assert abs(float(lm) - float(lw)) <= tol * abs(float(lw))
    assert relerr(om, ow) <= tol
    for k in gw:
        if gw[k] is not None and not is_dead(w.model, k):
            assert relerr(gm[k], gw[k]) <= (BF16_G if path == "bf16" else TOL), k


def test_region_shards_add_up_to_the_full_step():
    """two region shards run one after the other on one GPU: each divides by the FULL graph's valid counts (taken from
    the full y), so their losses and gradients add up to the unsharded step; a caller with local inputs only must pass
    the counts."""
    from regt_b200 import engine
    from regt_b200 import shard as S
    w = W.tiny_workload("RegionalTemporalGCN", N=300, T=3, H=64, O=5, R=6, B=3, seed=41)
    B = 3
    x, y = w.inputs(B)
    y = _targets(y, "zero")
    x, y = x.cuda(), y.cuda()
    state = build_oracle(w).state_dict()
    full = build_cuda(w, state, precision="tf32x3")
    lf, of, _ = full.fused_step(x, y, *to_dev(w.graph_args(), "cuda"), loss="mae", null_value=0.0)
    ei, reis, reas = w.edge_index.cuda(), [e.cuda() for e in w.reg_edge_index], [a.cuda() for a in w.reg_edge_attr]
    loss_sum, grad_sum = 0.0, {}
    out_full = torch.zeros(B, w.N, w.O, device="cuda")
    for rank in range(2):
        m = build_cuda(w, state, precision="tf32x3")
        sm = S.RegionShardedModel(m, ei, reis, reas, rank, 2)
        with pytest.raises(ValueError, match="loss_count"):
            sm.fused_step(None, None, local_inputs=sm.local_inputs(x, y), sync=False, loss="mae", null_value=0.0)
        lo, out, _ = sm.fused_step(x, y, sync=False, loss="mae", null_value=0.0)
        # the same step from local inputs and explicit counts
        m2 = build_cuda(w, state, precision="tf32x3")
        sm2 = S.RegionShardedModel(m2, ei, reis, reas, rank, 2)
        lo2, _, _ = sm2.fused_step(None, None, local_inputs=sm2.local_inputs(x, y), sync=False, loss="mae", null_value=0.0,
                                   loss_count=engine.loss_counts(y, 0.0))
        assert torch.equal(lo, lo2)
        loss_sum += float(lo)
        S.scatter_rows(out, sm.own, out_full)
        for k, p in m.named_parameters():
            if p.grad is not None:
                grad_sum[k] = p.grad.double() + grad_sum.get(k, 0.0)
    assert abs(loss_sum - float(lf)) <= TOL * abs(float(lf)), (loss_sum, float(lf))
    assert relerr(out_full, of) <= TOL
    for k, p in full.named_parameters():
        if p.grad is not None and not is_dead(w.model, k):
            assert relerr(grad_sum[k], p.grad) <= TOL, (k, relerr(grad_sum[k], p.grad))


@pytest.mark.parametrize("path", list(_PATHS))
def test_poisoned_workspace_and_graph_replay_give_the_same_bits(path):
    """the step on a workspace whose floats all start as NaN equals the step on a zeroed one, and a CUDA-graph replay of
    the masked step equals an eager step, bit for bit (the counts are rewritten by every step)."""
    w, B, prec = _workload(path), _PATHS[path][1], _PATHS[path][2]
    x, y = w.inputs(B)
    x, y = x.cuda(), _targets(y, "nan").cuda()
    g = to_dev(w.graph_args(), "cuda")
    state = build_oracle(w).state_dict()
    runs = []
    for poison in (True, False):
        m = build_cuda(w, state, precision=prec)
        m.fused_step(x, y, *g, loss="mae", null_value=NAN)        # sizes and creates the workspace
        ws = m._ws
        R = max(w.R, 1)
        tail = -(-4 * (R + 2) // 256) * 256                        # the int32 chunk table carved last (api.cu)
        ws.zero_()
        if poison:
            ws[:ws.numel() - tail].fill_(0xFF)
        for p in m.parameters():
            p.grad = None
        l, out, hid = m.fused_step(x, y, *g, loss="mae", null_value=NAN)
        runs.append((l, out, hid, _grads(m)))
    (a, b) = runs
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])
    for k in a[3]:
        assert (a[3][k] is None and b[3][k] is None) or torch.equal(a[3][k], b[3][k]), k
    # graph replay
    m = build_cuda(w, state, precision=prec)

    def step():
        return m.fused_step(x, y, *g, loss="mae", null_value=NAN)
    step()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    live = [p for p in m.parameters() if p.grad is not None]
    with torch.cuda.stream(s):
        for p in live:
            p.grad.zero_()
        step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    for p in live:
        p.grad.zero_()
    with torch.cuda.graph(graph):
        lg, og, _ = step()
    for p in live:
        p.grad.zero_()
    graph.replay()
    torch.cuda.synchronize()
    gg = _grads(m)
    assert torch.equal(lg, b[0]) and torch.equal(og, b[1])
    for k in gg:
        if b[3][k] is not None:
            assert torch.equal(gg[k], b[3][k]), k


def _series(N, F, T_total, seed, zero_frac=0.2):
    g = torch.Generator().manual_seed(seed)
    nd = torch.rand(N, F, T_total, generator=g)
    drop = torch.rand(N, T_total, generator=g) < zero_frac
    nd[:, -1][drop] = 0.0                                   # missing readings of the target feature
    return nd


def test_epoch_with_mask_matches_a_loop_of_autograd_steps():
    from oracle.masked_loss import masked_loss
    from regt_b200.loop import SlidingWindows, train_epoch
    w = W.tiny_workload("RegionalTemporalGCN", N=30, T=6, H=32, O=3, R=3, B=1, seed=11)
    nd = _series(w.N, 8, 6 + 3 + 8, 5)
    state = build_oracle(w).state_dict()
    gargs = to_dev(w.graph_args(), "cuda")
    m = build_cuda(w, state, precision="fp32")
    seen = {}

    class _Rec:   # the epoch's accumulated gradients at its one optimizer step
        def zero_grad(self):
            for p in m.parameters():
                p.grad = None

        def step(self):
            seen.update(_grads(m))
    sw = SlidingWindows(nd.cuda(), 6, 3)
    last, total = train_epoch(m, sw, gargs, _Rec(), batch=4, loss="mae", null_value=0.0)
    ref = build_cuda(w, state, precision="fp32")
    tot_ref, last_ref = 0.0, None
    for i in range(len(sw)):
        x, y = sw.gather(torch.tensor([i], device="cuda"))
        out, _ = ref(x[0], *gargs)
        lb = masked_loss(out, y[0], "mae", 0.0)
        lb.backward()
        tot_ref += float(lb)
        last_ref = float(lb)
    assert abs(float(last) - last_ref) <= TOL * abs(last_ref)
    assert abs(float(total) - tot_ref) <= TOL * abs(tot_ref)
    for k, p in ref.named_parameters():
        if p.grad is not None and not is_dead(w.model, k):
            assert relerr(seen[k], p.grad) <= TOL, k


def _np_metrics(outs, ys, null, q=95.0):
    n = s1 = s2 = 0.0
    mape_num = mape_den = 0.0
    for o, y in zip(outs, ys):
        v = ~np.isnan(y) & (y != null)
        if not v.any():
            continue
        e = (y - o)[v]
        n += v.sum()
        s1 += np.abs(e).astype(np.float64).sum()
        s2 += (e * e).astype(np.float64).sum()
        p = np.percentile(y[v], q)
        with np.errstate(divide="ignore"):
            r = np.abs(e / np.float32(p))
        if not np.isinf(r).any():
            mape_num += r.astype(np.float64).sum()
            mape_den += v.sum()
    return s1 / n, np.sqrt(s2 / n), mape_num / mape_den * 100


def test_evaluate_with_mask_matches_numpy():
    from regt_b200 import _lib
    from regt_b200.loop import SlidingWindows, evaluate, reduce_metrics
    w = W.tiny_workload("RegionalTemporalGCN", N=30, T=6, H=32, O=3, R=3, B=1, seed=11)
    nd = _series(w.N, 8, 6 + 3 + 8, 6)
    gargs = to_dev(w.graph_args(), "cuda")
    m = build_cuda(w, build_oracle(w).state_dict(), precision="fp32")
    sw = SlidingWindows(nd.cuda(), 6, 3)
    mae, rmse, mape = evaluate(m, sw, gargs, batch=4, null_value=0.0)
    with torch.no_grad():
        x, y = sw.gather(torch.arange(len(sw), device="cuda"))
        outs = m(x, *gargs)[0]
    rm = _np_metrics(list(outs.cpu().numpy()), list(y.cpu().numpy()), 0.0)
    for a, b in zip((mae, rmse, mape), rm):
        assert abs(a - b) <= 1e-5 * abs(b), (a, b)
    # the kernel itself: an all-missing snapshot drops out, NaNs are missing, the percentile runs over valid targets
    g = torch.Generator().manual_seed(3)
    yy = torch.rand(4, 50, 3, generator=g)
    oo = torch.rand(4, 50, 3, generator=g)
    yy[0, ::3] = 0.0
    yy[1] = 0.0
    yy[2, ::5] = NAN
    sums = torch.empty(4, 5, dtype=torch.float64, device="cuda")
    od, yd = oo.cuda(), yy.cuda()
    _lib.check(_lib.load().regt_eval_metrics_masked(od.data_ptr(), yd.data_ptr(), 4, 150, 95.0, 0.0, sums.data_ptr(),
                                                    torch.cuda.current_stream().cuda_stream), "masked")
    s = sums.cpu().numpy()
    for b in range(4):
        yb, ob = yy[b].numpy().ravel(), oo[b].numpy().ravel()
        v = ~np.isnan(yb) & (yb != 0.0)
        assert s[b, 0] == v.sum()
        if not v.any():
            assert s[b, 1] == 0 and s[b, 2] == 0 and np.isnan(s[b, 3])
            continue
        e = (yb - ob)[v]
        assert abs(s[b, 1] - np.abs(e).astype(np.float64).sum()) <= 1e-9 * s[b, 1]
        assert abs(s[b, 2] - (e * e).astype(np.float64).sum()) <= 1e-9 * s[b, 2]
        assert abs(s[b, 3] - np.percentile(yb[v], 95.0)) <= 1e-6 * abs(s[b, 3])
    r = reduce_metrics(sums.cpu(), 150)
    rr = _np_metrics(list(oo.numpy()), list(yy.numpy()), 0.0)
    for a, b in zip(r, rr):
        assert abs(a - b) <= 1e-5 * abs(b), (a, b)
