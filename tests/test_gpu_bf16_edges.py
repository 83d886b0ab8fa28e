"""The opt-in bf16 step (k_cell_fwd_tc / k_cell_bwd_tc of cell_tc.cu, k_head_tc of head_tc.cu, the bf16 branches of
head.cu) at the shapes where its work split changes, each against the fp64 oracle of the same batch:

1. config 2 at B = 64, the shape bench.py reports as ``cfg2_bf16``: 3 periods per work item, 4 partial chunks of
   out_hidden, up to 3 items per CTA; the step captured in a CUDA graph and replayed;
2. several items per CTA, whose weight gradients accumulate in the same persistent TMEM accumulators, and several
   k_head_tc tiles per CTA: pinned by an exact invariance (a 64-snapshot batch against its two 32-snapshot halves);
3. a period chunk strictly between 1 and T, and micro-batches;
4. 1, 7 and 64 periods; 65 is refused;
5. many regions (k_wgrad_m1_tc with z-splits) and a single region (h_pre on the tensor cores);
6. the head's output width: k_head_tc up to 16, k_head_fused summing the cell's partial chunks up to 44 (the widest its
   shared memory holds at hidden 64), k_hid_reduce + k_head_fwd beyond;
7. the autograd surface: losses on out, on out_hidden only and on both (G written in the tile layout);
8. determinism and a NaN-poisoned workspace.

The work split depends on the SM count, so every case reads it from the library (regt_debug_tc_split) and skips, with
the reason, when the shape does not split as the case needs on this device.

Bounds: the oracle at the stated bf16 tolerances (2e-2 activations and loss, 5e-2 gradients, 0.15 for the attention
gradient).  Invariances of the kernels' own arithmetic are checked far tighter: bit for bit where only which tile or CTA
holds a row differs, 1e-5 normwise (1e-4 for the attention gradient) where only the fp32 order of cross-row sums
differs.  Every test asserts which kernels ran and prints its split and measured errors (run with -s)."""
import ctypes as C
import functools

import pytest
import torch

from parity_util import W, build_cuda, build_oracle, is_dead, oracle_step, profiled, relerr, to_dev
from test_gpu_step_edges import _grads, _hidden_loss_oracle, _profiled_autograd, _run_on_workspace, _zero_grads

pytestmark = pytest.mark.gpu
ATOL, GTOL, ATT_TOL = 2e-2, 5e-2, 0.15       # stated bf16 tolerances against the oracle
ORDER_TOL, ORDER_ATT_TOL = 1e-5, 1e-4        # same rows, fp32 order of the cross-row sums differs
CELL = ("k_cell_fwd_tc", "k_cell_bwd_tc", "k_tc_wreduce")


# ------------------------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------------------------
def tc_split(B, N, T):
    """the work split of the bf16 kernels on this device (regt_debug_tc_split), plus the per-CTA maxima."""
    from regt_b200 import _lib
    o = (C.c_int32 * 7)()
    _lib.check(_lib.load().regt_debug_tc_split(B, N, T, o), "regt_debug_tc_split")
    s = dict(zip(("nqt", "tp", "ntc", "items", "fwd_grid", "bwd_grid", "head_grid"), list(o)))
    s["items_per_cta"] = -(-s["items"] // s["fwd_grid"])
    s["head_tiles_per_cta"] = -(-s["nqt"] // s["head_grid"])
    return s


def _need(cond, why):
    if not cond:
        pytest.skip(f"the split on this device does not give {why}")


def _show(tag, s):
    print(f"\n{tag}: nqt {s['nqt']} tp {s['tp']} ntc {s['ntc']} items {s['items']} grids {s['fwd_grid']}/{s['bwd_grid']}"
          f"/{s['head_grid']}: {s['items_per_cta']} items and {s['head_tiles_per_cta']} head tiles per CTA at most")


def _args(w, B):
    x, y = w.inputs(B)
    return x.cuda(), y.cuda(), to_dev(w.graph_args(), "cuda")


def _check(w, ref, loss, out, hid, grads, tag):
    """activations, loss and every live gradient against the oracle ``ref`` (oracle_step's form) at the bf16 bounds."""
    errs = {"out_hidden": relerr(hid, ref["hid"])}
    if out is not None:
        errs["out"] = relerr(out, ref["out"])
    if loss is not None:
        errs["loss"] = abs(float(loss) - ref["loss"]) / abs(ref["loss"])
    gerr = {}
    for k, g in ref["grads"].items():
        if is_dead(w.model, k):
            continue
        if g is None:      # the oracle's loss does not reach this parameter: the kernels must leave an exact zero
            assert grads[k] is None or float(grads[k].abs().max()) == 0.0, f"{tag}: grad {k} should be zero"
            continue
        gerr[k] = relerr(grads[k], g)
    att = {k: e for k, e in gerr.items() if k.endswith("_attention")}
    rest = {k: e for k, e in gerr.items() if k not in att}
    worst = max(rest, key=rest.get)
    print(f"{tag} vs oracle: " + ", ".join(f"{k} {e:.2e}" for k, e in errs.items()) +
          f", worst grad {worst} {rest[worst]:.2e}" + "".join(f", {k} {e:.2e}" for k, e in att.items()))
    for k, e in errs.items():
        assert e <= ATOL, f"{tag}: {k} {e:.3e} > {ATOL}"
    for k, e in gerr.items():
        bound = ATT_TOL if k in att else GTOL
        assert e <= bound, f"{tag}: grad {k} {e:.3e} > {bound}"


def _same_step(a, b, tag):
    """(loss, out, out_hidden, grads) bit for bit."""
    for i, what in enumerate(("loss", "out", "out_hidden")):
        assert torch.equal(a[i], b[i]), f"{tag}: {what} differs ({relerr(a[i], b[i]):.3e})"
    for k, t in a[3].items():
        assert (t is None) == (b[3][k] is None) and (t is None or torch.equal(t, b[3][k])), f"{tag}: grad {k}"


def _grads_agree(w, ga, gb, tag):
    """gradients of the same rows summed in another fp32 order: ORDER_TOL normwise, ORDER_ATT_TOL for d_attention."""
    errs = {k: relerr(ga[k], gb[k]) for k in ga if ga[k] is not None and not is_dead(w.model, k)}
    worst = max((k for k in errs if not k.endswith("_attention")), key=errs.get)
    att = [k for k in errs if k.endswith("_attention")]
    print(f"{tag}: worst grad {worst} {errs[worst]:.2e}" + "".join(f", {k} {errs[k]:.2e}" for k in att))
    for k, e in errs.items():
        bound = ORDER_ATT_TOL if k in att else ORDER_TOL
        assert e <= bound, f"{tag}: grad {k} {e:.3e} > {bound}"


@functools.lru_cache(maxsize=None)
def _oracle(key):
    """workload, batch and fp64 oracle step of a named case, once per module."""
    w, B = _WORKLOADS[key]()
    return w, B, oracle_step(w, B)


def _tiny(model, N, T, O, B, seed, R=5, **kw):
    return W.tiny_workload(model, N=N, T=T, H=64, O=O, R=R if model == "RegionalTemporalGCN" else 0, B=B, seed=seed, **kw)


_WORKLOADS = {
    "bench_cfg2": lambda: (W.make_workload(2), 64),
    "tp1_cfg2": lambda: (W.make_workload(2, B=3), 3),     # 5 tiles: tp = 1, 12 partial chunks
    # N = 592, T = 12: B = 64 -> 296 tiles, tp = 12, 2 items and 2 head tiles per CTA; B = 32 -> 148 tiles, 1 of each
    "multi_a3tgcn": lambda: (_tiny("TemporalGCN", 592, 12, 12, 64, 80, k_intra=5), 64),
    "multi_regional": lambda: (_tiny("RegionalTemporalGCN", 592, 12, 12, 64, 81, k_intra=4), 64),
    # B = 16 -> 74 tiles, tp = 6, ntc = 2 (a micro-batch of 8: 37 tiles, tp = 3)
    "mid_a3tgcn": lambda: (_tiny("TemporalGCN", 592, 12, 12, 16, 82, k_intra=5), 16),
    "mid_regional": lambda: (_tiny("RegionalTemporalGCN", 592, 12, 12, 16, 83, k_intra=4), 16),
    # config 5's generator: R = 256 regions of 4 nodes, k_wgrad_m1_tc with 1024 / 256 = 4 z-splits
    "many_regions": lambda: (W.cfg5_shaped(N=1024, T=3, H=64, R=256, O=5), 3),
    # one regional list: hmma = 1, h_pre of the regional combine on the tensor cores, dM1 from k_tc_wreduce
    "one_region": lambda: (_tiny("RegionalTemporalGCN", 300, 6, 5, 3, 84, R=1, k_intra=4), 3),
    **{f"width_{O}": (lambda O=O: (_tiny("TemporalGCN", 592, 12, O, 16, 90 + O, k_intra=5), 16)) for O in (16, 17, 44, 45, 64, 65)},
    **{f"periods_{m}_{T}": (lambda m=m, T=T: (_tiny(m, 70, T, 3, 2, 40 + T), 2))
       for m in ("TemporalGCN", "RegionalTemporalGCN") for T in (1, 7, 64)},
}


def _fused(key, micro_batch=None):
    """fused_step of case ``key`` on a model with the oracle's parameters: ((loss, out, hid), grads, kernel names)."""
    w, B, ref = _oracle(key)
    x, y, g = _args(w, B)
    m = build_cuda(w, ref["state"], precision="bf16")
    res, names = profiled(lambda: m.fused_step(x, y, *g, micro_batch=micro_batch or B))
    return res, _grads(m), names


def _ran(names, must=(), must_not=()):
    for k in must:
        assert k in names, (k, sorted(names))
    for k in must_not:
        assert k not in names, (k, sorted(names))


# ------------------------------------------------------------------------------------------------------------------
# 1. the bench's shape, eager and replayed from a CUDA graph
# ------------------------------------------------------------------------------------------------------------------
def test_bench_shape_matches_oracle_and_graph_replay():
    """config 2, B = 64 (tp = 3, ntc = 4, up to 3 items per CTA) through fused_step, then captured as bench.py's
    measure_cfg2_bf16 does.  A replay equals an eager step bit for bit; after new inputs are copied into the static
    buffers and one weight of each kind changes in place, a replay equals an eager step and a freshly built model bit
    for bit (nothing may be packed once at capture time)."""
    w, B, ref = _oracle("bench_cfg2")
    s = tc_split(B, w.N, w.T)
    _show("cfg2 B=64", s)
    _need(1 < s["tp"] < w.T and s["items_per_cta"] >= 2, "1 < tp < T and several items per CTA")
    (loss, out, hid), grads, names = _fused("bench_cfg2")
    _ran(names, CELL + ("k_head_tc",), ("k_hid_reduce", "k_head_fused", "k_head_fwd"))
    _check(w, ref, loss, out, hid, grads, "cfg2 B=64")

    m = build_cuda(w, ref["state"], precision="bf16")
    x, y = w.inputs(B)
    xs, ys = x.cuda(), y.cuda()
    g = to_dev(w.graph_args(), "cuda")

    def step():
        return m.fused_step(xs, ys, *g)

    for _ in range(2):
        step()
    sd = torch.cuda.Stream()
    sd.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(sd):
        _zero_grads(m)
        step()
    torch.cuda.current_stream().wait_stream(sd)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        st_loss, st_out, st_hid = step()
    torch.cuda.synchronize()

    def replay():
        _zero_grads(m)
        graph.replay()
        torch.cuda.synchronize()
        return st_loss.clone(), st_out.clone(), st_hid.clone(), _grads(m)

    def eager():
        _zero_grads(m)
        res = step()
        torch.cuda.synchronize()
        return (*(t.clone() for t in res), _grads(m))

    r0 = replay()
    _same_step(r0, eager(), "first replay vs eager")
    _check(w, ref, *r0, "cfg2 B=64 first replay")

    x2, y2 = w.inputs(B, seed_offset=1)
    xs.copy_(x2)
    ys.copy_(y2)
    gen = torch.Generator().manual_seed(3)
    p = m._param_dict()
    with torch.no_grad():
        for k in ("conv_w0", "lin_w1", "head_w2", "attention"):
            p[k].mul_(1.0 + 0.2 * (torch.rand(p[k].shape, generator=gen) - 0.5).cuda())
    r = replay()
    _same_step(r, eager(), "replay after the update vs eager")
    assert not torch.equal(r[1], r0[1])
    new_state = {k: v.detach().double().cpu() for k, v in m.state_dict().items()}
    fresh = build_cuda(w, new_state, precision="bf16")
    res = fresh.fused_step(xs, ys, *g)
    torch.cuda.synchronize()
    _same_step(r, (*res, _grads(fresh)), "replay after the update vs a fresh model")


# ------------------------------------------------------------------------------------------------------------------
# 2. several items per CTA: a batch against its halves
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("key", ["multi_a3tgcn", "multi_regional"])
def test_items_per_cta_split_invariance(key):
    """B = 64 gives every CTA 2 items (accumulated into the same TMEM weight-gradient accumulators) and 2 k_head_tc
    tiles; each B = 32 half gives it 1 of each, with the same tp.  A row's arithmetic does not depend on which tile or
    CTA holds it (an MMA row is independent of the others, bf16 rounding is per element, equal tp keeps the period order
    of the attention sum), so out and out_hidden of the batch equal those of the halves bit for bit, the loss agrees to
    1e-6 and the gradients (one step against two accumulating half steps) to the fp32 order of the cross-row sums."""
    w, B, ref = _oracle(key)
    full, half = tc_split(B, w.N, w.T), tc_split(B // 2, w.N, w.T)
    _show(f"{key} B={B}", full)
    _show(f"{key} B={B // 2}", half)
    _need(full["items_per_cta"] >= 2 and full["head_tiles_per_cta"] >= 2, "several items and head tiles per CTA")
    _need(half["items_per_cta"] == 1 and half["tp"] == full["tp"], "one item per CTA in a half at the same tp")
    (loss, out, hid), grads, names = _fused(key)
    _ran(names, CELL + ("k_head_tc",), ("k_hid_reduce",))
    if w.model == "RegionalTemporalGCN":
        _ran(names, ("k_wgrad_m1_tc",))
    _check(w, ref, loss, out, hid, grads, key)
    (loss2, out2, hid2), grads2, _ = _fused(key, micro_batch=B // 2)
    print(f"{key}: batch vs halves: out {relerr(out, out2):.2e}, out_hidden {relerr(hid, hid2):.2e}, "
          f"loss {abs(float(loss) - float(loss2)) / abs(float(loss)):.2e}")
    assert torch.equal(hid, hid2), f"out_hidden depends on the split: {relerr(hid, hid2):.3e}"
    assert torch.equal(out, out2), f"out depends on the split: {relerr(out, out2):.3e}"
    assert abs(float(loss) - float(loss2)) <= 1e-6 * abs(float(loss))
    _grads_agree(w, grads, grads2, f"{key} batch vs halves")


# ------------------------------------------------------------------------------------------------------------------
# 3. 1 < tp < T and micro-batches
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mb", [16, 8])
@pytest.mark.parametrize("key", ["mid_a3tgcn", "mid_regional"])
def test_partial_period_chunks_and_micro_batches(key, mb):
    """B = 16 at N = 592: tp = 6, two partial chunks of out_hidden summed by k_head_tc.  micro_batch = 8 runs two steps
    (tp = 3 each), the second accumulating into .grad: both meet the oracle, and the micro-batched gradients agree with
    the whole batch's to the fp32 order of the sums.  out_hidden agrees to 1e-6 (its chunks are summed in another
    grouping); out is held to the oracle only, because the head rounds out_hidden to bf16 and a last-bit difference can
    move an element to the neighbouring bf16 value."""
    w, B, ref = _oracle(key)
    s, sm = tc_split(B, w.N, w.T), tc_split(mb, w.N, w.T)
    _show(f"{key} B={B}", s)
    _show(f"{key} micro-batch {mb}", sm)
    _need(1 < s["tp"] < w.T and s["ntc"] < w.T, "1 < tp < T")
    (loss, out, hid), grads, names = _fused(key, micro_batch=mb)
    _ran(names, CELL + ("k_head_tc",), ("k_hid_reduce",))
    _check(w, ref, loss, out, hid, grads, f"{key}/mb={mb}")
    if mb < B:
        (_, out1, hid1), grads1, _ = _fused(key)
        print(f"{key}: micro-batches vs whole: out {relerr(out, out1):.2e}, out_hidden {relerr(hid, hid1):.2e}")
        assert relerr(hid, hid1) <= 1e-6
        _grads_agree(w, grads, grads1, f"{key} micro-batch {mb} vs whole")


# ------------------------------------------------------------------------------------------------------------------
# 4. periods
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T", [1, 7, 64])
@pytest.mark.parametrize("model", ["TemporalGCN", "RegionalTemporalGCN"])
def test_period_counts_match_oracle(model, T):
    """the bf16 kernels hold up to 64 periods (the constants image's probability slots, the per-lane attention-gradient
    sums of periods lane and 32 + lane).  At T = 1 the softmax over one period has a zero Jacobian: d_attention is 0."""
    key = f"periods_{model}_{T}"
    w, B, ref = _oracle(key)
    _show(key, tc_split(B, w.N, w.T))
    (loss, out, hid), grads, names = _fused(key)
    _ran(names, CELL + ("k_head_tc",))
    if T == 1:
        att = [k for k in grads if k.endswith("_attention")][0]
        assert float(grads[att].abs().max()) == 0.0, "d_attention must be exactly zero at one period"
        ref = dict(ref, grads={k: v for k, v in ref["grads"].items() if k != att})
    _check(w, ref, loss, out, hid, grads, key)


@pytest.mark.parametrize("model", ["TemporalGCN", "RegionalTemporalGCN"])
def test_65_periods_explicit_bf16_is_refused(model):
    w = _tiny(model, 70, 65, 3, 2, 105)
    m = build_cuda(w, build_oracle(w).state_dict(), precision="bf16")
    x, y, g = _args(w, 2)
    with pytest.raises(RuntimeError, match="up to 64 periods"):
        m.fused_step(x, y, *g)
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------------------------
# 5. regions
# ------------------------------------------------------------------------------------------------------------------
def test_many_regions_z_split_dm1():
    """R = 256: k_wgrad_m1_tc splits each region's (segment, snapshot) items over 1024 / R = 4 z-slices, several
    items per slice, summed by launch_reduce_splits."""
    w, B, ref = _oracle("many_regions")
    _show("many regions", tc_split(B, w.N, w.T))
    zs = max(1, min(64, 1024 // w.R))
    x, y, g = _args(w, B)
    m = build_cuda(w, ref["state"], precision="bf16")
    rseg_ptr = m._plan(x, g[0], g[1:]).t["rseg_ptr"].cpu()
    per = [-(-int(n) * B // zs) for n in rseg_ptr.diff()]
    print(f"many regions: {zs} z-splits, items per split up to {max(per)}")
    _need(zs > 1 and max(per) >= 2, "several z-splits with several items each")
    (loss, out, hid), names = profiled(lambda: m.fused_step(x, y, *g, micro_batch=B))
    _ran(names, CELL + ("k_wgrad_m1_tc", "k_head_tc"))
    _check(w, ref, loss, out, hid, _grads(m), "R=256")


def test_one_region_h_pre_on_tensor_cores():
    """a regional model with one regional list: every row uses the same M1 block, so h_pre runs as an MMA (hmma) in the
    forward and the backward, and dM1 comes out of the cell backward's own accumulators (no k_wgrad_m1_tc)."""
    w, B, ref = _oracle("one_region")
    _show("one region", tc_split(B, w.N, w.T))
    (loss, out, hid), grads, names = _fused("one_region")
    _ran(names, CELL + ("k_head_tc",), ("k_wgrad_m1_tc",))
    _check(w, ref, loss, out, hid, grads, "R=1")


# ------------------------------------------------------------------------------------------------------------------
# 6. head widths in fused_step
# ------------------------------------------------------------------------------------------------------------------
_FUSED_HEAD = (("k_head_fused", "k_head_grad_reduce"), ("k_head_tc", "k_hid_reduce", "k_head_fwd"))
_ROW_HEAD = (("k_hid_reduce", "k_head_fwd", "k_head_bwd"), ("k_head_tc", "k_head_fused"))
_HEADS = {16: (("k_head_tc",), ("k_head_fused", "k_hid_reduce", "k_head_fwd")),
          17: _FUSED_HEAD, 44: _FUSED_HEAD, 45: _ROW_HEAD, 64: _ROW_HEAD, 65: _ROW_HEAD}


@pytest.mark.parametrize("O", list(_HEADS))
def test_head_width(O):
    """on a tp > 1 shape (two partial chunks of out_hidden): O <= 16 -> k_head_tc; 17..44 -> k_head_fused, which sums
    the cell's chunks itself while loading its tiles; from 45 on, k_head_fused's weights and tiles exceed the 227 KB of
    shared memory a block may use at hidden 64 (O = 64 asked for 260 KB and failed to launch before head_fused_fits checked
    it): k_hid_reduce, then k_head_fwd / k_head_bwd."""
    key = f"width_{O}"
    w, B, ref = _oracle(key)
    s = tc_split(B, w.N, w.T)
    _show(key, s)
    _need(1 < s["ntc"] < w.T, "several partial chunks, fewer than T")
    (loss, out, hid), grads, names = _fused(key)
    _ran(names, CELL + _HEADS[O][0], _HEADS[O][1])
    _check(w, ref, loss, out, hid, grads, f"O={O}")


# ------------------------------------------------------------------------------------------------------------------
# 7. the autograd surface
# ------------------------------------------------------------------------------------------------------------------
_LOSSES = ("out", "hidden_only", "out_and_hidden")


@functools.lru_cache(maxsize=None)
def _loss_oracle(key, loss):
    """fp64 oracle of ``loss`` (sum over b of mean((out_b - y_b)^2), <c_b, hid_b>, or both) and its weights c."""
    w, B, ref = _oracle(key)
    if loss == "out":
        return ref, None
    c = (torch.rand(B, w.N, w.H, generator=torch.Generator().manual_seed(7), dtype=torch.float64) - 0.5) * (4.0 / (w.N * w.H))
    return _hidden_loss_oracle(w, B, c, loss == "out_and_hidden", torch.float64), c


@pytest.mark.parametrize("loss", _LOSSES)
@pytest.mark.parametrize("key", ["mid_regional", "tp1_cfg2"])
def test_autograd_losses(key, loss):
    """model(...) + backward in bf16: the forward leaves out_hidden through k_hid_reduce and runs k_head_fwd; the
    backward writes G in the tile layout the cell backward reads (k_head_bwd, or k_copy_or_zero when only out_hidden
    carries the loss).  out_hidden of the autograd forward matches fused_step's to 1e-6: both sum the same partials."""
    w, B, _ = _oracle(key)
    s = tc_split(B, w.N, w.T)
    _show(key, s)
    ref, c = _loss_oracle(key, loss)
    x, y, g = _args(w, B)
    m = build_cuda(w, ref["state"], precision="bf16")
    cd = None if c is None else c.float().cuda()

    def loss_of(out, hid):
        mse = ((out - y) ** 2).mean(dim=(1, 2)).sum()
        if loss == "out":
            return mse
        return (cd * hid).sum() + (mse if loss == "out_and_hidden" else 0.0)

    (lv, out, hid), names = _profiled_autograd(lambda: m(x, *g), loss_of)
    _ran(names, CELL + ("k_hid_reduce", "k_head_fwd") + (("k_copy_or_zero",) if loss == "hidden_only" else ("k_head_bwd",)),
         ("k_head_tc", "k_head_fused"))
    _check(w, ref, lv, out, hid, _grads(m), f"{key}/autograd/{loss}")
    _, _, hid_f = build_cuda(w, ref["state"], precision="bf16").fused_step(x, y, *g, micro_batch=B)
    print(f"{key}: out_hidden autograd vs fused_step {relerr(hid, hid_f):.2e}")
    assert relerr(hid, hid_f) <= 1e-6



# ------------------------------------------------------------------------------------------------------------------
# 8. determinism and an uninitialised workspace
# ------------------------------------------------------------------------------------------------------------------
def test_two_identical_steps_are_bit_identical():
    w, B, _ = _oracle("multi_regional")
    _show("multi_regional", tc_split(B, w.N, w.T))
    (l1, o1, h1), g1, _ = _fused("multi_regional")
    (l2, o2, h2), g2, _ = _fused("multi_regional")
    _same_step((l1, o1, h1, g1), (l2, o2, h2, g2), "two identical steps")


@pytest.mark.parametrize("key", ["multi_a3tgcn", "width_17"])
def test_poisoned_workspace_gives_the_same_step(key, monkeypatch):
    """the same step on a NaN-filled and on a zeroed workspace: finite and bit-identical results.  At several items per
    CTA (pad rows of the last tile, partial chunks written per item) and with k_head_fused reading the partial chunks."""
    monkeypatch.setenv("REGT_UNFUSED", "0")
    w, B, _ = _oracle(key)
    _show(key, tc_split(B, w.N, w.T))
    runs = [_run_on_workspace(w, B, "bf16", "fused", poison) for poison in (True, False)]
    _ran(runs[0][2], CELL + (("k_head_fused",) if key == "width_17" else ("k_head_tc",)))
    (res_p, grads_p, _), (res_z, grads_z, _) = runs
    for what, a in zip(("loss", "out", "out_hidden"), res_p):
        assert torch.isfinite(a).all(), f"{key}: {what} not finite on the poisoned workspace"
    for k, a in grads_p.items():
        assert a is None or torch.isfinite(a).all(), f"{key}: grad {k} not finite on the poisoned workspace"
    _same_step((*res_p, grads_p), (*res_z, grads_z), f"{key}: poisoned vs zeroed workspace")
