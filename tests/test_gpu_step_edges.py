"""The default tf32x3 training step (fused 3xTF32 cell of cell_f.cu + tensor-core head of head_f.cu) at the edges the
other parity tests do not reach, each against the fp64 oracle of the same batch:

1. micro-batched steps (``micro_batch`` 4 = 4 + 4 + 1, and 1): every micro-batch after the first ACCUMULATES into .grad;
2. the grouped dM1 contraction ``k_wgrad_m1_kt`` with several snapshots per group and a shorter last group;
3. the step captured in a CUDA graph and replayed (as bench.py runs it), also after inputs and parameters change in place;
4. a workspace whose bytes start as all-ones (every float NaN) against a zeroed one: no kernel may read a byte it did
   not write first (pad rows of the 128-row tiles, partial slots);
5. the period count: 1, 7, 63 and 64 periods on the fused kernels, 65 on the fp32 kernels under ``precision="auto"``;
6. the head's output width around the 16 outputs of ``k_hf_mid``'s shuffle exchange, and its B*N >= 128 cut-over;
7. a loss on ``out_hidden`` (d_hidden written into the tile layout of G the fused backward reads).

Tolerances are the suite's: 1e-5 normwise for activations and loss; gradients <= 1e-5 or 4x the fp32 twin's own error
(parity_util.twin_limits); the period-attention gradient, a softmax-Jacobian difference of nearly equal sums, within
the 3xTF32 paths' stated 1e-4.  Every test asserts which kernels ran, so a silent fallback cannot pass for the path."""
import functools

import pytest
import torch

from parity_util import W, build_cuda, build_oracle, is_dead, oracle_step, profiled, relerr, to_dev, twin_limits

pytestmark = pytest.mark.gpu
TOL = 1e-5
ATT_TOL = 1e-4
FUSED = ("k_cell_fwd_f", "k_cell_bwd_f")


def _profiled_autograd(forward, loss_of):
    """``forward()`` -> (out, out_hidden) and ``loss_of(out, hid).backward()``; returns ((loss, out, hid), kernel names of
    both).  Autograd runs the model node's backward on its own thread and the recorder is per thread, so hooks on that
    node switch the recorder on and off around it there."""
    from regt_b200 import _lib
    lib = _lib.load()
    (out, hid), names = profiled(forward)

    def pre(grad_outputs):
        lib.regt_profile(1, torch.cuda.current_stream().cuda_stream)

    def post(grad_inputs, grad_outputs):
        torch.cuda.synchronize()
        names.update(n for n, _ in _lib.profile_read())
        lib.regt_profile(0, None)

    node = hid.grad_fn
    hooks = [node.register_prehook(pre), node.register_hook(post)]
    try:
        loss = loss_of(out, hid)
        loss.backward()
        torch.cuda.synchronize()
    finally:
        for h in hooks:
            h.remove()
    return (loss.detach(), out.detach(), hid.detach()), names


def _grads(m):
    return {k: (None if p.grad is None else p.grad.detach().clone()) for k, p in m.named_parameters()}


def _check(w, ref, lims, loss, out, hid, grads, tag):
    """activations, loss and every live gradient against the oracle ``ref`` (dict of oracle_step's form)."""
    if out is not None:
        assert relerr(out, ref["out"]) <= TOL, f"{tag}: out {relerr(out, ref['out']):.3e}"
    assert relerr(hid, ref["hid"]) <= TOL, f"{tag}: out_hidden {relerr(hid, ref['hid']):.3e}"
    if loss is not None:
        assert abs(float(loss) - ref["loss"]) <= TOL * abs(ref["loss"]), f"{tag}: loss {float(loss)} vs {ref['loss']}"
    for k, g in ref["grads"].items():
        if is_dead(w.model, k):
            continue
        if g is None:      # the oracle's loss does not reach this parameter: the kernels must leave an exact zero
            assert grads[k] is None or float(grads[k].abs().max()) == 0.0, f"{tag}: grad {k} should be zero"
            continue
        e = relerr(grads[k], g)
        bound = max(lims[k], ATT_TOL) if k.endswith("_attention") else lims[k]
        assert e <= bound, f"{tag}: grad {k} {e:.3e} > {bound:.3e}"


@functools.lru_cache(maxsize=None)
def _oracle(key):
    """fp64 oracle step and fp32-twin gradient bounds of a named case, once per module (the large ones take minutes)."""
    w, B = _WORKLOADS[key]()
    ref = oracle_step(w, B)
    lims, _ = twin_limits(w, B, ref)
    return w, B, ref, lims


_WORKLOADS = {
    # 9 * 700 = 6300 rows: the last 128-row tile holds 28 rows; micro-batches of 4 (2800 rows) and 1 (700) are ragged too
    "regional_h128": lambda: (W.tiny_workload("RegionalTemporalGCN", N=700, T=4, H=128, O=4, R=5, B=9, seed=9), 9),
    "regional_h64": lambda: (W.tiny_workload("RegionalTemporalGCN", N=300, T=6, H=64, O=5, R=7, B=9, seed=31, k_intra=4), 9),
    # config 5's generator: bper = 2 snapshots per dM1 group, groups 2+2+2+2+1 (NPW = 8 kernel, H = 128) ...
    "grouped_h128": lambda: (W.cfg5_shaped(N=1024, T=2, H=128, R=256), 9),
    # ... and 2+2+1 (NPW = 4 kernel, H = 64)
    "grouped_h64": lambda: (W.cfg5_shaped(N=1024, T=3, H=64, R=512), 5),
}


# ------------------------------------------------------------------------------------------------------------------
# 1. micro-batches
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mb", [None, 4, 1], ids=["whole", "mb4", "mb1"])
@pytest.mark.parametrize("key", ["regional_h128", "regional_h64"])
def test_micro_batched_step_matches_oracle(key, mb):
    """``fused_step(micro_batch=mb)`` runs B / mb steps of the kernels, each after the first accumulating into .grad (and
    the loss), the last one ragged at B = 9, mb = 4.  Whole-batch oracle; out and out_hidden agree with the single-pass
    run to 3e-6 (not bit for bit: whether an item's h_pre takes the MMA or the CUDA-core path depends on which rows
    share its 128-row tile)."""
    w, B, ref, lims = _oracle(key)
    x, y = w.inputs(B)
    x, y = x.cuda(), y.cuda()
    g = to_dev(w.graph_args(), "cuda")
    m = build_cuda(w, ref["state"], precision="tf32x3")
    (loss, out, hid), names = profiled(lambda: m.fused_step(x, y, *g, micro_batch=mb or B))
    for k in FUSED + ("k_wgrad_m1_kt", "k_chain", "k_hf_mid"):
        assert k in names, (k, sorted(names))
    _check(w, ref, lims, loss, out, hid, _grads(m), f"{key}/mb={mb}")
    one = build_cuda(w, ref["state"], precision="tf32x3")
    _, out1, hid1 = one.fused_step(x, y, *g, micro_batch=B)
    assert relerr(out, out1) <= 3e-6 and relerr(hid, hid1) <= 3e-6


# ------------------------------------------------------------------------------------------------------------------
# 2. grouped dM1 contraction
# ------------------------------------------------------------------------------------------------------------------
def _m1_groups(B, R):
    """launch_wgrad_m1_kt (cell.cu): snapshots per group and group count of the per-region dM1 contraction."""
    nbg = min(B, max(1, 2048 // max(R, 1)))
    bper = -(-B // nbg)
    return bper, -(-B // bper)


@pytest.mark.parametrize("key", ["grouped_h128", "grouped_h64"])
def test_grouped_dm1_contraction_matches_oracle(key):
    """config 5 runs the contraction with 2 snapshots per group (R = 256, micro-batch 16); here groups of 2 and a last
    group of 1, so both the in-group loop over snapshots and its ragged end meet the oracle."""
    w, B, ref, lims = _oracle(key)
    bper, nbg = _m1_groups(B, w.R)
    assert bper > 1 and B % bper != 0, (B, w.R, bper, nbg)      # the case still exercises what it is named for
    x, y = w.inputs(B)
    m = build_cuda(w, ref["state"], precision="tf32x3")
    (loss, out, hid), names = profiled(lambda: m.fused_step(x.cuda(), y.cuda(), *to_dev(w.graph_args(), "cuda"),
                                                            micro_batch=B))
    for k in FUSED + ("k_wgrad_m1_kt",):
        assert k in names, (k, sorted(names))
    _check(w, ref, lims, loss, out, hid, _grads(m), key)


# ------------------------------------------------------------------------------------------------------------------
# 3. CUDA-graph replay
# ------------------------------------------------------------------------------------------------------------------
def _oracle_at(w, state, x, y):
    """fp64 oracle step (and fp32-twin bounds) at the parameters ``state`` and the inputs (x, y)."""
    from oracle import regt_oracle as O
    out = {}
    for dt in (torch.float64, torch.float32):
        m = build_oracle(w, dt)
        m.load_state_dict({k: v.to(dt) for k, v in state.items()})
        o, h, loss = O.batched_step(m, x.to(dt), y.to(dt), w.graph_args())
        out[dt] = dict(out=o, hid=h, loss=loss, grads={k: p.grad for k, p in m.named_parameters()})
    ref, twin = out[torch.float64], out[torch.float32]
    lims = {k: max(TOL, 4.0 * relerr(twin["grads"][k], g)) for k, g in ref["grads"].items() if g is not None}
    return ref, lims


def _zero_grads(m):
    for p in m.parameters():
        if p.grad is not None:
            p.grad.zero_()


def test_graph_replay_matches_eager_and_follows_inplace_updates():
    """bench.py's loop: warm-up on a side stream, capture fused_step(micro_batch=4), replay with .grad zeroed in place.
    A replay equals an eager step bit for bit and meets the oracle; after new inputs are copied into the static buffers and
    one weight of each kind changes in place, the next replay equals an eager step and a freshly built model bit for bit,
    and its activations and loss meet the oracle at the new values (nothing may be packed once at capture time)."""
    w = W.tiny_workload("RegionalTemporalGCN", N=700, T=4, H=128, O=4, R=5, B=8, seed=9)
    B = 8
    state = build_oracle(w).state_dict()
    m = build_cuda(w, state, precision="tf32x3")
    x, y = w.inputs(B)
    xs, ys = x.cuda(), y.cuda()
    g = to_dev(w.graph_args(), "cuda")

    def step():
        return m.fused_step(xs, ys, *g, micro_batch=4)

    # the graph's content is first seen through other tensors (as after the reference's per-snapshot .to(device)): the
    # capture below must still find the plan by the identity of ``g`` without hashing or building it on the device
    m.fused_step(xs, ys, *[t.clone() for t in g], micro_batch=4)
    _, names = profiled(step)                      # eager warm-up: creates .grad, the workspace and the plan
    for k in FUSED + ("k_wgrad_m1_kt", "k_hf_mid"):
        assert k in names, (k, sorted(names))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        _zero_grads(m)
        step()
    torch.cuda.current_stream().wait_stream(s)
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
        loss, out, hid = step()
        torch.cuda.synchronize()
        return loss.clone(), out.clone(), hid.clone(), _grads(m)

    def same(a, b, tag):
        for i, what in enumerate(("loss", "out", "out_hidden")):
            assert torch.equal(a[i], b[i]), f"{tag}: {what} of the replay differs from the eager step"
        for k, t in a[3].items():
            assert (t is None) == (b[3][k] is None) and (t is None or torch.equal(t, b[3][k])), f"{tag}: grad {k}"

    r0 = replay()
    same(r0, eager(), "first replay")
    ref0, lims0 = _oracle_at(w, {k: v.double() for k, v in state.items()}, x, y)
    _check(w, ref0, lims0, r0[0], r0[1], r0[2], r0[3], "first replay")

    x2, y2 = w.inputs(B, seed_offset=1)
    xs.copy_(x2)
    ys.copy_(y2)
    gen = torch.Generator().manual_seed(3)
    p = m._param_dict()
    with torch.no_grad():
        for k in ("lin_w1", "comb_w", "head_w2", "attention"):
            p[k].mul_(1.0 + 0.2 * (torch.rand(p[k].shape, generator=gen) - 0.5).cuda())
    r = replay()
    same(r, eager(), "replay after the update")
    new_state = {k: v.detach().double().cpu() for k, v in m.state_dict().items()}
    assert not torch.equal(new_state["linear2.weight"], state["linear2.weight"].double())
    fresh = build_cuda(w, new_state, precision="tf32x3")       # no history: its own workspace, plan lookup and .grad
    res = fresh.fused_step(xs, ys, *g, micro_batch=4)
    torch.cuda.synchronize()
    same(r, (*res, _grads(fresh)), "replay after the update vs a fresh model")
    # the new values are in effect: activations and loss meet the oracle at them.  Gradients are pinned by the bit-identity
    # with the fresh model above; their oracle bound is checked at the original values (first replay).
    ref, _ = _oracle_at(w, new_state, x2, y2)
    _check(w, dict(ref, grads={}), {}, r[0], r[1], r[2], r[3], "replay after the update")


# ------------------------------------------------------------------------------------------------------------------
# 4. uninitialised workspace
# ------------------------------------------------------------------------------------------------------------------
def _m1cp_offset(nbytes, R):
    """byte offset of the int32 dM1 chunk table ``m1cp`` in a workspace of ``nbytes`` = regt_workspace_bytes(args).
    make_layout (api.cu) carves it last, R + 2 entries (R = max(plan.R, 1)) at a 256-byte aligned offset, and rounds the
    total up to 256 bytes: it occupies the last align_up(4 (R + 2), 256) bytes.  Its entries are chunk bounds that index
    other buffers, so the poisoned runs leave it zero: the test is about float data, not about out-of-range indices."""
    return nbytes - (-(-4 * (max(R, 1) + 2) // 256) * 256)


def _workspace(nbytes, R, poison):
    ws = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
    if poison:
        ws[:_m1cp_offset(nbytes, R)].fill_(0xFF)          # 0xFFFFFFFF: a NaN in every float slot
    return ws


_POISON_CASES = {
    # (workload, B, precision, path, REGT_UNFUSED, kernels that must run)
    # 3 * 700 = 2100 rows: the last 128-row tile holds 52 real rows
    "fused_h128": (lambda: W.tiny_workload("RegionalTemporalGCN", N=700, T=4, H=128, O=4, R=5, B=3, seed=9), 3,
                   "tf32x3", "fused", "0", FUSED + ("k_wgrad_m1_kt", "k_hf_mid")),
    # R = 256 regions of 1-2 nodes: one tile spans ~100 regions; 2 * 333 = 666 rows (26 in the last tile)
    "fused_h64_many_regions": (lambda: W.cfg5_shaped(N=333, T=3, H=64, R=256, O=5), 2, "tf32x3", "fused", "0",
                               FUSED + ("k_wgrad_m1_kt", "k_hf_mid")),
    "unfused_h128": (lambda: W.tiny_workload("RegionalTemporalGCN", N=700, T=4, H=128, O=4, R=5, B=3, seed=9), 3,
                     "tf32x3", "fused", "1", ("k_g_zr", "k_g_b1")),
    # 2 * 20 * 3 = 120 rows: fewer than one 128-row tile of the GEMMs (TMA reads the rows past M as zeros)
    "unfused_h128_one_partial_tile": (lambda: W.tiny_workload("RegionalTemporalGCN", N=20, T=3, H=128, O=4, R=3, B=2, seed=10), 2,
                                      "tf32x3", "fused", "1", ("k_g_zr", "k_gemm_nt_tma_ts", "k_gemm_tn_tma")),
    "fp32_h64": (lambda: W.tiny_workload("RegionalTemporalGCN", N=300, T=6, H=64, O=5, R=7, B=3, seed=31, k_intra=4), 3,
                 "fp32", "fused", "0", ("k_cell_fwd", "k_cell_bwd")),
    "bf16_h64": (lambda: W.tiny_workload("TemporalGCN", N=150, T=12, H=64, O=12, R=0, B=3, seed=7, k_intra=5), 3,
                 "bf16", "fused", "0", ("k_cell_fwd_tc", "k_cell_bwd_tc")),
    "autograd_h128": (lambda: W.tiny_workload("RegionalTemporalGCN", N=700, T=4, H=128, O=4, R=5, B=3, seed=9), 3,
                      "tf32x3", "autograd", "0", FUSED + ("k_hf_mid", "k_hf_gmask")),
    "inference_h128": (lambda: W.tiny_workload("RegionalTemporalGCN", N=700, T=4, H=128, O=4, R=5, B=3, seed=9), 3,
                       "tf32x3", "inference", "0", ("k_cell_fwd_f", "k_hf_mid")),
}


def _run_on_workspace(w, B, precision, path, poison):
    """one step on a workspace of exactly the size the step asks for, either poisoned or zeroed.
    ``fused``: fused_step with the workspace pre-seeded as the model's cached one; ``autograd``: what the autograd Function
    runs (forward, then backward of sum_b mean((out_b - y_b)^2) with d_out computed here, gradients overwritten);
    ``inference``: the forward-only step of torch.no_grad() call sites."""
    from regt_b200 import engine
    x, y = w.inputs(B)
    x, y = x.cuda(), y.cuda()
    g = to_dev(w.graph_args(), "cuda")
    m = build_cuda(w, build_oracle(w).state_dict(), precision=precision)
    plan = m._plan(x, g[0], g[1:]) if w.model == "RegionalTemporalGCN" else m._plan(x, g[0], g[1])
    prec = m._prec(w.T)
    params = m._param_dict()

    def ws_for(**kw):
        st = engine.build_state(m._mode, prec, plan, x, w.H, w.O, params, **kw)     # sizes the request only
        return _workspace(st.args.workspace_bytes, w.R, poison)

    if path == "fused":
        m._ws = ws_for(y=y, fuse_head=True)
        (loss, out, hid), names = profiled(lambda: m.fused_step(x, y, *g, micro_batch=B))
        return (loss, out, hid), _grads(m), names
    if path == "inference":
        def fwd():
            st = engine.build_state(m._mode, prec, plan, x, w.H, w.O, params, inference=True,
                                    workspace=ws_for(inference=True))
            engine.run_forward(st, True)
            return st.out, st.out_hidden
        (out, hid), names = profiled(fwd)
        return (None, out, hid), {}, names

    def fwd_bwd():
        st = engine.build_state(m._mode, prec, plan, x, w.H, w.O, params, workspace=ws_for())
        engine.run_forward(st, True)
        d_out = (2.0 / (w.N * w.O)) * (st.out - y)
        grads = {k: torch.empty_like(t) for k, t in params.items()}
        engine.run_backward(st, grads, d_out, None, False, True)
        return st.out, st.out_hidden, grads
    (out, hid, grads), names = profiled(fwd_bwd)
    return (None, out, hid), grads, names


@pytest.mark.parametrize("case", list(_POISON_CASES))
def test_poisoned_workspace_gives_the_same_step(case, monkeypatch):
    """the same step on a NaN-filled and on a zeroed workspace: finite and bit-identical outputs, loss and gradients.
    Workspaces are torch.empty in use, so a read of a pad row or a slot no kernel wrote would make results depend on
    whatever the allocator hands out."""
    make, B, precision, path, unfused, kernels = _POISON_CASES[case]
    monkeypatch.setenv("REGT_UNFUSED", unfused)
    w = make()
    runs = [_run_on_workspace(w, B, precision, path, poison) for poison in (True, False)]
    for k in kernels:
        assert k in runs[0][2], (k, sorted(runs[0][2]))
    (res_p, grads_p, _), (res_z, grads_z, _) = runs
    for what, a, b in zip(("loss", "out", "out_hidden"), res_p, res_z):
        if a is None:
            continue
        assert torch.isfinite(a).all(), f"{case}: {what} not finite on the poisoned workspace"
        assert torch.equal(a, b), f"{case}: {what} depends on the workspace's initial bytes"
    for k, a in grads_p.items():
        if a is None:
            continue
        assert torch.isfinite(a).all(), f"{case}: grad {k} not finite on the poisoned workspace"
        assert torch.equal(a, grads_z[k]), f"{case}: grad {k} depends on the workspace's initial bytes"


# ------------------------------------------------------------------------------------------------------------------
# 5. period limits
# ------------------------------------------------------------------------------------------------------------------
def _period_case(model, T):
    if model == "regional":
        return W.tiny_workload("RegionalTemporalGCN", N=60, T=T, H=128, O=3, R=3, B=2, seed=41), 2
    return W.tiny_workload("TemporalGCN", N=70, T=T, H=64, O=2, R=0, B=2, seed=42), 2


@pytest.mark.parametrize("T", [1, 7, 63, 64])
@pytest.mark.parametrize("model", ["regional", "a3tgcn"])
def test_fused_period_counts_match_oracle(model, T):
    """the fused kernels hold up to 64 periods (per-period partials of k_cell_bwd_f, the constants image's probability
    slots, k_f_sum_dpp's 64 threads).  At T = 1 the softmax over one period has a zero Jacobian: d_attention is exactly 0."""
    w, B = _period_case(model, T)
    ref = oracle_step(w, B)
    lims, _ = twin_limits(w, B, ref)
    m = build_cuda(w, ref["state"], precision="auto")       # the default picks the fused kernels up to 64 periods
    x, y = w.inputs(B)
    (loss, out, hid), names = profiled(lambda: m.fused_step(x.cuda(), y.cuda(), *to_dev(w.graph_args(), "cuda")))
    for k in FUSED + ("k_f_sum_dpp",):
        assert k in names, (k, sorted(names))
    grads = _grads(m)
    if T == 1:
        att = [k for k in grads if k.endswith("_attention")][0]
        assert float(grads[att].abs().max()) == 0.0, "d_attention must be exactly zero at one period"
        ref = dict(ref, grads={k: v for k, v in ref["grads"].items() if k != att})
    _check(w, ref, lims, loss, out, hid, grads, f"{model}/T={T}")


def test_65_periods_auto_runs_fp32_kernels():
    """``precision="auto"`` promises fp32-equivalent arithmetic at any period count: past the fused kernels' 64 it runs
    the FFMA kernels, for the training step and for the forward."""
    w = W.tiny_workload("RegionalTemporalGCN", N=60, T=65, H=128, O=3, R=3, B=2, seed=41)
    ref = oracle_step(w, 2)
    lims, _ = twin_limits(w, 2, ref)
    m = build_cuda(w, ref["state"], precision="auto")
    x, y = w.inputs(2)
    g = to_dev(w.graph_args(), "cuda")
    (loss, out, hid), names = profiled(lambda: m.fused_step(x.cuda(), y.cuda(), *g))
    assert "k_cell_fwd" in names and "k_cell_bwd" in names, sorted(names)
    assert not names & {"k_cell_fwd_f", "k_cell_bwd_f", "k_g_zr"}, sorted(names)
    _check(w, ref, lims, loss, out, hid, _grads(m), "T=65/auto")
    with torch.no_grad():
        out_f, hid_f = m(x.cuda(), *g)
    assert relerr(out_f, ref["out"]) <= TOL and relerr(hid_f, ref["hid"]) <= TOL


def test_65_periods_explicit_tf32x3_is_refused():
    w = W.tiny_workload("RegionalTemporalGCN", N=60, T=65, H=128, O=3, R=3, B=2, seed=41)
    m = build_cuda(w, build_oracle(w).state_dict(), precision="tf32x3")
    x, y = w.inputs(2)
    with pytest.raises(RuntimeError, match="up to 64 periods"):
        m.fused_step(x.cuda(), y.cuda(), *to_dev(w.graph_args(), "cuda"))
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------------------------
# 6. head limits
# ------------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _head_case(O, H, N=150, B=2):
    w = W.tiny_workload("RegionalTemporalGCN", N=N, T=3, H=H, O=O, R=3, B=B, seed=50 + O)
    ref = oracle_step(w, B)
    lims, _ = twin_limits(w, B, ref)
    return w, B, ref, lims


@pytest.mark.parametrize("path", ["fused_step", "autograd"])
@pytest.mark.parametrize("H", [64, 128])
@pytest.mark.parametrize("O", [15, 16, 17, 32])
def test_head_output_width(O, H, path):
    """k_hf_mid reduces up to 16 outputs by a halving shuffle exchange (out[o] on lanes 2o, 2o+1): O = 16 uses every
    lane.  Wider heads take the other head kernels (k_head_fused inside the fused step at H = 64, the FFMA row kernels
    with tensor-core weight gradients otherwise)."""
    w, B, ref, lims = _head_case(O, H)
    m = build_cuda(w, ref["state"], precision="tf32x3")
    x, y = w.inputs(B)
    x, y = x.cuda(), y.cuda()
    if path == "fused_step":
        res, names = profiled(lambda: m.fused_step(x, y, *to_dev(w.graph_args(), "cuda")))
    else:
        res, names = _profiled_autograd(lambda: m(x, *to_dev(w.graph_args(), "cuda")),
                                        lambda out, hid: ((out - y) ** 2).mean(dim=(1, 2)).sum())
    assert ("k_hf_mid" in names) == (O <= 16), sorted(names)
    if O > 16 and path == "fused_step" and H == 64:
        assert "k_head_fused" in names, sorted(names)
    for k in FUSED:
        assert k in names, (k, sorted(names))
    _check(w, ref, lims, *res, _grads(m), f"O={O}/H={H}/{path}")


@pytest.mark.parametrize("N", [127, 128])
def test_head_row_threshold(N):
    """route_of (api.cu) takes the tensor-core head from B*N = 128 rows on; 127 rows run the FFMA head.  Both meet the oracle."""
    w, B, ref, lims = _head_case(4, 128, N=N, B=1)
    m = build_cuda(w, ref["state"], precision="tf32x3")
    x, y = w.inputs(B)
    (loss, out, hid), names = profiled(lambda: m.fused_step(x.cuda(), y.cuda(), *to_dev(w.graph_args(), "cuda")))
    assert ("k_hf_mid" in names) == (N >= 128), sorted(names)
    _check(w, ref, lims, loss, out, hid, _grads(m), f"B*N={N}")


# ------------------------------------------------------------------------------------------------------------------
# 7. gradient through out_hidden
# ------------------------------------------------------------------------------------------------------------------
def _hidden_loss_oracle(w, B, c, with_mse, dtype):
    """the oracle, one [N,F,T] snapshot per call, loss_b = [mean((out_b - y_b)^2)] + <c_b, hid_b>, summed over b."""
    m = build_oracle(w, dtype)
    x, y = w.inputs(B)
    outs, hids, total = [], [], 0.0
    for b in range(B):
        out, hid = m(x[b].to(dtype), *w.graph_args())
        loss = (c[b].to(dtype) * hid).sum()
        if with_mse:
            loss = loss + torch.mean((out - y[b].to(dtype)) ** 2)
        loss.backward()
        outs.append(out.detach())
        hids.append(hid.detach())
        total += float(loss.detach())
    grads = {k: p.grad for k, p in m.named_parameters()}
    return dict(out=torch.stack(outs), hid=torch.stack(hids), loss=total, grads=grads, state=m.state_dict())


@pytest.mark.parametrize("with_mse", [True, False], ids=["mse_plus_hidden", "hidden_only"])
@pytest.mark.parametrize("H", [128, 64])
def test_loss_on_out_hidden(H, with_mse):
    """autograd with a loss on out_hidden: d_hidden is added to the head's G (k_hf_gmask) or, with no loss on out, copied
    into it (k_copy_or_zero), in the tile layout the fused backward reads.  c is scaled so both terms of the loss weigh alike."""
    N, B = 300, 3      # 900 rows: the last 128-row tile holds 4
    w = W.tiny_workload("RegionalTemporalGCN", N=N, T=4, H=H, O=3, R=5, B=B, seed=60 + H)
    c = (torch.rand(B, N, H, generator=torch.Generator().manual_seed(7), dtype=torch.float64) - 0.5) * (4.0 / (N * H))
    ref = _hidden_loss_oracle(w, B, c, with_mse, torch.float64)
    twin = _hidden_loss_oracle(w, B, c, with_mse, torch.float32)
    lims = {k: max(TOL, 4.0 * relerr(twin["grads"][k], gr)) for k, gr in ref["grads"].items() if gr is not None}
    m = build_cuda(w, ref["state"], precision="tf32x3")
    x, y = w.inputs(B)
    x, y, cd = x.cuda(), y.cuda(), c.float().cuda()

    def loss_of(out, hid):
        loss = (cd * hid).sum()
        return loss + ((out - y) ** 2).mean(dim=(1, 2)).sum() if with_mse else loss

    (loss, out, hid), names = _profiled_autograd(lambda: m(x, *to_dev(w.graph_args(), "cuda")), loss_of)
    for k in FUSED + (("k_hf_gmask",) if with_mse else ("k_copy_or_zero",)):
        assert k in names, (k, sorted(names))
    _check(w, ref, lims, loss, out, hid, _grads(m), f"H={H}/{'mse+' if with_mse else ''}hidden")
