"""The gradient wrt the input features x (regt_cell_backward_x) against the fp64 oracle, which is pure torch and
differentiates through x as written.  Bound: 1e-5 normwise, or 4x the fp32 twin's own x.grad error (as
parity_util.twin_limits does for parameters).  Every parity test asserts which kernels ran, so a silent fallback
cannot pass for the path.  Then the properties the feature promises beside its values: parameter gradients and
launches unchanged by it, determinism, no read of uninitialised workspace, the transposed operator bit for bit
against a numpy construction, CUDA-graph replay, and the refusals."""
import ctypes as C

import numpy as np
import pytest
import torch

from parity_util import W, build_cuda, build_oracle, relerr, to_dev

pytestmark = pytest.mark.gpu
TOL = 1e-5
XG = ("k_xg_contract", "k_xg_layout")
PATH_KERNELS = {"fp32": ("k_cell_bwd",), "fused": ("k_cell_fwd_f", "k_cell_bwd_f"), "unfused": ("k_g_b1", "k_g_b3")}


def _find_node(t):
    """the autograd node of the kernels' Function behind ``t``."""
    seen, todo = set(), [t.grad_fn]
    while todo:
        n = todo.pop()
        if n is None or n in seen:
            continue
        seen.add(n)
        if "_ModelFn" in type(n).__name__:
            return n
        todo += [f for f, _ in n.next_functions]
    raise AssertionError("no _ModelFn node behind the output")


def _profiled_backward(forward, loss_of):
    """``forward()`` -> output(s), then ``loss_of(outputs).backward()``; returns (outputs, kernel names of the forward
    and of the backward).  Autograd runs the node's backward on its own thread and the recorder is per thread, so hooks
    on that node switch the recorder on and off around it there."""
    from regt_b200 import _lib
    lib = _lib.load()
    torch.cuda.synchronize()
    lib.regt_profile(1, torch.cuda.current_stream().cuda_stream)
    try:
        outs = forward()
        torch.cuda.synchronize()
        fwd = [n for n, _ in _lib.profile_read()]
    finally:
        lib.regt_profile(0, None)
    bwd = []

    def pre(grad_outputs):
        lib.regt_profile(1, torch.cuda.current_stream().cuda_stream)

    def post(grad_inputs, grad_outputs):
        torch.cuda.synchronize()
        bwd.extend(n for n, _ in _lib.profile_read())
        lib.regt_profile(0, None)

    node = _find_node(outs[0] if isinstance(outs, tuple) else outs)
    hooks = [node.register_prehook(pre), node.register_hook(post)]
    try:
        loss_of(outs).backward()
        torch.cuda.synchronize()
    finally:
        for h in hooks:
            h.remove()
    return outs, fwd, bwd


def _weights(B, N, H, seed=7):
    return (torch.rand(B, N, H, generator=torch.Generator().manual_seed(seed), dtype=torch.float64) - 0.5) * (4.0 / (N * H))


def _loss(kind, out, hid, y, c):
    """per snapshot: mean((out - y)^2) ('out'), <c, out_hidden> ('hidden') or both, summed over the batch."""
    total = 0
    if kind in ("out", "both"):
        total = total + ((out - y) ** 2).mean(dim=(-2, -1)).sum()
    if kind in ("hidden", "both"):
        total = total + (c * hid).sum()
    return total


def _oracle_xgrad(w, B, kind, dtype):
    """x.grad and the parameter gradients of the oracle, one [N,F,T] snapshot per call as the reference runs it."""
    m = build_oracle(w, dtype)
    x, y = w.inputs(B)
    c = _weights(B, w.N, w.H)
    xd = x.to(dtype).requires_grad_()
    for b in range(B):
        out, hid = m(xd[b], *w.graph_args())
        _loss(kind, out, hid, y[b].to(dtype), c[b].to(dtype)).backward()
    return xd.grad.detach(), {k: p.grad for k, p in m.named_parameters()}, m.state_dict()


_CASES = {
    # (workload, B, precision, path, loss).  B*N below is never a multiple of 128.
    # adversarial graphs: weighted self-loops, duplicate edges, an isolated node (in no regional list), a node in two lists
    "regional_fp32": (lambda: W.tiny_workload("RegionalTemporalGCN", N=40, T=6, H=64, O=2, R=5, B=3, seed=5, adversarial=True),
                      3, "fp32", "fp32", "both"),
    "regional_fused_h128": (lambda: W.tiny_workload("RegionalTemporalGCN", N=300, T=4, H=128, O=4, R=5, B=3, seed=9,
                                                    adversarial=True), 3, "tf32x3", "fused", "out"),
    "regional_fused_h64": (lambda: W.tiny_workload("RegionalTemporalGCN", N=150, T=3, H=64, O=5, R=5, B=3, seed=31,
                                                   adversarial=True), 3, "tf32x3", "fused", "hidden"),
    "regional_unfused_h256": (lambda: W.tiny_workload("RegionalTemporalGCN", N=60, T=3, H=256, O=3, R=3, B=2, seed=12,
                                                      adversarial=True), 2, "tf32x3", "unfused", "both"),
    # config 5's generator: R = 256 regions of 4 nodes, one 128-row tile spans ~30 regions
    "cfg5_shaped_fused": (lambda: W.cfg5_shaped(N=1000, T=2, H=128, R=256), 2, "tf32x3", "fused", "out"),
    # config 2's shape: the edge weights reach both gcn_norm and the ChebConv
    "a3tgcn_cfg2_fp32": (lambda: W.tiny_workload("TemporalGCN", N=207, T=12, H=64, O=12, R=0, B=2, seed=102,
                                                 k_intra=8, adversarial=True), 2, "fp32", "fp32", "both"),
    "a3tgcn_cfg2_fused": (lambda: W.tiny_workload("TemporalGCN", N=207, T=12, H=64, O=12, R=0, B=2, seed=102,
                                                  k_intra=8, adversarial=True), 2, "tf32x3", "fused", "out"),
    "regional_T1_fused": (lambda: W.tiny_workload("RegionalTemporalGCN", N=70, T=1, H=128, O=3, R=3, B=2, seed=41,
                                                  adversarial=True), 2, "tf32x3", "fused", "both"),
    "regional_T64_fused": (lambda: W.tiny_workload("RegionalTemporalGCN", N=50, T=64, H=64, O=3, R=3, B=2, seed=42,
                                                   adversarial=True), 2, "tf32x3", "fused", "out"),
    "regional_T65_fp32": (lambda: W.tiny_workload("RegionalTemporalGCN", N=50, T=65, H=64, O=3, R=3, B=2, seed=43,
                                                  adversarial=True), 2, "fp32", "fp32", "out"),
}


def _run_cuda(w, B, precision, kind, state, x=None, frozen=False):
    m = build_cuda(w, state, precision=precision)
    if frozen:
        m.requires_grad_(False)
    xs, y = w.inputs(B)
    x = (xs.cuda() if x is None else x).detach().requires_grad_()
    y, c = y.cuda(), _weights(B, w.N, w.H).float().cuda()
    g = to_dev(w.graph_args(), "cuda")
    _, fwd, bwd = _profiled_backward(lambda: m(x, *g), lambda o: _loss(kind, o[0], o[1], y.to(o[0].dtype), c.to(o[0].dtype)))
    return m, x.grad, fwd + bwd


def _assert_kernels(names, path):
    for k in PATH_KERNELS[path] + XG:
        assert k in names, (k, sorted(set(names)))
    assert "k_spmm_blk" in names or "k_spmm_rows" in names, sorted(set(names))


@pytest.mark.parametrize("case", list(_CASES))
def test_input_grad_matches_oracle(case):
    make, B, precision, path, kind = _CASES[case]
    w = make()
    ref, _, state = _oracle_xgrad(w, B, kind, torch.float64)
    twin, _, _ = _oracle_xgrad(w, B, kind, torch.float32)
    lim = max(TOL, 4.0 * relerr(twin, ref))
    _, xg, names = _run_cuda(w, B, precision, kind, state)
    _assert_kernels(names, path)
    e = relerr(xg, ref)
    assert e <= lim, f"{case}: x.grad {e:.3e} > {lim:.3e}"


def test_unbatched_float64_input_and_frozen_model():
    """x given as one [N,F,T] snapshot in float64 (the reference's call form), and a model with no parameter that
    requires grad (saliency): x.grad arrives in x's dtype and shape and meets the oracle."""
    w = W.tiny_workload("RegionalTemporalGCN", N=300, T=4, H=128, O=4, R=5, B=1, seed=9, adversarial=True)
    ref, _, state = _oracle_xgrad(w, 1, "out", torch.float64)
    twin, _, _ = _oracle_xgrad(w, 1, "out", torch.float32)
    lim = max(TOL, 4.0 * relerr(twin, ref))
    x, y = w.inputs(1)
    for precision, path in (("tf32x3", "fused"), ("fp32", "fp32")):
        m = build_cuda(w, state, precision=precision).requires_grad_(False)
        x64 = x[0].double().cuda().requires_grad_()
        yd = y[0].double().cuda()
        g = to_dev(w.graph_args(), "cuda")
        (out, hid), fwd, bwd = _profiled_backward(lambda: m(x64, *g), lambda o: ((o[0] - yd) ** 2).mean())
        _assert_kernels(fwd + bwd, path)
        assert x64.grad.dtype == torch.float64 and x64.grad.shape == x64.shape
        assert all(p.grad is None for p in m.parameters())
        assert relerr(x64.grad, ref[0]) <= lim, (path, relerr(x64.grad, ref[0]), lim)


# ------------------------------------------------------------------------------------------------------------------
# models.utils.TGCN: dX beside dH
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("with_h", [True, False], ids=["X_and_H", "H_None"])
def test_tgcn_cell_gives_dX(with_h):
    from oracle import regt_oracle as O
    from models.utils import TGCN
    N, Hd = 150, 32
    w = W.tiny_workload("TemporalGCN", N=N, T=1, H=Hd, O=1, R=0, B=1, seed=77, adversarial=True)
    gen = torch.Generator().manual_seed(5)
    X = torch.rand(N, 8, generator=gen, dtype=torch.float64)
    H0 = torch.rand(N, Hd, generator=gen, dtype=torch.float64) - 0.5 if with_h else None
    c = torch.rand(N, Hd, generator=gen, dtype=torch.float64) - 0.5

    def oracle(dtype):
        torch.manual_seed(0)
        m = O.TGCN(8, Hd)
        W.init_params_synthetic(m, 1234)
        m = m.to(dtype)
        Xd = X.to(dtype).clone().requires_grad_()
        Hd_ = None if H0 is None else H0.to(dtype).clone().requires_grad_()
        (c.to(dtype) * m(Xd, w.edge_index, w.edge_attr.to(dtype), Hd_)).sum().backward()
        return Xd.grad, (None if Hd_ is None else Hd_.grad), m.state_dict()

    rX, rH, state = oracle(torch.float64)
    tX, tH, _ = oracle(torch.float32)
    cell = TGCN(8, Hd, precision="fp32")
    cell.load_state_dict({k: v.float() for k, v in state.items()}, strict=True)
    cell = cell.cuda()
    Xc = X.float().cuda().requires_grad_()
    Hc = None if H0 is None else H0.float().cuda().requires_grad_()
    cd = c.float().cuda()
    ei, ew = w.edge_index.cuda(), w.edge_attr.cuda()
    _, fwd, bwd = _profiled_backward(lambda: cell(Xc, ei, ew, Hc), lambda o: (cd * o).sum())
    _assert_kernels(fwd + bwd, "fp32")
    assert relerr(Xc.grad, rX) <= max(TOL, 4.0 * relerr(tX, rX)), relerr(Xc.grad, rX)
    if with_h:
        assert relerr(Hc.grad, rH) <= max(TOL, 4.0 * relerr(tH, rH)), relerr(Hc.grad, rH)


# ------------------------------------------------------------------------------------------------------------------
# properties beside the values
# ------------------------------------------------------------------------------------------------------------------
_SMALL = lambda: W.tiny_workload("RegionalTemporalGCN", N=300, T=4, H=128, O=4, R=5, B=3, seed=9, adversarial=True)  # noqa: E731


@pytest.mark.parametrize("precision", ["tf32x3", "fp32"])
def test_x_grad_changes_nothing_else(precision, monkeypatch):
    """with x requiring grad the parameter gradients are bitwise those without, and the launches are those without
    followed by the input-gradient kernels; with x not requiring grad the workspace request is unchanged."""
    from regt_b200 import engine
    w = _SMALL()
    state = build_oracle(w).state_dict()
    sizes = []
    real = engine.build_state

    def spy(*a, **kw):
        st = real(*a, **kw)
        sizes.append(st.args.workspace_bytes)
        return st
    monkeypatch.setattr(engine, "build_state", spy)
    runs = {}
    for xg in (False, True):
        m = build_cuda(w, state, precision=precision)
        x, y = w.inputs(3)
        x, y = x.cuda().requires_grad_(xg), y.cuda()
        g = to_dev(w.graph_args(), "cuda")
        m(x, *g)                 # plan (and, with x grad, its transposed operator) outside the recorded window
        _, fwd, bwd = _profiled_backward(lambda: m(x, *g), lambda o: ((o[0] - y) ** 2).mean(dim=(1, 2)).sum())
        runs[xg] = (fwd, bwd, {k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None}, x.grad)
    (f0, b0, g0, xg0), (f1, b1, g1, xg1) = runs[False], runs[True]
    assert xg0 is None and xg1 is not None
    assert f0 == f1
    assert b1[:len(b0)] == b0 and not set(b0) & set(XG), (b0, b1)
    assert set(b1[len(b0):]) <= {"k_xg_m1h", "k_spmm_blk", "k_spmm_rows"} | set(XG) and set(XG) <= set(b1[len(b0):])
    assert g0.keys() == g1.keys() and all(torch.equal(g0[k], g1[k]) for k in g0)
    assert len(set(sizes)) == 1, sizes


def test_two_backwards_are_bitwise_identical():
    w = W.cfg5_shaped(N=1000, T=2, H=128, R=256)
    state = build_oracle(w).state_dict()
    grads = [_run_cuda(w, 3, "tf32x3", "both", state)[1] for _ in range(2)]
    assert torch.isfinite(grads[0]).all() and torch.equal(grads[0], grads[1])


@pytest.mark.parametrize("precision,unfused,path", [("tf32x3", "0", "fused"), ("tf32x3", "1", "unfused"), ("fp32", "0", "fp32")])
def test_poisoned_workspace_and_scratch_give_the_same_x_grad(precision, unfused, path, monkeypatch):
    """forward, backward and backward_x on a workspace and scratch whose bytes start as all-ones (NaN in every float
    slot) and on zeroed ones: the same finite x.grad.  The pad rows of the last 128-row tile must never be read.  The
    int32 dM1 chunk table at the end of the workspace is left zero (it indexes other buffers)."""
    from regt_b200 import _lib, engine
    monkeypatch.setenv("REGT_UNFUSED", unfused)
    lib = _lib.load()
    w = _SMALL()
    m = build_cuda(w, build_oracle(w).state_dict(), precision=precision)
    x, y = w.inputs(3)
    x, y = x.cuda(), y.cuda()
    g = to_dev(w.graph_args(), "cuda")
    plan = m._plan(x, g[0], g[1:])
    params = m._param_dict()
    xp = plan.xgrad_struct()
    res = []
    for poison in (True, False):
        st = engine.build_state(m._mode, m._prec(w.T), plan, x, w.H, w.O, params)
        nbytes = st.args.workspace_bytes
        ws = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
        tail = -(-4 * (w.R + 2) // 256) * 256
        if poison:
            ws[:nbytes - tail].fill_(0xFF)
        st = engine.build_state(m._mode, m._prec(w.T), plan, x, w.H, w.O, params, workspace=ws)
        lib.regt_profile(1, torch.cuda.current_stream().cuda_stream)
        try:
            engine.run_forward(st, True)
            d_out = (2.0 / (w.N * w.O)) * (st.out - y)
            engine.run_backward(st, {k: torch.empty_like(t) for k, t in params.items()}, d_out, None, False, True)
            sb = lib.regt_cell_backward_x_scratch_bytes(C.byref(st.args), C.byref(xp))
            scratch = torch.full((sb,), 0xFF if poison else 0, dtype=torch.uint8, device="cuda")
            d_x = torch.full_like(x, float("nan"))
            _lib.check(lib.regt_cell_backward_x(C.byref(st.args), C.byref(xp), d_x.data_ptr(), scratch.data_ptr(), sb),
                       "regt_cell_backward_x")
            torch.cuda.synchronize()
            names = [n for n, _ in _lib.profile_read()]
        finally:
            lib.regt_profile(0, None)
        _assert_kernels(names, path)
        res.append(d_x)
    assert torch.isfinite(res[0]).all() and torch.equal(res[0], res[1])


def test_transposed_operator_is_the_numpy_construction():
    """regt_xgrad_plan bit for bit against a stable argsort by input node of [identity | A_hat entries | regional
    entries], each in canonical CSR order."""
    w = W.tiny_workload("RegionalTemporalGCN", N=200, T=2, H=64, O=2, R=5, B=1, seed=5, adversarial=True)
    m = build_cuda(w, build_oracle(w).state_dict(), precision="fp32")
    g = to_dev(w.graph_args(), "cuda")
    x = torch.zeros(1, w.N, 8, 2, device="cuda")
    plan = m._plan(x, g[0], g[1:])
    xp = plan.xgrad_struct()
    torch.cuda.synchronize()
    t = {k: v.cpu().numpy() for k, v in plan.t.items()}
    N, ng, nc, nseg = plan.N, plan.nnz_gcn, plan.nnz_cheb, plan.nseg
    assert nc > 0 and nseg > 0
    g_dst = np.repeat(np.arange(N), np.diff(t["g_rowptr"]))
    c_seg = np.repeat(np.arange(nseg), np.diff(t["seg_eptr"][:nseg + 1]))
    key = np.concatenate([np.arange(N), t["g_col"][:ng], t["c_col"][:nc]])
    src = np.concatenate([np.arange(N), N + g_dst, 2 * N + c_seg]).astype(np.int32)
    val = np.concatenate([np.ones(N, np.float32), t["g_val"][:ng], t["c_val"][:nc]])
    order = np.argsort(key, kind="stable")
    rowptr = np.concatenate([[0], np.cumsum(np.bincount(key, minlength=N))]).astype(np.int32)
    assert (xp.N, xp.nnz, xp.n_src) == (N, N + ng + nc, 2 * N + nseg)
    np.testing.assert_array_equal(plan.xg["rowptr"].cpu().numpy(), rowptr)
    np.testing.assert_array_equal(plan.xg["col"].cpu().numpy(), src[order])
    assert plan.xg["val"].cpu().numpy().tobytes() == val[order].tobytes()


def test_graph_replay_of_forward_and_backward_with_x_grad():
    """after one eager step (which builds the plan and its transposed operator), forward + backward with x requiring
    grad captured in a CUDA graph replays bit for bit, also after x changes in place."""
    w = _SMALL()
    m = build_cuda(w, build_oracle(w).state_dict(), precision="tf32x3").requires_grad_(False)
    x, y = w.inputs(3)
    xs, ys = x.cuda().requires_grad_(), y.cuda()
    g = to_dev(w.graph_args(), "cuda")

    def step():
        out, hid = m(xs, *g)
        (gx,) = torch.autograd.grad(((out - ys) ** 2).mean(dim=(1, 2)).sum(), xs)
        return gx

    eager0 = step().clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        st_gx = step()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(st_gx, eager0)
    with torch.no_grad():
        xs.copy_(w.inputs(3, seed_offset=1)[0])
    graph.replay()
    torch.cuda.synchronize()
    eager1 = step()
    assert not torch.equal(eager1, eager0) and torch.equal(st_gx, eager1)


def test_bf16_and_shard_plans_are_refused_at_the_forward():
    from regt_b200 import engine, shard
    w = W.tiny_workload("TemporalGCN", N=150, T=12, H=64, O=12, R=0, B=1, seed=7, k_intra=5)
    m = build_cuda(w, build_oracle(w).state_dict(), precision="bf16")
    x = w.inputs(1)[0].cuda().requires_grad_()
    with pytest.raises(RuntimeError, match="not available in precision bf16"):
        m(x, *to_dev(w.graph_args(), "cuda"))
    with torch.no_grad():          # inference is unaffected
        m(x, *to_dev(w.graph_args(), "cuda"))

    w = W.tiny_workload("RegionalTemporalGCN", N=120, T=3, H=64, O=2, R=4, B=1, seed=3, n_cross=40)
    m = build_cuda(w, build_oracle(w).state_dict(), precision="fp32")
    sh = shard.make_shard(w.N, w.edge_index, w.reg_edge_index, 0, 2)
    plan = shard.build_local_plan(sh, torch.device("cuda"), w.edge_index.cuda(), None, [e.cuda() for e in w.reg_edge_index],
                                  [a.cuda() for a in w.reg_edge_attr])
    assert plan.n_halo > 0
    xl = torch.rand(1, sh.n_own + sh.n_halo, 8, 3, device="cuda", requires_grad=True)
    with pytest.raises(RuntimeError, match="region shards"):
        engine.model_apply(m._mode, m._prec(3), plan, w.H, w.O, xl, m._param_dict(), None, True)
