"""node_features F from 1 to 8 on every cell path.  The kernels work at 8 features: x is read at its own width and the
features F..7 (and the matching columns of the collapsed weights) are written as zeros, so an F-feature model must compute
bit for bit what the 8-feature model computes on zero-padded x with zero-padded [H, F] weights.  That is checked first, on
each path at the shapes the benchmark runs; then parity with the fp64 oracle (which is F-general as written), the edges of
the new code (unaligned micro-batch slices of x, period limits, forward-only, graph replay, uninitialised workspace,
determinism) and the callers (region shards, the epoch loop, state_dict).  Every test asserts which kernels ran."""
import copy
import functools

import pytest
import torch

from parity_util import W, is_dead, profiled, relerr, to_dev

pytestmark = pytest.mark.gpu
TOL = 1e-5
BF16_ATOL, BF16_GTOL = 2e-2, 5e-2          # the stated bf16 tolerances (tests/test_gpu_bf16_edges.py)
PATH_KERNELS = {"fp32": ("k_cell_fwd", "k_widen_x"), "unfused": ("k_g_h", "k_widen_x"), "fused": ("k_cell_fwd_f", "k_feat_tc"),
                "bf16": ("k_cell_fwd_tc", "k_feat_tc")}


def _is_fw(key: str) -> bool:
    """the [H, F] parameters: conv_{z,r,h}.lin.weight of the TGCN cell and lins.{0,1}.weight of the ChebConv."""
    return key.endswith(".lin.weight") or ".conv.lins." in key


def _pad_state(state, F):
    return {k: (torch.nn.functional.pad(v, (0, 8 - F)) if _is_fw(k) else v) for k, v in state.items()}


def _pad_x(x):
    return torch.nn.functional.pad(x, (0, 0, 0, 8 - x.shape[2]))


def build_oracle_f(w, dtype=torch.float64, seed=1234):
    from oracle import regt_oracle as O
    torch.manual_seed(0)
    if w.model == "TemporalGCN":
        m = O.TemporalGCN(w.F, w.T, w.O, hidden=w.H)
    else:
        m = O.RegionalTemporalGCN(w.F, w.N, w.T, w.O, hidden=w.H, n_regions=w.R)
    W.init_params_synthetic(m, seed)
    return m.to(dtype)


def build_cuda_f(w, state, F=None, precision="fp32"):
    from models import RegionalTemporalGCN, TemporalGCN
    F = w.F if F is None else F
    if w.model == "TemporalGCN":
        m = TemporalGCN(F, w.T, w.O, hidden=w.H, precision=precision)
    else:
        m = RegionalTemporalGCN(F, w.N, w.T, w.O, hidden=w.H, n_regions=w.R, precision=precision)
    m.load_state_dict({k: v.float() for k, v in state.items()}, strict=True)
    return m.cuda()


def oracle_f(w, B, x, y, state=None, dtype=torch.float64):
    """fp64 (or fp32 twin) oracle step with x.grad: dict(out, hid, loss, grads, x_grad, state)."""
    from oracle import regt_oracle as O
    m = build_oracle_f(w, dtype)
    if state is not None:
        m.load_state_dict({k: v.to(dtype) for k, v in state.items()})
    xr = x.detach().to(dtype).clone().requires_grad_(True)
    out, hid, loss = O.batched_step(m, xr, y.to(dtype), w.graph_args())
    grads = {k: (None if p.grad is None else p.grad.detach().clone()) for k, p in m.named_parameters()}
    return dict(out=out, hid=hid, loss=loss, grads=grads, x_grad=xr.grad.detach().clone(),
                state=copy.deepcopy(m.state_dict()))


@functools.lru_cache(maxsize=None)
def _oracle_case(key):
    """(w, B, x, y, fp64 reference, per-gradient limits): limit = 1e-5 or 4x the fp32 twin's own error."""
    w, B = _PARITY_WORKLOADS[key[0]](key[1])
    x, y = w.inputs(B)
    ref = oracle_f(w, B, x, y)
    twin = oracle_f(w, B, x, y, ref["state"], torch.float32)
    lims = {k: max(TOL, 4.0 * relerr(twin["grads"][k], g)) for k, g in ref["grads"].items() if g is not None}
    lims["x"] = max(TOL, 4.0 * relerr(twin["x_grad"], ref["x_grad"]))
    return w, B, x, y, ref, lims


def _grads(m):
    return {k: (None if p.grad is None else p.grad.detach().clone()) for k, p in m.named_parameters()}


def _autograd(m, w, x, y, x_grad=True):
    """forward with autograd, backward of sum_b mean((out_b - y_b)^2); -> (loss, out, hid, grads, x.grad)."""
    xs = x.detach().cuda().requires_grad_(x_grad)
    out, hid = m(xs, *to_dev(w.graph_args(), "cuda"))
    loss = ((out - y.cuda()) ** 2).mean(dim=(-2, -1)).sum()
    loss.backward()
    torch.cuda.synchronize()
    return loss.detach(), out.detach(), hid.detach(), _grads(m), (xs.grad if x_grad else None)


def _fused(m, w, x, y, micro_batch=None):
    loss, out, hid = m.fused_step(x.cuda(), y.cuda(), *to_dev(w.graph_args(), "cuda"), micro_batch=micro_batch)
    torch.cuda.synchronize()
    return loss, out, hid, _grads(m), None


def _assert_kernels(names, path, F):
    for k in PATH_KERNELS[path]:
        if k == "k_widen_x" and F == 8:
            continue
        assert k in names, (path, k, sorted(names))


# ------------------------------------------------------------------------------------------------------------------
# 1. padding is exact
# ------------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _cfg5_full():
    return W.make_workload(5)


_PAD_CASES = {
    # name: (workload factory(F), B, precision, path, step kinds)
    "cfg2_fp32": (lambda F: W.make_workload(2), 64, "fp32", "fp32", ("autograd", "fused")),
    "cfg2_tf32x3_h64": (lambda F: W.make_workload(2), 64, "tf32x3", "fused", ("autograd", "fused")),
    "cfg2_bf16_h64": (lambda F: W.make_workload(2), 64, "bf16", "bf16", ("autograd", "fused")),
    "cfg5_shaped_tf32x3_h128": (lambda F: W.cfg5_shaped(), 2, "tf32x3", "fused", ("autograd", "fused")),
    "cfg5_shaped_fp32": (lambda F: W.cfg5_shaped(), 2, "fp32", "fp32", ("autograd", "fused")),
    "cfg5_shaped_tf32x3_h256_unfused": (lambda F: W.cfg5_shaped(H=256), 2, "tf32x3", "unfused", ("autograd", "fused")),
    "cfg5_full_tf32x3_b4": (lambda F: _cfg5_full(), 4, "tf32x3", "fused", ("fused",)),
}


@pytest.mark.parametrize("F", [1, 2, 3, 5, 7])
@pytest.mark.parametrize("case", list(_PAD_CASES))
def test_padding_is_exact(case, F):
    make, B, precision, path, kinds = _PAD_CASES[case]
    w = copy.copy(make(F))
    w.F = 8
    state8 = build_oracle_f(w, torch.float32).state_dict()
    state = {k: (v[:, :F].clone() if _is_fw(k) else v) for k, v in state8.items()}
    state8 = _pad_state(state, F)
    wF = copy.copy(w)
    wF.F = F
    x, y = wF.inputs(B)
    x8 = _pad_x(x)
    for kind in kinds:
        x_grad = kind == "autograd" and precision != "bf16"
        runs = []
        for FF, st, xx in ((F, state, x), (8, state8, x8)):
            m = build_cuda_f(w, st, FF, precision)
            fn = (lambda: _autograd(m, w, xx, y, x_grad)) if kind == "autograd" else (lambda: _fused(m, w, xx, y))
            res, names = profiled(fn)
            _assert_kernels(names, path, FF)
            if FF == 8:
                assert "k_widen_x" not in names
            runs.append(res)
        (lf, of, hf, gf, xgf), (l8, o8, h8, g8, xg8) = runs
        tag = f"{case}/{kind}/F={F}"
        assert torch.equal(lf, l8), f"{tag}: loss"
        assert torch.equal(of, o8), f"{tag}: out"
        assert torch.equal(hf, h8), f"{tag}: out_hidden"
        for k, g in gf.items():
            if g is None:
                assert g8[k] is None, (tag, k)
                continue
            ref = g8[k][:, :F] if _is_fw(k) else g8[k]
            assert g.shape == ref.shape and torch.equal(g, ref), f"{tag}: grad {k}"
        if x_grad:
            assert xgf.shape == x.shape and torch.equal(xgf, xg8[:, :, :F]), f"{tag}: x.grad"


# ------------------------------------------------------------------------------------------------------------------
# 2. oracle parity
# ------------------------------------------------------------------------------------------------------------------
_PARITY_WORKLOADS = {
    "regional_r5": lambda F: (W.tiny_workload("RegionalTemporalGCN", N=48, T=6, H=64, O=3, R=5, B=3, seed=21, adversarial=True,
                                              F=F), 3),
    "regional_r32": lambda F: (W.tiny_workload("RegionalTemporalGCN", N=160, T=4, H=64, O=3, R=32, B=2, seed=22, F=F), 2),
    "regional_r5_h96": lambda F: (W.tiny_workload("RegionalTemporalGCN", N=48, T=6, H=96, O=3, R=5, B=3, seed=23, F=F), 3),
    "a3tgcn": lambda F: (W.tiny_workload("TemporalGCN", N=40, T=6, H=64, O=3, R=0, B=3, seed=24, adversarial=True, F=F), 3),
    "regional_t1": lambda F: (W.tiny_workload("RegionalTemporalGCN", N=40, T=1, H=64, O=2, R=3, B=2, seed=25, F=F), 2),
    "regional_t64": lambda F: (W.tiny_workload("RegionalTemporalGCN", N=30, T=64, H=64, O=2, R=3, B=2, seed=26, F=F), 2),
}
_PARITY = [  # (workload, precision, path)
    ("regional_r5", "fp32", "fp32"), ("regional_r5", "tf32x3", "fused"), ("regional_r5_h96", "tf32x3", "unfused"),
    ("regional_r32", "tf32x3", "fused"), ("a3tgcn", "fp32", "fp32"), ("a3tgcn", "tf32x3", "fused"),
    ("regional_r5", "bf16", "bf16"), ("a3tgcn", "bf16", "bf16"),
    ("regional_t1", "tf32x3", "fused"), ("regional_t1", "fp32", "fp32"),
    ("regional_t64", "tf32x3", "fused"), ("regional_t64", "fp32", "fp32"),
]


def _check_oracle(w, ref, lims, res, tag, bf16=False):
    loss, out, hid, grads, x_grad = res
    atol = BF16_ATOL if bf16 else TOL
    assert relerr(hid, ref["hid"]) <= atol, f"{tag}: out_hidden {relerr(hid, ref['hid']):.3e}"
    assert relerr(out, ref["out"]) <= atol, f"{tag}: out {relerr(out, ref['out']):.3e}"
    assert abs(float(loss) - ref["loss"]) <= atol * abs(ref["loss"]), f"{tag}: loss"
    for k, g in ref["grads"].items():
        if g is None or is_dead(w.model, k):
            continue
        lim = BF16_GTOL if bf16 else (max(lims[k], 1e-4) if k.endswith("_attention") else lims[k])
        if bf16 and k.endswith("_attention"):
            lim = 0.15
        e = relerr(grads[k], g)
        assert e <= lim, f"{tag}: grad {k} {e:.3e} > {lim:.3e}"
    if x_grad is not None:
        e = relerr(x_grad, ref["x_grad"])
        assert e <= lims["x"], f"{tag}: x.grad {e:.3e} > {lims['x']:.3e}"


@pytest.mark.parametrize("kind", ["autograd", "fused"])
@pytest.mark.parametrize("F", [1, 2, 5])
@pytest.mark.parametrize("key,precision,path", _PARITY)
def test_modules_match_oracle(key, precision, path, F, kind, monkeypatch):
    monkeypatch.setenv("REGT_UNFUSED", "0")
    w, B, x, y, ref, lims = _oracle_case((key, F))
    m = build_cuda_f(w, ref["state"], precision=precision)
    bf16 = precision == "bf16"
    fn = (lambda: _autograd(m, w, x, y, not bf16)) if kind == "autograd" else (lambda: _fused(m, w, x, y))
    res, names = profiled(fn)
    _assert_kernels(names, path, F)
    assert (res[4] is not None) == (kind == "autograd" and not bf16)
    _check_oracle(w, ref, lims, res, f"{key}/{precision}/{kind}/F={F}", bf16)


@pytest.mark.parametrize("with_h", [False, True])
@pytest.mark.parametrize("F", [1, 2, 5])
def test_tgcn_cell_matches_oracle(F, with_h):
    """models.utils.TGCN(in_channels=F): H' and the gradients wrt the parameters, X and H."""
    from models.utils import TGCN
    from oracle import regt_oracle as O
    w = W.tiny_workload("TemporalGCN", N=50, T=1, H=32, O=1, R=0, B=1, seed=27, F=F)
    g = torch.Generator().manual_seed(5)
    X = torch.rand(w.N, F, generator=g)
    H0 = torch.rand(w.N, w.H, generator=g) - 0.5 if with_h else None
    c = torch.rand(w.N, w.H, generator=g) - 0.5
    res = {}
    for dt in (torch.float64, torch.float32):
        torch.manual_seed(0)
        om = O.TGCN(F, w.H).to(dt)
        W.init_params_synthetic(om, 1234)
        Xr = X.to(dt).clone().requires_grad_(True)
        Hr = None if H0 is None else H0.to(dt).clone().requires_grad_(True)
        out = om(Xr, w.edge_index, w.edge_attr, Hr)
        (c.to(dt) * out).sum().backward()
        res[dt] = (om, out.detach(), {k: p.grad for k, p in om.named_parameters()}, Xr.grad, None if Hr is None else Hr.grad)
    om, ref_out, ref_g, ref_xg, ref_hg = res[torch.float64]
    _, _, tw_g, tw_xg, tw_hg = res[torch.float32]
    m = TGCN(F, w.H).cuda()
    m.load_state_dict({k: v.float() for k, v in om.state_dict().items()}, strict=True)
    Xd = X.cuda().requires_grad_(True)
    Hd = None if H0 is None else H0.cuda().requires_grad_(True)

    def run():
        out = m(Xd, w.edge_index.cuda(), w.edge_attr.cuda(), Hd)
        (c.cuda() * out).sum().backward()
        torch.cuda.synchronize()
        return out.detach()
    out, names = profiled(run)
    assert "k_cell_fwd" in names and "k_widen_x" in names, sorted(names)
    assert relerr(out, ref_out) <= TOL
    pairs = [(p.grad, ref_g[k], tw_g[k], k) for k, p in m.named_parameters()] + [(Xd.grad, ref_xg, tw_xg, "X")]
    if with_h:
        pairs.append((Hd.grad, ref_hg, tw_hg, "H"))
    for got, ref, twin, k in pairs:
        lim = max(TOL, 4.0 * relerr(twin, ref))
        assert got.shape == ref.shape and relerr(got, ref) <= lim, f"F={F}: grad {k} {relerr(got, ref):.3e} > {lim:.3e}"


# ------------------------------------------------------------------------------------------------------------------
# 3. edges of the new code
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision,path", [("fp32", "fp32"), ("tf32x3", "fused")])
@pytest.mark.parametrize("mb", [1, 3])
def test_unaligned_micro_batches(mb, precision, path):
    """N = 207, F = 1, T = 6: one snapshot of x is 4968 bytes, so micro-batch slices start off 16-byte boundaries."""
    w = copy.copy(W.make_workload(2))
    w.F, w.T, w.B = 1, 6, 6
    x, y = w.inputs(6)
    assert (w.N * w.F * w.T * 4) % 16 != 0
    state = build_oracle_f(w, torch.float32).state_dict()
    whole = _fused(build_cuda_f(w, state, precision=precision), w, x, y)
    m = build_cuda_f(w, state, precision=precision)
    res, names = profiled(lambda: _fused(m, w, x, y, micro_batch=mb))
    _assert_kernels(names, path, 1)
    assert relerr(res[0], whole[0]) <= 1e-6
    assert relerr(res[1], whole[1]) <= 1e-6 and relerr(res[2], whole[2]) <= 1e-6
    for k, g in whole[3].items():     # the micro-batches add their gradients in another order
        if g is not None:
            assert relerr(res[3][k], g) <= (1e-4 if k.endswith("_attention") else 1e-5), k
    ref = oracle_f(w, 6, x, y, state)
    _check_oracle(w, ref, {k: 1e-4 for k in list(ref["grads"]) + ["x"]}, res, f"mb={mb}/{precision}")


@pytest.mark.parametrize("precision,path", [("fp32", "fp32"), ("tf32x3", "fused"), ("tf32x3_h96", "unfused"), ("bf16", "bf16")])
def test_forward_only_matches_autograd_forward(precision, path):
    H = 96 if precision == "tf32x3_h96" else 64
    precision = precision.split("_")[0]
    w = W.tiny_workload("RegionalTemporalGCN", N=120, T=6, H=H, O=3, R=4, B=3, seed=31, F=2)
    x, y = w.inputs(3)
    m = build_cuda_f(w, build_oracle_f(w, torch.float32).state_dict(), precision=precision)
    g = to_dev(w.graph_args(), "cuda")
    with torch.no_grad():
        (out0, hid0), names = profiled(lambda: m(x.cuda(), *g))
    _assert_kernels(names, path, 2)
    out1, hid1 = m(x.cuda(), *g)
    assert out1.requires_grad
    assert torch.equal(out0, out1.detach()) and torch.equal(hid0, hid1.detach())


@pytest.mark.parametrize("precision,path", [("fp32", "fp32"), ("tf32x3", "fused"), ("bf16", "bf16")])
def test_graph_replay_and_determinism(precision, path):
    """fused_step captured in a CUDA graph: each replay equals an eager step bit for bit, and two eager steps agree."""
    w = W.tiny_workload("RegionalTemporalGCN", N=300, T=4, H=64, O=4, R=5, B=4, seed=33, F=2)
    x, y = w.inputs(4)
    xs, ys = x.cuda(), y.cuda()
    g = to_dev(w.graph_args(), "cuda")
    m = build_cuda_f(w, build_oracle_f(w, torch.float32).state_dict(), precision=precision)

    def step():
        for p in m.parameters():
            if p.grad is not None:
                p.grad.zero_()
        return m.fused_step(xs, ys, *g, micro_batch=2)

    def snap(res):
        torch.cuda.synchronize()
        return [t.clone() for t in res] + [p.grad.clone() for p in m.parameters() if p.grad is not None]

    e1, names = profiled(lambda: snap(step()))
    _assert_kernels(names, path, 2)
    e2 = snap(step())
    assert all(torch.equal(a, b) for a, b in zip(e1, e2)), "two eager steps differ"
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static = step()
    for _ in range(2):
        for p in m.parameters():
            if p.grad is not None:
                p.grad.zero_()
        graph.replay()
        r = snap(static)
        assert all(torch.equal(a, b) for a, b in zip(r, e1)), "replay differs from the eager step"


@pytest.mark.parametrize("precision,path,H", [("fp32", "fp32", 64), ("tf32x3", "unfused", 96), ("tf32x3", "fused", 64)])
def test_poisoned_workspace_and_scratch(precision, path, H):
    """a NaN-filled workspace (widened x included) and x-gradient scratch give the same step as zeroed ones: the pad
    features and weight columns are written by every step, never left to whatever the allocator hands out."""
    from regt_b200 import _lib, engine
    import ctypes as C
    w = W.tiny_workload("RegionalTemporalGCN", N=200, T=4, H=H, O=3, R=4, B=3, seed=35, F=3)
    x, y = w.inputs(3)
    x, y = x.cuda(), y.cuda()
    g = to_dev(w.graph_args(), "cuda")
    m = build_cuda_f(w, build_oracle_f(w, torch.float32).state_dict(), precision=precision)
    plan = m._plan(x, g[0], g[1:])
    prec, params = m._prec(w.T), m._param_dict()
    lib = _lib.load()
    R = max(w.R, 1)

    def run(poison):
        st = engine.build_state(m._mode, prec, plan, x, w.H, w.O, params)
        nbytes = st.args.workspace_bytes
        ws = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
        if poison:
            ws[:nbytes - (-(-4 * (R + 2) // 256) * 256)].fill_(0xFF)    # all but the int32 chunk table carved last
        st = engine.build_state(m._mode, prec, plan, x, w.H, w.O, params, workspace=ws)
        engine.run_forward(st, True)
        d_out = (2.0 / (w.N * w.O)) * (st.out - y)
        grads = {k: torch.empty_like(t) for k, t in params.items()}
        engine.run_backward(st, grads, d_out, None, False, True)
        xp = plan.xgrad_struct()
        a = st.args
        nb = lib.regt_cell_backward_x_scratch_bytes(C.byref(a), C.byref(xp))
        scratch = torch.full((nb,), 0xFF if poison else 0, dtype=torch.uint8, device="cuda")
        d_x = torch.full_like(x, float("nan"))
        a.stream = torch.cuda.current_stream().cuda_stream
        _lib.check(lib.regt_cell_backward_x(C.byref(a), C.byref(xp), d_x.data_ptr(), scratch.data_ptr(), nb),
                   "regt_cell_backward_x")
        torch.cuda.synchronize()
        return [st.out, st.out_hidden, d_x] + [grads[k] for k in sorted(grads)]

    res_p, names = profiled(lambda: run(True))
    _assert_kernels(names, path, 3)
    assert "k_xg_layout" in names
    res_z = run(False)
    for a, b in zip(res_p, res_z):
        assert torch.isfinite(a).all() and torch.equal(a, b)


# ------------------------------------------------------------------------------------------------------------------
# 4. callers
# ------------------------------------------------------------------------------------------------------------------
def test_sum_of_region_shards_at_two_features():
    """config 5's generator (R = 256) at F = 2 as 8 region shards run one after the other: outputs scatter back to global
    order, losses and gradients add up to the unsharded fp64 oracle."""
    from regt_b200 import shard as S
    w = W.cfg5_shaped()
    w.F = 2
    B = 2
    x, y = w.inputs(B)
    ref = oracle_f(w, B, x, y)
    twin = oracle_f(w, B, x, y, ref["state"], torch.float32)
    lims = {k: max(TOL, 4.0 * relerr(twin["grads"][k], g)) for k, g in ref["grads"].items() if g is not None}
    lims["x"] = 1.0
    xd, yd = x.cuda(), y.cuda()
    ei, reis, reas = w.edge_index.cuda(), [e.cuda() for e in w.reg_edge_index], [a.cuda() for a in w.reg_edge_attr]
    loss_sum, grad_sum = 0.0, {}
    out_full = torch.zeros(B, w.N, w.O, device="cuda")
    hid_full = torch.zeros(B, w.N, w.H, device="cuda")
    for rank in range(8):
        m = build_cuda_f(w, ref["state"], precision="tf32x3")
        sm = S.RegionShardedModel(m, ei, reis, reas, rank, 8)
        (loss, out, hid), names = profiled(lambda: sm.fused_step(xd, yd, sync=False))
        assert "k_feat_tc" in names, sorted(names)
        loss_sum += float(loss)
        S.scatter_rows(out, sm.own, out_full)
        S.scatter_rows(hid, sm.own, hid_full)
        for k, p in m.named_parameters():
            if p.grad is not None:
                grad_sum[k] = p.grad.double().cpu() + grad_sum.get(k, 0.0)
    _check_oracle(w, ref, lims, (loss_sum, out_full, hid_full, grad_sum, None), "shards8/F=2")


@pytest.mark.parametrize("model_name", ["RegionalTemporalGCN", "TemporalGCN"])
def test_epoch_and_evaluate_at_two_features(model_name):
    """one epoch of run.py over device-resident windows of node_data [N, 2, T_total] and predict.py's metrics, against
    the oracle loop on the same series."""
    from oracle import loop_oracle as LO
    from regt_b200.loop import FlatRMSprop, SlidingWindows, evaluate, train_epoch
    w = W.tiny_workload(model_name, N=30, T=6, H=32, O=3, R=3 if model_name == "RegionalTemporalGCN" else 0, B=1, seed=11,
                        F=2)
    nd = torch.rand(w.N, 2, 6 + 3 + 8, generator=torch.Generator().manual_seed(5))
    ref = build_oracle_f(w, torch.float64)
    state = copy.deepcopy(ref.state_dict())
    feats, targ = LO.windows(nd.double(), 6, 3)
    ref_grads = {}
    last_ref, total_ref = LO.train_epoch(ref, feats, targ, w.graph_args(), _Spy(torch.optim.RMSprop(ref.parameters(), lr=1e-3),
                                                                               ref, ref_grads))
    m = build_cuda_f(w, state, precision="fp32")
    gargs = to_dev(w.graph_args(), "cuda")
    sw = SlidingWindows(nd.cuda(), 6, 3)
    grads = {}
    (last, total), names = profiled(lambda: train_epoch(m, sw, gargs, _Spy(FlatRMSprop(list(m.parameters()), lr=1e-3), m, grads),
                                                        batch=4))
    assert "k_widen_x" in names, sorted(names)
    assert abs(float(last) - float(last_ref)) <= 1e-5 * abs(float(last_ref))
    assert abs(float(total) - float(total_ref)) <= 1e-5 * abs(float(total_ref))
    for k, g in ref_grads.items():        # the epoch's accumulated gradients, right before the optimizer step
        if not is_dead(w.model, k):
            assert relerr(grads[k], g) <= 1e-5, k
    mae, rmse, mape = evaluate(m, sw, gargs, batch=4)
    with torch.no_grad():
        x, y = sw.gather(torch.arange(len(sw), device="cuda"))
        outs = m(x, *gargs)[0]
    rmae, rrmse, rmape = LO.predict_metrics(list(outs.cpu()), list(y.cpu()))
    assert abs(mae - rmae) <= 1e-5 * rmae and abs(rmse - rrmse) <= 1e-5 * rrmse and abs(mape - rmape) <= 1e-5 * abs(rmape)


class _Spy:
    """records the accumulated gradients right before the optimizer step"""

    def __init__(self, opt, model, store):
        self.opt, self.model, self.store = opt, model, store

    def zero_grad(self):
        self.opt.zero_grad()

    def step(self):
        for k, p in self.model.named_parameters():
            if p.grad is not None:
                self.store[k] = p.grad.detach().clone()
        self.opt.step()


def test_state_dict_round_trip_at_two_features():
    from models import RegionalTemporalGCN
    w = W.tiny_workload("RegionalTemporalGCN", N=40, T=4, H=64, O=2, R=3, B=2, seed=37, F=2)
    a = build_cuda_f(w, build_oracle_f(w, torch.float32).state_dict(), precision="tf32x3")
    sd = a.state_dict()
    assert tuple(sd["tgnn._base_tgcn.conv_z.lin.weight"].shape) == (64, 2)
    assert tuple(sd["tgnn.conv.lins.1.weight"].shape) == (64, 2)
    b = RegionalTemporalGCN(2, w.N, w.T, w.O, hidden=64, n_regions=3, precision="tf32x3").cuda()
    b.load_state_dict(sd, strict=True)
    x, _ = w.inputs(2)
    g = to_dev(w.graph_args(), "cuda")
    with torch.no_grad():
        (oa, ha), names = profiled(lambda: a(x.cuda(), *g))
        ob, hb = b(x.cuda(), *g)
    assert "k_feat_tc" in names
    assert torch.equal(oa, ob) and torch.equal(ha, hb)
    with pytest.raises(ValueError, match="built for 2"):
        b(_pad_x(x).cuda(), *g)
