"""train_epoch / evaluate with share_periods=True (regt_b200/loop.py, csrc/combine.cu): the cell runs once per time step of
a pass and the windows combine the steps, against the windowed epoch on the same state and series and against the fp64
epoch of oracle/loop_oracle.py."""
import copy
import os

import pytest
import torch

from parity_util import W, build_cuda, build_oracle, is_dead, relerr, to_dev

pytestmark = pytest.mark.gpu


def _series(N, F, T_total, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(N, F, T_total, generator=g)          # MinMax-scaled features (load_dataset.py:430)


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


def _epoch(m, sw, gargs, share, **kw):
    """one epoch from the model's current state; returns (gradients before the step, last loss, total) and restores the
    parameters, so that the next call starts from the same state"""
    from regt_b200.loop import FlatRMSprop, train_epoch
    saved = {k: v.detach().clone() for k, v in m.state_dict().items()}
    opt = FlatRMSprop(list(m.parameters()), lr=1e-3)
    grads = {}
    last, total = train_epoch(m, sw, gargs, _Spy(opt, m, grads), share_periods=share, **kw)
    torch.cuda.synchronize()
    out = grads, float(last), float(total)
    with torch.no_grad():
        for k, v in m.state_dict().items():
            v.copy_(saved[k])
    return out


def _oracle_epoch(w, nd, first, last):
    """fp64 gradients, last loss and total of run.py's epoch over windows [first, last) (before the optimizer step)"""
    from oracle import loop_oracle as LO
    feats, targ = LO.windows(nd.double(), w.T, w.O)
    ref = build_oracle(w, torch.float64)
    total, loss = 0.0, None
    for x, y in list(zip(feats, targ))[first:last]:
        o, _ = ref(x, *w.graph_args())
        loss = torch.mean((o - y) ** 2)
        loss.backward()
        total += float(loss.detach())
    grads = {k: p.grad for k, p in ref.named_parameters() if p.grad is not None and not is_dead(w.model, k)}
    return grads, float(loss.detach()), total, copy.deepcopy(ref.state_dict())


def _att(k):
    return k.endswith("_attention")


def _close(ga, gb, tol, att_tol, model):
    for k, g in gb.items():
        if is_dead(model, k):
            continue
        e = relerr(ga[k], g)
        assert e <= (att_tol if _att(k) else tol), (k, e)


# (model, H, precision, N, T, O, cell path) -- every cell path at T = 1 over the steps
_PATHS = [("TemporalGCN", 32, "fp32", 30, 6, 3, "fp32"),
          ("TemporalGCN", 64, "tf32x3", 30, 6, 3, "fused tf32x3"),
          ("RegionalTemporalGCN", 128, "tf32x3", 30, 6, 3, "fused tf32x3"),
          ("RegionalTemporalGCN", 256, "tf32x3", 30, 6, 3, "unfused tf32x3"),
          ("TemporalGCN", 64, "bf16", 150, 12, 12, "fused bf16"),
          ("RegionalTemporalGCN", 128, "bf16", 60, 12, 6, "bf16 GEMM")]


def _case(model, H, prec, N, T, O, n_windows, seed=11, **kw):
    w = W.tiny_workload(model, N=N, T=T, H=H, O=O, R=3 if model == "RegionalTemporalGCN" else 0, B=1, seed=seed, **kw)
    nd = _series(w.N, 8, T + O + n_windows - 1, 5)
    return w, nd


@pytest.mark.parametrize("case", _PATHS, ids=[p[-1].replace(" ", "_") + f"_{p[0][:8]}_H{p[1]}" for p in _PATHS])
def test_epoch_parity_every_cell_path(case):
    from regt_b200.loop import SlidingWindows
    model, H, prec, N, T, O, _ = case
    n = 12 if prec != "bf16" else 9
    w, nd = _case(model, H, prec, N, T, O, n, k_intra=5 if prec == "bf16" else 3)
    g_ref, last_ref, total_ref, state = _oracle_epoch(w, nd, 0, n)
    m = build_cuda(w, state, "cuda", precision=prec)
    gargs = to_dev(w.graph_args(), "cuda")
    sw = SlidingWindows(nd.cuda(), T, O)
    g_win, last_win, total_win = _epoch(m, sw, gargs, False, batch=5)
    g_sh, last_sh, total_sh = _epoch(m, sw, gargs, True, batch=5)
    if prec == "bf16":   # the stated bf16 bounds: loss 2e-2, gradients 5e-2, attention 0.15
        assert abs(last_sh - last_ref) <= 2e-2 * abs(last_ref) and abs(total_sh - total_ref) <= 2e-2 * abs(total_ref)
        _close(g_sh, g_ref, 5e-2, 0.15, w.model)
        return
    for lw, tw in ((last_win, total_win), (last_ref, total_ref)):
        assert abs(last_sh - lw) <= 1e-5 * abs(lw) and abs(total_sh - tw) <= 1e-5 * abs(tw)
    _close(g_sh, g_win, 1e-5, 1e-4, w.model)
    _close(g_sh, g_ref, 1e-5, 1e-4, w.model)


@pytest.mark.parametrize("case", _PATHS[:4], ids=[p[-1].replace(" ", "_") + f"_H{p[1]}" for p in _PATHS[:4]])
def test_forward_matches_the_windowed_model(case):
    """out and out_hidden of the shared forward against model(x_windows).  On the fp32 path out_hidden is bitwise equal: the
    FFMA cell computes each period's H' with the same arithmetic at T = 1, and k_comb_fwd sums probs[t] H'_t with the same
    fmaf chain as k_attn_accum.  The fused tf32x3 cell folds the attention into its gate epilogue, so it agrees to rounding."""
    from regt_b200.loop import SlidingWindows, _SharedPlan
    model, H, prec, N, T, O, _ = case
    w, nd = _case(model, H, prec, N, T, O, 10)
    m = build_cuda(w, build_oracle(w).state_dict(), "cuda", precision=prec)
    gargs = to_dev(w.graph_args(), "cuda")
    sw = SlidingWindows(nd.cuda(), T, O)
    with torch.no_grad():
        sp = _SharedPlan(m, sw, gargs, 10, 10)
        out, _, _, _ = sp.run_pass(0, 10, False)
        hid = sp.bufs["hid"][:10]
        x, _ = sw.gather(torch.arange(10, device="cuda"))
        out_w, hid_w = m(x, *gargs)
    assert relerr(hid, hid_w) <= 1e-6 and relerr(out, out_w) <= 1e-6
    if prec == "fp32":
        assert torch.equal(hid, hid_w)


@pytest.mark.parametrize("case", [_PATHS[0], _PATHS[2]], ids=["fp32", "fused_tf32x3"])
def test_pass_size_invariance(case, monkeypatch):
    from regt_b200 import loop
    from regt_b200.loop import SlidingWindows, _SharedPlan
    model, H, prec, N, T, O, _ = case
    n = 12
    w, nd = _case(model, H, prec, N, T, O, n)
    m = build_cuda(w, build_oracle(w).state_dict(), "cuda", precision=prec)
    gargs = to_dev(w.graph_args(), "cuda")
    sw = SlidingWindows(nd.cuda(), T, O)
    g_all, l_all, t_all = _epoch(m, sw, gargs, True, batch=n)
    runs = [_epoch(m, sw, gargs, True, batch=b) for b in (1, T - 1, T)]
    need3 = _SharedPlan(m, sw, gargs, 3, n)._bytes(3)
    m._shared_bufs = None
    monkeypatch.setattr(loop, "_shared_budget", lambda have=0: need3)   # a pass of n windows does not fit: it shrinks to 3
    runs.append(_epoch(m, sw, gargs, True, batch=n))
    assert m._shared_bufs["C"] == 3
    # losses to 1e-6.  Gradients to the bound the step holds for regrouped micro-batches (1e-5, 1e-4 for the attention):
    # each pass's cell backward sums its S * N rows in its own split-K partition, so the pass size regroups the fp32 sums
    # of the weight gradients (up to 2.1e-6 measured at these shapes)
    for g, lst, tot in runs:
        assert abs(lst - l_all) <= 1e-6 * abs(l_all) and abs(tot - t_all) <= 1e-6 * abs(t_all)
        _close(g, g_all, 1e-5, 1e-4, w.model)


@pytest.mark.parametrize("N,O", [(30, 3), (207, 24)])
def test_every_head_route_of_a_pass(N, O):
    """tf32x3 at hidden 64: the head-only calls of a pass route differently -- the training head (the tf32x3 head from 128
    rows and up to 16 outputs, else the fused FFMA head), the final window alone and evaluation (the row head where the
    tf32x3 head does not apply) -- and the one cached head workspace holds every one: passes of 1 and 5 windows, evaluate"""
    from regt_b200.loop import SlidingWindows, evaluate
    w, nd = _case("TemporalGCN", 64, "tf32x3", N, 6, O, 7)
    m = build_cuda(w, build_oracle(w).state_dict(), "cuda", precision="tf32x3")
    gargs = to_dev(w.graph_args(), "cuda")
    sw = SlidingWindows(nd.cuda(), 6, O)
    for b in (1, 5):
        m._shared_bufs = None
        g_win, l_win, t_win = _epoch(m, sw, gargs, False, batch=b)
        g_sh, l_sh, t_sh = _epoch(m, sw, gargs, True, batch=b)
        assert abs(l_sh - l_win) <= 1e-5 * abs(l_win) and abs(t_sh - t_win) <= 1e-5 * abs(t_win)
        _close(g_sh, g_win, 1e-5, 1e-4, w.model)
    for b in (1, 5):
        m._shared_bufs = None                      # evaluate first: its own (inference-sized) buffers
        a = evaluate(m, sw, gargs, batch=b)
        c = evaluate(m, sw, gargs, batch=b, share_periods=True)
        for u, v in zip(a, c):
            assert abs(u - v) <= 1e-6 * abs(u), (a, c)
    _epoch(m, sw, gargs, True, batch=5)            # training after an evaluation re-sizes the cached buffers
    assert m._shared_bufs["train"]


@pytest.mark.parametrize("edge", ["one_window", "t_in_1", "t_in_64_fused_tf32x3", "inner_range", "two_features",
                                  "t_in_257_fp32"])
def test_edges(edge):
    from models import TemporalGCN
    from regt_b200.loop import SlidingWindows
    model, H, prec, N, T, O, n, first, last, F = "TemporalGCN", 32, "fp32", 30, 6, 3, 12, 0, None, 8
    if edge == "one_window":
        n = 1
    elif edge == "t_in_1":
        T = 1
    elif edge == "t_in_64_fused_tf32x3":
        H, prec, T, n = 64, "tf32x3", 64, 5
    elif edge == "inner_range":
        first, last = 2, 9
    elif edge == "t_in_257_fp32":                  # beyond the combine kernels' 256 periods: the windowed epoch runs
        T, n = 257, 2
    w, nd = _case(model, H, prec, N, T, O, n)
    state = build_oracle(w).state_dict()
    if edge == "two_features":
        F = 2
        nd = nd[:, :2].contiguous()
        torch.manual_seed(3)
        m = TemporalGCN(2, T, O, hidden=H, precision=prec).cuda()
    else:
        m = build_cuda(w, state, "cuda", precision=prec)
    gargs = to_dev(w.graph_args(), "cuda")
    sw = SlidingWindows(nd.cuda(), T, O)
    kw = dict(batch=5, first=first, last=last)
    g_win, l_win, t_win = _epoch(m, sw, gargs, False, **kw)
    g_sh, l_sh, t_sh = _epoch(m, sw, gargs, True, **kw)
    assert abs(l_sh - l_win) <= 1e-5 * abs(l_win) and abs(t_sh - t_win) <= 1e-5 * abs(t_win)
    _close(g_sh, g_win, 1e-5, 1e-4, w.model)
    assert F == sw.F
    if edge == "t_in_257_fp32":
        assert l_sh == l_win and t_sh == t_win and all(torch.equal(g_sh[k], g_win[k]) for k in g_win)


def _masked_series(nd, T, O, n, kind):
    nd = nd.clone()
    g = torch.Generator().manual_seed(9)
    if kind == "zeros":
        hit = torch.rand(nd.shape[0], nd.shape[2], generator=g) < 0.2
        nd[:, -1][hit] = 0.0
        nd[:, -1, 3 + T:3 + T + O] = 0.0          # window 3: every target missing
    elif kind == "nan":                            # NaN only where no window of the epoch reads an input
        tail = nd[:, -1, n + T - 1:]
        tail[torch.rand(tail.shape, generator=g) < 0.5] = float("nan")
    return nd


@pytest.mark.parametrize("loss,null", [("mae", None), ("mse", "zeros"), ("mae", "zeros"), ("mse", "nan")])
def test_losses(loss, null):
    from regt_b200.loop import SlidingWindows
    model, H, prec, N, T, O, _ = _PATHS[1]
    n = 12
    w, nd = _case(model, H, prec, N, T, O, n)
    nd = _masked_series(nd, T, O, n, null)
    m = build_cuda(w, build_oracle(w).state_dict(), "cuda", precision=prec)
    gargs = to_dev(w.graph_args(), "cuda")
    sw = SlidingWindows(nd.cuda(), T, O)
    nv = None if null is None else (0.0 if null == "zeros" else float("nan"))
    kw = dict(batch=5, loss=loss, null_value=nv)
    g_win, l_win, t_win = _epoch(m, sw, gargs, False, **kw)
    g_sh, l_sh, t_sh = _epoch(m, sw, gargs, True, **kw)
    assert abs(l_sh - l_win) <= 1e-5 * abs(l_win) and abs(t_sh - t_win) <= 1e-5 * abs(t_win)
    _close(g_sh, g_win, 1e-5, 1e-4, w.model)
    if null == "zeros":   # the all-missing window adds no loss and no gradient
        g1, l1, t1 = _epoch(m, sw, gargs, True, batch=5, first=3, last=4, loss=loss, null_value=0.0)
        assert l1 == 0.0 and t1 == 0.0 and all(float(g.abs().max()) == 0.0 for g in g1.values())


@pytest.mark.parametrize("null", [None, 0.0])
def test_evaluate_matches_windowed(null):
    from regt_b200.loop import SlidingWindows, evaluate
    model, H, prec, N, T, O, _ = _PATHS[2]
    w, nd = _case(model, H, prec, N, T, O, 14)
    if null is not None:
        nd = _masked_series(nd, T, O, 14, "zeros")
    m = build_cuda(w, build_oracle(w).state_dict(), "cuda", precision=prec)
    gargs = to_dev(w.graph_args(), "cuda")
    sw = SlidingWindows(nd.cuda(), T, O)
    a = evaluate(m, sw, gargs, 1, 14, batch=4, null_value=null)
    b = evaluate(m, sw, gargs, 1, 14, batch=4, null_value=null, share_periods=True)
    for u, v in zip(a, b):
        assert abs(u - v) <= 1e-6 * abs(u), (a, b)


def test_sharing_really_happens(monkeypatch):
    """per pass: one launch of the cell forward and backward, over the C + T - 1 steps of the pass at one period each (the
    regt_args the cell entry points receive), and one of each combine kernel"""
    from regt_b200 import _lib
    from regt_b200.loop import SlidingWindows
    model, H, prec, N, T, O, _ = _PATHS[1]
    n = 12
    w, nd = _case(model, H, prec, N, T, O, n)
    m = build_cuda(w, build_oracle(w).state_dict(), "cuda", precision=prec)
    gargs = to_dev(w.graph_args(), "cuda")
    sw = SlidingWindows(nd.cuda(), T, O)
    lib = _lib.load()
    _epoch(m, sw, gargs, True, batch=5)            # warm
    calls = []

    def recorded(name):
        fn = getattr(lib, name)

        def call(a):
            calls.append((name, a._obj.B, a._obj.T))
            return fn(a)
        return call

    for name in ("regt_cell_forward", "regt_cell_backward"):
        monkeypatch.setattr(lib, name, recorded(name))
    torch.cuda.synchronize()
    lib.regt_profile(1, torch.cuda.current_stream().cuda_stream)
    try:
        _epoch(m, sw, gargs, True, batch=5)
        torch.cuda.synchronize()
        names = [nm for nm, _ in _lib.profile_read()]
    finally:
        lib.regt_profile(0, None)
    passes = [5, 5, 2]                             # 12 windows, 5 per pass
    for k in ("k_cell_fwd_f", "k_cell_bwd_f", "k_comb_fwd", "k_comb_bwd", "k_comb_attn"):
        assert names.count(k) == len(passes), (k, names.count(k))
    want = [(f, c + T - 1, 1) for c in passes for f in ("regt_cell_forward", "regt_cell_backward")]
    assert calls == want, calls                    # no cell call covers T periods


def test_determinism_and_poisoned_cache():
    from regt_b200.loop import SlidingWindows
    model, H, prec, N, T, O, _ = _PATHS[2]
    w, nd = _case(model, H, prec, N, T, O, 12)
    m = build_cuda(w, build_oracle(w).state_dict(), "cuda", precision=prec)
    gargs = to_dev(w.graph_args(), "cuda")
    sw = SlidingWindows(nd.cuda(), T, O)
    runs = [_epoch(m, sw, gargs, True, batch=5) for _ in range(2)]
    for k, t in m._shared_bufs.items():             # every cached buffer but the constant zero attention of the steps
        if isinstance(t, torch.Tensor) and k != "att0":
            t.fill_(255) if t.dtype == torch.uint8 else t.fill_(float("nan"))
    runs.append(_epoch(m, sw, gargs, True, batch=5))
    g0, l0, t0 = runs[0]
    for g, lst, tot in runs[1:]:
        assert lst == l0 and tot == t0
        assert all(torch.equal(g[k], g0[k]) for k in g0)


def test_refusals():
    from models.utils import TGCN
    from regt_b200 import shard as S
    from regt_b200.loop import FlatRMSprop, SlidingWindows, train_epoch
    w, nd = _case("RegionalTemporalGCN", 64, "fp32", 30, 6, 3, 8)
    sw = SlidingWindows(nd.cuda(), 6, 3)
    gargs = to_dev(w.graph_args(), "cuda")
    t = TGCN(8, 32).cuda()
    with pytest.raises(TypeError, match="share_periods"):
        train_epoch(t, sw, gargs, FlatRMSprop(list(t.parameters())), share_periods=True)
    m = build_cuda(w, build_oracle(w).state_dict(), "cuda", precision="fp32")
    sm = S.RegionShardedModel(m, w.edge_index.cuda(), [e.cuda() for e in w.reg_edge_index],
                              [a.cuda() for a in w.reg_edge_attr], 0, 2)
    with pytest.raises(TypeError, match="share_periods"):
        train_epoch(sm, sw, gargs, FlatRMSprop(list(m.parameters())), share_periods=True)
    w65, nd65 = _case("TemporalGCN", 64, "tf32x3", 30, 65, 1, 2)
    m65 = build_cuda(w65, build_oracle(w65).state_dict(), "cuda", precision="tf32x3")
    sw65 = SlidingWindows(nd65.cuda(), 65, 1)
    g65 = to_dev(w65.graph_args(), "cuda")
    for share in (False, True):                    # the same refusal as the windowed step
        with pytest.raises(RuntimeError, match=r"precision tf32x3 supports up to 64 periods \(got 65\)"):
            train_epoch(m65, sw65, g65, FlatRMSprop(list(m65.parameters())), share_periods=share)


def test_run_py_share_periods_one_epoch(tmp_path, monkeypatch):
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("regt_run", os.path.join(root, "run.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    monkeypatch.chdir(tmp_path)
    rc = mod.main("--num_timesteps_in 6 --num_timesteps_out 1 --tr 0.5 --tf occrate --dataloading_type 2 --epochs 1 "
                  "--decomp_type regional --model RegionalTemporalGCN --synthetic_steps 30 --bs 8 --share_periods".split())
    assert rc == 0
    ck = tmp_path / "pretrained" / "occrate" / "RegionalTemporalGCN" / "model_in6_out1_epoch0.pt"
    state = torch.load(ck, map_location="cpu")
    assert all(torch.isfinite(v).all() for v in state.values())
