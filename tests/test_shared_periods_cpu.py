"""CPU tests of the period-sharing epoch (share_periods): the combine entry points and the head-only mode of regt_args are
declared, exported and checked on the host without a GPU; the flags parse."""
import ctypes as C
import importlib.util
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _lib():
    from regt_b200 import _lib
    return _lib, _lib.load()


def test_combine_entry_points_declared_and_exported():
    _l, lib = _lib()
    src = open(os.path.join(ROOT, "include", "regt_b200.h")).read()
    for n in ("regt_combine_scratch_bytes", "regt_combine_forward", "regt_combine_backward"):
        assert n + "(" in src and n in _l.EXPORTS and hasattr(lib, n)
    assert lib.regt_combine_scratch_bytes(12) >= 12 * 8 and lib.regt_combine_scratch_bytes(0) == 0


@pytest.mark.parametrize("S,C,T,width,msg", [(10, 4, 6, 64, b"C + T - 1"), (9, 5, 6, 64, b"C + T - 1"), (4, 4, 0, 64, b"T=0"),
                                             (8, 0, 6, 64, b"C=0"), (9, 4, 6, 62, b"multiple of 4")])
def test_combine_rejects_inconsistent_sizes(S, C, T, width, msg):
    _l, lib = _lib()
    fake = 0x10000                                        # never dereferenced: the checks run before any CUDA call
    assert lib.regt_combine_forward(fake, fake, S, C, T, width, fake, None) != 0
    assert msg in lib.regt_last_error()
    assert lib.regt_combine_backward(fake, fake, fake, S, C, T, width, fake, fake, fake, 1 << 20, None) != 0
    assert msg in lib.regt_last_error()


def test_combine_rejects_null_and_small_scratch():
    _l, lib = _lib()
    fake = 0x10000
    assert lib.regt_combine_forward(None, fake, 9, 4, 6, 64, fake, None) != 0 and b"NULL" in lib.regt_last_error()
    assert lib.regt_combine_forward(fake, fake, 9, 4, 6, 64, None, None) != 0 and b"NULL" in lib.regt_last_error()
    assert lib.regt_combine_backward(fake, fake, None, 9, 4, 6, 64, fake, fake, fake, 1 << 20, None) != 0
    assert b"NULL" in lib.regt_last_error()
    small = lib.regt_combine_scratch_bytes(6) - 8
    assert lib.regt_combine_backward(fake, fake, fake, 9, 4, 6, 64, fake, fake, fake, small, None) != 0
    assert b"scratch" in lib.regt_last_error()


def _args(head_only, B=64, N=207, T=12, H=64, O=12, prec=1, mode=1, nseg=600):
    _l, lib = _lib()
    a = _l.Args()
    a.B, a.N, a.T, a.H, a.O, a.mode, a.precision, a.fuse_head = B, N, T, H, O, mode, prec, 1
    a.plan.N, a.plan.R, a.plan.nseg = N, 3, nseg
    a.y, a.loss, a.d_out, a.out = 0x1000, 0x2000, 0x3000, 0x4000   # never dereferenced
    a.head_only = head_only
    return a


def test_args_field_appended_and_zero_by_default():
    _l, _ = _lib()
    a = _l.Args()
    assert a.head_only == 0
    names = [f[0] for f in _l.Args._fields_]
    assert names[-1] == "head_only" and names[-2] == "loss_count"
    assert _l.Args.head_only.offset >= _l.Args.loss_count.offset + C.sizeof(C.c_void_p)
    src = open(os.path.join(ROOT, "include", "regt_b200.h")).read()
    assert src.index("const float* loss_count;") < src.index("int32_t head_only;") < src.index("} regt_args;")


@pytest.mark.parametrize("prec,H", [(0, 32), (1, 64), (1, 128), (1, 256), (2, 64), (2, 128)])
def test_head_only_workspace_holds_no_cell_planes(prec, H):
    _l, lib = _lib()
    sizes = [lib.regt_workspace_bytes(C.byref(_args(1, T=T, H=H, prec=prec))) for T in (1, 12, 64)]
    assert sizes[0] > 0 and sizes[0] == sizes[1] == sizes[2]            # nothing scales with the periods
    full = lib.regt_workspace_bytes(C.byref(_args(0, T=12, H=H, prec=prec)))
    assert sizes[1] * 4 < full


@pytest.mark.parametrize("prec,H,O,BN,step", [(2, 64, 16, 256, True), (2, 64, 12, 100, True), (2, 128, 12, 256, True),
                                              (1, 64, 16, 256, True), (1, 128, 16, 100, True), (1, 128, 17, 256, True),
                                              (0, 32, 12, 256, True), (0, 64, 12, 256, False), (0, 128, 12, 256, True)])
def test_head_only_route(prec, H, O, BN, step):
    """head_only: no cell (5), never k_head_tc (3), row-major G, no out_hidden partials; the head choice otherwise follows the
    same rules (tf32x3 head from 128 rows and at most 16 outputs, the fused FFMA head in a training step at hidden 32 / 64)"""
    _l, lib = _lib()
    a = _args(1, B=1, N=BN, H=H, O=O, prec=prec)
    a.fuse_head = int(step)
    o = (C.c_int32 * 4)()
    _l.check(lib.regt_debug_route(C.byref(a), o), "regt_debug_route")
    cell, head, g_tiled, partials = list(o)
    assert cell == 5 and head != 3 and g_tiled == 0 and partials == 0
    if prec == 1 and H % 32 == 0 and O <= 16 and BN >= 128:
        assert head == 2
    elif step and H in (32, 64) and O <= 44:
        assert head == 1
    else:
        assert head == 0


def test_cell_entry_points_refuse_head_only():
    _l, lib = _lib()
    a = _args(1, B=2, N=16, H=64, prec=0, nseg=0)
    a.workspace, a.workspace_bytes = 0x100000, lib.regt_workspace_bytes(C.byref(a))
    a.x, a.out_hidden = 0x5000, 0x6000
    for fn in (lib.regt_cell_forward, lib.regt_cell_backward):
        assert fn(C.byref(a)) != 0
        assert b"head_only" in lib.regt_last_error()


def _mod(name):
    spec = importlib.util.spec_from_file_location(f"regt_{name}", os.path.join(ROOT, f"{name}.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.parametrize("script", ["run", "predict"])
def test_share_periods_flag(script):
    p = _mod(script).build_parser()
    assert p.parse_args([]).share_periods is False
    assert p.parse_args(["--share_periods"]).share_periods is True


@pytest.mark.parametrize("prec,H,N,O,windows", [(1, 64, 207, 24, 64), (1, 64, 30, 3, 1), (1, 64, 30, 3, 5), (1, 32, 100, 12, 2),
                                          (1, 128, 207, 12, 64), (0, 64, 30, 3, 1), (2, 64, 207, 12, 64)])
def test_head_only_workspace_holds_every_head_call_of_a_pass(prec, H, N, O, windows):
    """a pass sizes one head-only workspace for its training call over C windows; the evaluation call over C windows and the
    final window's own call (B = 1, targets, no fused head) route to other heads and must fit it too"""
    _l, lib = _lib()

    def need(B, train, y):
        a = _args(1, B=B, N=N, H=H, O=O, prec=prec)
        a.fuse_head = int(train)
        if not y:
            a.y, a.loss, a.d_out = 0, 0, 0
        return lib.regt_workspace_bytes(C.byref(a))
    sized = need(windows, True, True)
    assert need(windows, False, False) <= sized and need(1, False, True) <= sized

