"""precision bf16 at every hidden width divisible by 32, decided on the host without a GPU: which cell and head kernels
regt_debug_route picks (the fused H = 64 cell of cell_tc.cu where it is built for the shape, the GEMM-by-GEMM cell of
cell_g.cu on the single-pass bf16 GEMMs everywhere else), the refusal of other widths before any launch, and the test
hooks of the bf16 GEMMs."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "regt_b200.h")

_BF16 = 2
_A3TGCN, _REGIONAL, _TGCN = 0, 1, 2
_CELL = {"bf16": 3, "bf16_gemm": 4}
_HEAD = {"rows": 0, "fused_ffma": 1, "tf32x3": 2, "bf16": 3}
# (H, O, mode, fused training step, REGT_UNFUSED) -> (cell, head, G tiled, out_hidden partials)
_ROUTES = [
    ((32, 12, _REGIONAL, True, None), ("bf16_gemm", "fused_ffma", 0, 0)),
    ((32, 12, _REGIONAL, False, None), ("bf16_gemm", "rows", 0, 0)),
    ((96, 12, _REGIONAL, True, None), ("bf16_gemm", "rows", 0, 0)),
    ((128, 16, _REGIONAL, True, None), ("bf16_gemm", "rows", 0, 0)),
    ((128, 16, _REGIONAL, False, None), ("bf16_gemm", "rows", 0, 0)),
    ((256, 1, _REGIONAL, True, None), ("bf16_gemm", "rows", 0, 0)),
    ((256, 4, _A3TGCN, True, None), ("bf16_gemm", "rows", 0, 0)),
    ((128, 4, _A3TGCN, False, None), ("bf16_gemm", "rows", 0, 0)),
    ((32, 1, _TGCN, False, None), ("bf16_gemm", "rows", 0, 0)),
    ((64, 1, _TGCN, False, None), ("bf16_gemm", "rows", 0, 0)),
    ((64, 16, _TGCN, True, None), ("bf16_gemm", "fused_ffma", 0, 0)),   # k_head_tc's partials need the fused cell backward
    ((256, 1, _TGCN, False, None), ("bf16_gemm", "rows", 0, 0)),
    # the fused H = 64 cell keeps its shapes ...
    ((64, 16, _REGIONAL, True, None), ("bf16", "bf16", 1, 1)),
    ((64, 16, _A3TGCN, True, None), ("bf16", "bf16", 1, 1)),
    ((64, 12, _REGIONAL, False, None), ("bf16", "rows", 1, 0)),
    # ... and REGT_UNFUSED (a switch of the tf32x3 cells) changes no bf16 route
    ((64, 16, _REGIONAL, True, "1"), ("bf16", "bf16", 1, 1)),
    ((128, 16, _REGIONAL, True, "1"), ("bf16_gemm", "rows", 0, 0)),
    ((32, 12, _TGCN, True, "1"), ("bf16_gemm", "fused_ffma", 0, 0)),
]


def _args(H, O, mode, step, BN=256, T=12):
    from regt_b200 import _lib
    a = _lib.Args()
    a.B, a.N, a.T, a.H, a.O, a.mode, a.precision, a.fuse_head = 1, BN, T, H, O, mode, _BF16, int(step)
    a.plan.N = BN
    a.y, a.loss, a.d_out, a.out = 0x1000, 0x2000, 0x3000, 0x4000   # never dereferenced
    return a


@pytest.mark.parametrize("case,want", _ROUTES)
def test_bf16_route(case, want, monkeypatch):
    from regt_b200 import _lib
    lib = _lib.load()
    H, O, mode, step, unfused = case
    if unfused is None:
        monkeypatch.delenv("REGT_UNFUSED", raising=False)
    else:
        monkeypatch.setenv("REGT_UNFUSED", unfused)
    o = (C.c_int32 * 4)()
    _lib.check(lib.regt_debug_route(C.byref(_args(H, O, mode, step)), o), "regt_debug_route")
    cell, head, g_tiled, partials = want
    assert list(o) == [_CELL[cell], _HEAD[head], g_tiled, partials]


@pytest.mark.parametrize("H", [48, 40, 72])
@pytest.mark.parametrize("entry", ["regt_cell_forward", "regt_cell_backward"])
def test_width_not_divisible_by_32_is_refused_on_the_host(H, entry):
    """the argument check runs before any launch: no device, and the workspace pointer is never dereferenced."""
    from regt_b200 import _lib
    lib = _lib.load()
    a = _args(H, 4, _REGIONAL, False)
    a.x, a.out_hidden = 0x5000, 0x6000
    a.workspace, a.workspace_bytes = 0x7000, lib.regt_workspace_bytes(C.byref(a))
    assert a.workspace_bytes > 0
    assert getattr(lib, entry)(C.byref(a)) != 0
    msg = lib.regt_last_error().decode()
    assert "bf16" in msg and "hidden % 32" in msg and f"got {H}" in msg, msg


def test_bf16_workspace_holds_the_gemm_cell_planes():
    """the GEMM-by-GEMM bf16 cell takes the row-major planes of make_layout: its workspace grows with H like the
    tf32x3 one, and the bf16 image of the weights is smaller than the tf32 hi | lo pair."""
    from regt_b200 import _lib
    lib = _lib.load()
    sizes = {}
    for prec in (_lib.PREC_TF32X3, _BF16):
        a = _args(256, 4, _TGCN, False)
        a.precision = prec
        sizes[prec] = lib.regt_workspace_bytes(C.byref(a))
    assert 0 < sizes[_BF16] <= sizes[_lib.PREC_TF32X3]
    a = _args(128, 4, _REGIONAL, False)
    small = lib.regt_workspace_bytes(C.byref(a))
    a = _args(256, 4, _REGIONAL, False)
    assert lib.regt_workspace_bytes(C.byref(a)) > small


def test_bf16_gemm_hooks_are_exported_and_declared():
    from regt_b200 import _lib
    lib = _lib.load()
    src = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    hooks = src[src.index("regt_debug_gemm_nt_tma"):]
    for name in ("regt_debug_gemm_nt_bf16", "regt_debug_gemm_tn_bf16"):
        assert hasattr(lib, name), name
        assert re.search(r"\bint %s\s*\(" % name, hooks), f"{name} is not declared among the test hooks"
        tf32 = getattr(lib, name.replace("bf16", "tma"))
        assert getattr(lib, name).argtypes == tf32.argtypes
