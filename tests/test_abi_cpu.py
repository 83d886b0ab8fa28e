"""CPU tests of the drop-in boundary: the C-ABI library loads without a GPU and exports every symbol
that include/regt_b200.h declares (no compute calls), the ctypes structs mirror the header, the host-side
argument checks fail loudly, and the product package never imports the oracle."""
import ctypes as C
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "regt_b200.h")


def _declared_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(regt_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from regt_b200 import _lib
    lib = _lib.load()                      # builds with nvcc if missing; dlopen needs no GPU
    names = _declared_functions()
    assert len(names) >= 16
    for n in names:
        assert hasattr(lib, n), f"{n} is declared in include/regt_b200.h but not exported"
    assert set(_lib.EXPORTS) <= set(names)
    assert lib.regt_version() == 100
    assert lib.regt_last_error() is not None


def test_library_exports_nothing_undeclared():
    """every regt_* symbol the shared library exports is declared in the header (product entry points or the TEST HOOKS
    section): no hidden entry points."""
    import subprocess
    from regt_b200 import _lib
    _lib.load()
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.lib_path()], capture_output=True, text=True, check=True).stdout
    exported = {ln.split()[-1] for ln in out.splitlines() if ln.split() and ln.split()[-1].startswith("regt_") and " T " in ln}
    undeclared = sorted(exported - set(_declared_functions()))
    assert not undeclared, f"exported but not declared in include/regt_b200.h: {undeclared}"


def test_tc_split_hook():
    """regt_debug_tc_split (the work split of the bf16 kernels) is consistent in itself and, with 148 SMs (a B200, or
    the count assumed without a device), gives the splits tests/test_gpu_bf16_edges.py is built around."""
    from regt_b200 import _lib
    lib = _lib.load()

    def split(B, N, T):
        o = (C.c_int32 * 7)()
        _lib.check(lib.regt_debug_tc_split(B, N, T, o), "regt_debug_tc_split")
        return list(o)

    shapes = {(64, 207, 12): [104, 3, 4, 416], (3, 207, 12): [5, 1, 12, 60], (64, 592, 12): [296, 12, 1, 296],
              (32, 592, 12): [148, 12, 1, 148], (16, 592, 12): [74, 6, 2, 148], (8, 592, 12): [37, 3, 4, 148]}
    slots = split(64, 592, 12)[4]
    for (B, N, T), want in shapes.items():
        nqt, tp, ntc, items, fwd, bwd, head = split(B, N, T)
        assert nqt == -(-B * N // 128) and T % tp == 0 and ntc == T // tp and items == nqt * ntc
        assert fwd == min(slots, items) and bwd == min(fwd, 160) and head == min(148, nqt)
        if slots == 148:
            assert [nqt, tp, ntc, items] == want, (B, N, T)
    with pytest.raises(RuntimeError, match="must be positive"):
        _lib.check(lib.regt_debug_tc_split(0, 207, 12, (C.c_int32 * 7)()), "regt_debug_tc_split")


_FP32, _TF32X3, _BF16 = 0, 1, 2
_REGIONAL, _TGCN = 1, 2
_CELL = {"fp32": 0, "unfused": 1, "fused": 2, "bf16": 3}
_HEAD = {"rows": 0, "fused_ffma": 1, "tf32x3": 2, "bf16": 3}
# (precision, H, O, B*N, T, mode, fused training step, REGT_UNFUSED) -> (cell, head, G tiled, out_hidden partials)
_ROUTES = [
    ((_BF16, 64, 16, 256, 12, _REGIONAL, True, None), ("bf16", "bf16", 1, 1)),
    ((_BF16, 64, 17, 256, 12, _REGIONAL, True, None), ("bf16", "fused_ffma", 1, 1)),
    ((_BF16, 64, 44, 256, 12, _REGIONAL, True, None), ("bf16", "fused_ffma", 1, 1)),
    ((_BF16, 64, 45, 256, 12, _REGIONAL, True, None), ("bf16", "rows", 1, 0)),     # k_head_fused needs 229 KB of shared memory
    ((_BF16, 64, 65, 256, 12, _REGIONAL, True, None), ("bf16", "rows", 1, 0)),
    ((_BF16, 64, 16, 256, 12, _REGIONAL, False, None), ("bf16", "rows", 1, 0)),
    ((_BF16, 64, 17, 256, 12, _REGIONAL, False, None), ("bf16", "rows", 1, 0)),
    ((_BF16, 64, 44, 256, 12, _REGIONAL, False, None), ("bf16", "rows", 1, 0)),
    ((_BF16, 64, 45, 256, 12, _REGIONAL, False, None), ("bf16", "rows", 1, 0)),
    ((_BF16, 64, 65, 256, 12, _REGIONAL, False, None), ("bf16", "rows", 1, 0)),
    ((_BF16, 64, 16, 256, 12, _REGIONAL, True, "1"), ("bf16", "bf16", 1, 1)),
    ((_TF32X3, 128, 16, 256, 12, _REGIONAL, True, None), ("fused", "tf32x3", 1, 0)),
    ((_TF32X3, 128, 17, 256, 12, _REGIONAL, True, None), ("fused", "rows", 1, 0)),
    ((_TF32X3, 128, 16, 127, 12, _REGIONAL, True, None), ("fused", "rows", 1, 0)),
    ((_TF32X3, 128, 16, 128, 12, _REGIONAL, True, None), ("fused", "tf32x3", 1, 0)),
    ((_TF32X3, 64, 16, 127, 12, _REGIONAL, True, None), ("fused", "fused_ffma", 1, 0)),
    ((_TF32X3, 256, 16, 256, 12, _REGIONAL, True, None), ("unfused", "tf32x3", 0, 0)),
    ((_TF32X3, 128, 16, 256, 65, _REGIONAL, True, None), ("unfused", "tf32x3", 0, 0)),
    ((_TF32X3, 128, 16, 256, 12, _TGCN, True, None), ("unfused", "tf32x3", 0, 0)),
    ((_TF32X3, 128, 16, 256, 12, _REGIONAL, True, "1"), ("unfused", "tf32x3", 0, 0)),
    ((_TF32X3, 64, 17, 256, 12, _REGIONAL, True, "1"), ("unfused", "fused_ffma", 0, 0)),
    ((_FP32, 32, 12, 256, 12, _REGIONAL, True, None), ("fp32", "fused_ffma", 0, 0)),
    ((_FP32, 64, 12, 256, 12, _REGIONAL, True, None), ("fp32", "fused_ffma", 0, 0)),
    ((_FP32, 128, 12, 256, 12, _REGIONAL, True, None), ("fp32", "rows", 0, 0)),
    ((_FP32, 64, 12, 256, 12, _REGIONAL, False, None), ("fp32", "rows", 0, 0)),
]


@pytest.mark.parametrize("case,want", _ROUTES)
def test_route_table(case, want, monkeypatch):
    """regt_debug_route: which cell and head kernels the entry points run, decided on the host without a GPU.  A fused
    training step passes fuse_head with y, d_out and loss; outside one fuse_head is 0."""
    from regt_b200 import _lib
    lib = _lib.load()
    prec, H, O, BN, T, mode, step, unfused = case
    if unfused is None:
        monkeypatch.delenv("REGT_UNFUSED", raising=False)
    else:
        monkeypatch.setenv("REGT_UNFUSED", unfused)
    a = _lib.Args()
    a.B, a.N, a.T, a.H, a.O, a.mode, a.precision, a.fuse_head = 1, BN, T, H, O, mode, prec, int(step)
    a.plan.N = BN
    a.y, a.loss, a.d_out, a.out = 0x1000, 0x2000, 0x3000, 0x4000   # never dereferenced
    o = (C.c_int32 * 4)()
    _lib.check(lib.regt_debug_route(C.byref(a), o), "regt_debug_route")
    cell, head, g_tiled, partials = want
    assert list(o) == [_CELL[cell], _HEAD[head], g_tiled, partials]


def test_ctypes_structs_mirror_header():
    from regt_b200 import _lib
    src = open(HEADER).read()

    def fields(struct):
        body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (struct, struct), src, re.S).group(1)
        body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
        out = []
        for decl in body.split(";"):
            decl = decl.strip()
            if not decl:
                continue
            for part in decl.split(","):
                name = re.sub(r"\[.*?\]", "", part.strip().split()[-1].lstrip("*"))
                out.append(name)
        return out
    assert fields("regt_graph_plan") == [f[0] for f in _lib.GraphPlan._fields_]
    assert fields("regt_params") == [f[0] for f in _lib.Params._fields_]
    assert fields("regt_args") == [f[0] for f in _lib.Args._fields_]
    # layout: 12 leading int32, then the plan (8-byte aligned)
    assert _lib.Args.plan.offset == 48 and C.sizeof(_lib.GraphPlan) == 24 + 13 * 8


def test_null_args_and_missing_workspace_are_rejected_without_a_gpu():
    from regt_b200 import _lib
    lib = _lib.load()
    assert lib.regt_cell_forward(None) != 0
    assert b"NULL" in lib.regt_last_error()
    a = _lib.Args()
    a.B, a.N, a.T, a.H, a.O = 1, 4, 2, 8, 1
    a.plan.N = 4
    assert lib.regt_cell_forward(C.byref(a)) != 0           # no workspace: refused before any launch
    assert b"workspace" in lib.regt_last_error()
    a.H = 7
    assert lib.regt_cell_forward(C.byref(a)) != 0 and b"multiple of 8" in lib.regt_last_error()
    assert lib.regt_workspace_bytes(C.byref(a)) > 0


def test_cpu_tensors_raise_no_fallback():
    from models import TemporalGCN
    m = TemporalGCN(8, 3, 2, hidden=16)
    x = torch.rand(5, 8, 3)
    ei = torch.tensor([[0, 1, 2], [1, 2, 3]])
    with pytest.raises(RuntimeError, match="CUDA"):
        m(x, ei, torch.ones(3))


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "regt-gcn_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dp, f)).read()
                assert "import oracle" not in txt and "from oracle" not in txt, os.path.join(dp, f)


def test_reference_state_dict_keys():
    """the 26 keys of the shipped checkpoints (SURVEY 8(b)), on the drop-in module."""
    from models import RegionalTemporalGCN
    m = RegionalTemporalGCN(8, 104, 6, 1)
    keys = set(m.state_dict().keys())
    want = {"tgnn._attention", "tgnn._weight_att1", "tgnn._weight_att2", "tgnn._bias_att1", "tgnn._bias_att2",
            "tgnn.conv.bias", "tgnn.conv.lins.0.weight", "tgnn.conv.lins.1.weight", "tgnn.linear.weight", "tgnn.linear.bias",
            "linear1.weight", "linear1.bias", "linear2.weight", "linear2.bias"}
    for g in "zrh":
        want |= {f"tgnn._base_tgcn.conv_{g}.bias", f"tgnn._base_tgcn.conv_{g}.lin.weight",
                 f"tgnn._base_tgcn.linear_{g}.weight", f"tgnn._base_tgcn.linear_{g}.bias"}
    assert keys == want and len(keys) == 26
    assert tuple(m.state_dict()["tgnn.linear.weight"].shape) == (256, 1280)
    from parity_util import shipped_checkpoint_state
    m.load_state_dict(shipped_checkpoint_state("model_in6_out1_epoch50.pt")[1], strict=True)


def test_run_py_keeps_the_reference_flags():
    """run.py:24-44 / SURVEY section 5: every flag of the reference's parser exists with the reference's default."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("regt_run", os.path.join(ROOT, "run.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    ns = mod.build_parser().parse_args([])
    ref_defaults = dict(seed=42, epochs=30, lr=1e-3, decay=1e-4, momentum=0.9, bs=32, tr=0.8, tf="available", edge_cut=None,
                        dataset_path="./dataset", checkpoint_path="../checkpoints/", dataloading_type=2, decomp_type=None,
                        num_timesteps_in=8, num_timesteps_out=4, model="TemporalGCN", is_preprocessed=False,
                        is_pretrained=False, pretrained_model="", pretrained_model_epoch="0", logs=False)
    for k, v in ref_defaults.items():
        assert getattr(ns, k) == v, k
    # the scripts' flag line parses (scripts/RegionalTemporalGCN.sh:1)
    ns = mod.build_parser().parse_args("--num_timesteps_in 6 --num_timesteps_out 1 --tr 0.2 --tf occrate --dataloading_type 2 "
                                       "--epochs 50 --decomp_type regional --model RegionalTemporalGCN".split())
    assert (ns.num_timesteps_in, ns.num_timesteps_out, ns.tr, ns.tf, ns.epochs, ns.decomp_type) == (6, 1, 0.2, "occrate", 50, "regional")


def test_spmm_partition_algorithm_on_host_arrays():
    """regt_spmm_partition's block-cutting rule, run on host arrays (no GPU): blocks cover the rows, respect the staged kernel's
    row and edge capacity, and on a graph whose node ids are ordered by region (contiguous regions, a few inter-region edges)
    the cuts fall on region borders -- far fewer edges leave their block than with uniform blocks of the same count."""
    import ctypes as C
    import numpy as np
    from regt_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(5)
    deg, W = 6, 96
    sizes = rng.integers(250, 421, size=12)                   # regions of unequal size: uniform blocks cannot line up with them
    starts = np.concatenate([[0], np.cumsum(sizes)])
    N = int(starts[-1])
    region = np.repeat(np.arange(12), sizes)
    rows, cols = [], []
    for i in range(N):
        r0, r1 = starts[region[i]], starts[region[i] + 1]
        nb = rng.integers(r0, r1, size=deg)                   # neighbours inside the node's region
        if rng.random() < 0.02:
            nb[0] = rng.integers(0, N)                        # a rare inter-region edge
        rows += [i] * (deg + 1)
        cols += [i] + list(nb)                                # self loop first, as the gcn_norm CSR has it
    rowptr = np.zeros(N + 1, dtype=np.int32)
    np.add.at(rowptr, np.asarray(rows) + 1, 1)
    rowptr = np.cumsum(rowptr).astype(np.int32)
    col = np.asarray(cols, dtype=np.int32)
    blk = np.zeros(N + 2, dtype=np.int32)
    nblk = C.c_int32(0)
    cap = np.zeros(2, dtype=np.int32)
    rc = lib.regt_debug_spmm_partition_host(rowptr.ctypes.data, col.ctypes.data, N, W, blk.ctypes.data, C.byref(nblk), cap.ctypes.data)
    _lib.check(rc, "regt_debug_spmm_partition_host")
    b = blk[: nblk.value + 1]
    assert b[0] == 0 and b[-1] == N and (np.diff(b) > 0).all()
    assert np.diff(b).max() <= cap[0] and (rowptr[b[1:]] - rowptr[b[:-1]]).max() <= cap[1]
    r = np.asarray(rows)

    def crossing(bounds):
        return int((np.searchsorted(bounds, r, side="right") != np.searchsorted(bounds, col, side="right")).sum())
    uniform = np.minimum(np.arange(nblk.value + 1) * -(-N // nblk.value), N)
    assert crossing(b) <= 0.05 * len(col) < crossing(uniform)
    assert set(b[1:-1].tolist()) <= set(starts[1:-1].tolist())   # every interior cut is a region border
