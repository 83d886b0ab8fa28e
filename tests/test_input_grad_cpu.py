"""CPU tests of the input-gradient boundary (include/regt_b200.h, regt_cell_backward_x): the ctypes mirror of
``regt_xgrad_plan`` matches the header, and the entry point refuses what it cannot differentiate without a GPU."""
import ctypes as C
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "regt_b200.h")


def _fields(struct):
    src = open(HEADER).read()
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (struct, struct), src, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    return [d.strip().split()[-1].lstrip("*") for d in body.split(";") if d.strip()]


def test_xgrad_plan_struct_mirrors_header():
    from regt_b200 import _lib
    assert _fields("regt_xgrad_plan") == [f[0] for f in _lib.XgradPlan._fields_]
    assert C.sizeof(_lib.XgradPlan) == 16 + 3 * 8 and _lib.XgradPlan.rowptr.offset == 16


def test_backward_x_refusals_name_the_reason():
    from regt_b200 import _lib
    lib = _lib.load()
    a = _lib.Args()
    a.B, a.N, a.T, a.H, a.O = 1, 4, 2, 8, 1
    a.plan.N = 4
    xp = _lib.XgradPlan()
    xp.N, xp.n_src = 4, 8
    a.workspace_bytes = lib.regt_workspace_bytes(C.byref(a))
    a.workspace = 256                      # never dereferenced: every case below is refused on the host first
    for field, value, reason in (("precision", _lib.PREC_BF16, b"bf16"), ("x_rows", 6, b"region shards"),
                                 ("inference", 1, b"inference=1")):
        setattr(a, field, value)
        assert lib.regt_cell_backward_x(C.byref(a), C.byref(xp), 256, 256, 1 << 20) != 0
        assert reason in lib.regt_last_error(), lib.regt_last_error()
        setattr(a, field, 0)
    assert lib.regt_cell_backward_x(C.byref(a), C.byref(xp), 256, 256, 1 << 20) != 0   # plan arrays missing
    assert b"transposed plan" in lib.regt_last_error()
    assert lib.regt_cell_backward_x_scratch_bytes(C.byref(a), C.byref(xp)) > 0
