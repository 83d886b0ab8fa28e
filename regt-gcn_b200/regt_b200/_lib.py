"""ctypes binding of libregt_b200.so (include/regt_b200.h).  No torch types cross the ABI:
only raw device pointers, sizes and the CUDA stream handle.

The library is required: there is no CPU or eager-PyTorch fallback.  If it is missing it is
built in-tree with nvcc (csrc/build.py); if that fails the error is raised as is."""
from __future__ import annotations

import ctypes as C
import os
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.normpath(os.path.join(_HERE, "..", "csrc"))

c_i32p = C.POINTER(C.c_int32)
c_i64p = C.POINTER(C.c_int64)
vp = C.c_void_p


class GraphPlan(C.Structure):
    _fields_ = [("N", C.c_int32), ("nnz_gcn", C.c_int32), ("nnz_cheb", C.c_int32), ("nseg", C.c_int32),
                ("R", C.c_int32), ("_pad", C.c_int32),
                ("g_rowptr", vp), ("g_col", vp), ("g_val", vp),
                ("c_rowptr", vp), ("c_col", vp), ("c_val", vp), ("c_reg", vp),
                ("seg_ptr", vp), ("seg_eptr", vp), ("seg_reg", vp), ("seg_node", vp),
                ("rseg_ptr", vp), ("rseg_list", vp)]


class XgradPlan(C.Structure):
    _fields_ = [("N", C.c_int32), ("nnz", C.c_int32), ("n_src", C.c_int32), ("_pad", C.c_int32),
                ("rowptr", vp), ("col", vp), ("val", vp)]


class Params(C.Structure):
    _fields_ = [("attention", vp), ("conv_w", vp * 3), ("conv_b", vp * 3), ("lin_w", vp * 3), ("lin_b", vp * 3),
                ("cheb_w0", vp), ("cheb_w1", vp), ("cheb_b", vp), ("comb_w", vp), ("comb_b", vp),
                ("head_w1", vp), ("head_b1", vp), ("head_w2", vp), ("head_b2", vp)]


class Args(C.Structure):
    _fields_ = [("B", C.c_int32), ("N", C.c_int32), ("T", C.c_int32), ("H", C.c_int32), ("O", C.c_int32),
                ("mode", C.c_int32), ("precision", C.c_int32), ("accumulate", C.c_int32),
                ("fuse_head", C.c_int32), ("x_rows", C.c_int32), ("loss_nodes", C.c_int32), ("inference", C.c_int32),
                ("plan", GraphPlan),
                ("x", vp), ("y", vp), ("h_ext", vp),
                ("p", Params), ("g", Params),
                ("out_hidden", vp), ("out", vp), ("loss", vp), ("d_out", vp), ("d_hidden", vp), ("d_h_ext", vp),
                ("workspace", vp), ("workspace_bytes", C.c_size_t), ("stream", vp), ("F", C.c_int32),
                ("loss_kind", C.c_int32), ("loss_masked", C.c_int32), ("loss_null", C.c_float), ("loss_count", vp),
                ("head_only", C.c_int32)]


MODE_A3TGCN, MODE_REGIONAL, MODE_TGCN = 0, 1, 2
LOSS_MSE, LOSS_MAE = 0, 1
LOSSES = {"mse": LOSS_MSE, "mae": LOSS_MAE}
PREC_FP32, PREC_TF32X3, PREC_BF16 = 0, 1, 2
PRECISIONS = {"fp32": PREC_FP32, "tf32x3": PREC_TF32X3, "bf16": PREC_BF16}

EXPORTS = ["regt_version", "regt_last_error", "regt_launch_count", "regt_plan_workspace_bytes",
           "regt_gcn_plan_build", "regt_cheb_plan_build", "regt_spmm_f8", "regt_spmm_partition_capacity", "regt_spmm_partition",
           "regt_spmm_f8_blocked", "regt_gather_rows", "regt_scatter_rows", "regt_workspace_bytes",
           "regt_cell_forward", "regt_head_forward", "regt_head_backward", "regt_cell_backward",
           "regt_xgrad_plan_workspace_bytes", "regt_xgrad_plan_build", "regt_cell_backward_x_scratch_bytes",
           "regt_cell_backward_x",
           "regt_profile", "regt_profile_begin", "regt_profile_read",
           "regt_comm_region_bytes", "regt_comm_data_offset", "regt_comm_alloc", "regt_comm_free", "regt_comm_export",
           "regt_comm_import", "regt_comm_unimport", "regt_peer_allreduce_f32", "regt_peer_push_max_floats", "regt_comm_error",
           "regt_window_gather", "regt_rmsprop_step", "regt_eval_metrics", "regt_eval_metrics_masked",
           "regt_combine_scratch_bytes", "regt_combine_forward", "regt_combine_backward"]

_lib = None


def lib_path() -> str:
    return os.path.normpath(os.path.join(_HERE, "..", "lib", "libregt_b200.so"))


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        sys.path.insert(0, _CSRC)
        try:
            import build as _build  # csrc/build.py
            _build.build()
        finally:
            sys.path.remove(_CSRC)
    lib = C.CDLL(path)
    lib.regt_version.restype = C.c_int
    lib.regt_last_error.restype = C.c_char_p
    lib.regt_launch_count.restype = C.c_int64
    lib.regt_launch_count.argtypes = [C.c_int]
    lib.regt_plan_workspace_bytes.restype = C.c_size_t
    lib.regt_plan_workspace_bytes.argtypes = [C.c_int64, C.c_int64]
    lib.regt_gcn_plan_build.restype = C.c_int
    lib.regt_gcn_plan_build.argtypes = [vp, vp, C.c_int64, C.c_int64, vp, vp, vp, vp, c_i32p, vp, C.c_size_t, vp]
    lib.regt_cheb_plan_build.restype = C.c_int
    lib.regt_cheb_plan_build.argtypes = [vp, vp, c_i64p, C.c_int32, C.c_int64, C.c_int64] + [vp] * 12 + \
                                        [c_i32p, vp, C.c_size_t, vp]
    lib.regt_spmm_f8.restype = C.c_int
    lib.regt_spmm_f8.argtypes = [vp, vp, vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, vp]
    lib.regt_spmm_partition_capacity.restype = C.c_int32
    lib.regt_spmm_partition_capacity.argtypes = [C.c_int32, C.c_int32]
    lib.regt_spmm_partition.restype = C.c_int
    lib.regt_spmm_partition.argtypes = [vp, vp, C.c_int32, C.c_int32, vp, c_i32p, vp]
    lib.regt_spmm_f8_blocked.restype = C.c_int
    lib.regt_spmm_f8_blocked.argtypes = [vp, vp, vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, vp, C.c_int32, vp]
    for name in ("regt_gather_rows", "regt_scatter_rows"):
        fn = getattr(lib, name)
        fn.restype = C.c_int
        fn.argtypes = [vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, vp]
    lib.regt_workspace_bytes.restype = C.c_size_t
    lib.regt_workspace_bytes.argtypes = [C.POINTER(Args)]
    for name in ("regt_cell_forward", "regt_head_forward", "regt_head_backward", "regt_cell_backward"):
        fn = getattr(lib, name)
        fn.restype = C.c_int
        fn.argtypes = [C.POINTER(Args)]
    lib.regt_xgrad_plan_workspace_bytes.restype = C.c_size_t
    lib.regt_xgrad_plan_workspace_bytes.argtypes = [C.POINTER(GraphPlan)]
    lib.regt_xgrad_plan_build.restype = C.c_int
    lib.regt_xgrad_plan_build.argtypes = [C.POINTER(GraphPlan), vp, vp, vp, vp, C.c_size_t, vp]
    lib.regt_cell_backward_x_scratch_bytes.restype = C.c_size_t
    lib.regt_cell_backward_x_scratch_bytes.argtypes = [C.POINTER(Args), C.POINTER(XgradPlan)]
    lib.regt_cell_backward_x.restype = C.c_int
    lib.regt_cell_backward_x.argtypes = [C.POINTER(Args), C.POINTER(XgradPlan), vp, vp, C.c_size_t]
    lib.regt_profile.restype = C.c_int
    lib.regt_profile.argtypes = [C.c_int, vp]
    lib.regt_profile_begin.restype = C.c_int
    lib.regt_profile_begin.argtypes = [vp]
    lib.regt_profile_read.restype = C.c_int
    lib.regt_profile_read.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(C.c_float), C.c_int]
    lib.regt_comm_region_bytes.restype = C.c_size_t
    lib.regt_comm_region_bytes.argtypes = [C.c_int64]
    lib.regt_comm_data_offset.restype = C.c_size_t
    lib.regt_comm_alloc.restype = C.c_int
    lib.regt_comm_alloc.argtypes = [C.c_size_t, C.POINTER(C.c_void_p)]
    lib.regt_comm_free.restype = C.c_int
    lib.regt_comm_free.argtypes = [vp]
    lib.regt_comm_export.restype = C.c_int
    lib.regt_comm_export.argtypes = [vp, C.POINTER(C.c_ubyte)]
    lib.regt_comm_import.restype = C.c_int
    lib.regt_comm_import.argtypes = [C.POINTER(C.c_ubyte), C.POINTER(C.c_void_p)]
    lib.regt_comm_unimport.restype = C.c_int
    lib.regt_comm_unimport.argtypes = [vp]
    lib.regt_peer_allreduce_f32.restype = C.c_int
    lib.regt_peer_allreduce_f32.argtypes = [C.POINTER(C.c_void_p), C.c_int32, C.c_int32, C.c_int64, vp, vp, vp]
    lib.regt_peer_push_max_floats.restype = C.c_int64
    lib.regt_comm_error.restype = C.c_int
    lib.regt_comm_error.argtypes = [vp]
    lib.regt_window_gather.restype = C.c_int
    lib.regt_window_gather.argtypes = [vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_int32, vp, vp, vp]
    lib.regt_rmsprop_step.restype = C.c_int
    lib.regt_rmsprop_step.argtypes = [vp, vp, vp, C.c_int64, C.c_float, C.c_float, C.c_float, C.c_float, vp]
    lib.regt_eval_metrics.restype = C.c_int
    lib.regt_eval_metrics.argtypes = [vp, vp, C.c_int32, C.c_int64, C.c_double, vp, vp]
    lib.regt_eval_metrics_masked.restype = C.c_int
    lib.regt_eval_metrics_masked.argtypes = [vp, vp, C.c_int32, C.c_int64, C.c_double, C.c_float, vp, vp]
    lib.regt_combine_scratch_bytes.restype = C.c_size_t
    lib.regt_combine_scratch_bytes.argtypes = [C.c_int32]
    lib.regt_combine_forward.restype = C.c_int
    lib.regt_combine_forward.argtypes = [vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int64, vp, vp]
    lib.regt_combine_backward.restype = C.c_int
    lib.regt_combine_backward.argtypes = [vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int64, vp, vp, vp, C.c_size_t, vp]
    lib.regt_debug_gemm_nt_tma.restype = C.c_int
    lib.regt_debug_gemm_nt_tma.argtypes = [vp, C.c_int64, vp, C.c_int64, vp, C.c_int64, C.c_int64, C.c_int32, C.c_int32, vp, vp]
    lib.regt_debug_gemm_tn_tma.restype = C.c_int
    lib.regt_debug_gemm_tn_tma.argtypes = [vp, C.c_int64, vp, C.c_int64, vp, C.c_int64, C.c_int32, C.c_int32, C.c_int32,
                                           vp, C.c_int64, vp, vp]
    lib.regt_debug_gemm_nt_bf16.restype = C.c_int
    lib.regt_debug_gemm_nt_bf16.argtypes = lib.regt_debug_gemm_nt_tma.argtypes
    lib.regt_debug_gemm_tn_bf16.restype = C.c_int
    lib.regt_debug_gemm_tn_bf16.argtypes = lib.regt_debug_gemm_tn_tma.argtypes
    lib.regt_debug_gemm_tn_multi.restype = C.c_int
    lib.regt_debug_gemm_tn_multi.argtypes = [vp, C.c_int64, C.c_int64, C.c_int32, vp, vp, vp, vp, C.c_int32, vp, vp, vp]
    lib.regt_debug_gemm_tn_multi_bf16.restype = C.c_int
    lib.regt_debug_gemm_tn_multi_bf16.argtypes = lib.regt_debug_gemm_tn_multi.argtypes
    lib.regt_debug_spmm_partition_host.restype = C.c_int
    lib.regt_debug_spmm_partition_host.argtypes = [vp, vp, C.c_int32, C.c_int32, vp, c_i32p, vp]
    lib.regt_debug_gemm_kt.restype = C.c_int
    lib.regt_debug_gemm_kt.argtypes = [vp, C.c_int64, C.c_int32, vp, vp, vp, vp, vp, vp, C.c_int32, vp]
    lib.regt_debug_f_timestamps.restype = C.c_int
    lib.regt_debug_f_timestamps.argtypes = [vp]
    lib.regt_debug_umma_selftest.restype = C.c_int
    lib.regt_debug_umma_selftest.argtypes = [C.c_int, C.c_int, vp, vp, vp, C.c_int, C.c_int, vp]
    lib.regt_debug_tc_split.restype = C.c_int
    lib.regt_debug_tc_split.argtypes = [C.c_int32, C.c_int32, C.c_int32, c_i32p]
    lib.regt_debug_route.restype = C.c_int
    lib.regt_debug_route.argtypes = [C.POINTER(Args), c_i32p]
    _lib = lib
    return lib


def profile_read(max_n: int = 4096):
    """-> list of (kernel name, ms) recorded since regt_profile(1, stream)."""
    lib = load()
    names = C.create_string_buffer(max_n * 24)
    ms = (C.c_float * max_n)()
    n = lib.regt_profile_read(names, len(names), ms, max_n)
    if n < 0:
        raise RuntimeError("regt_profile_read failed")
    return list(zip(names.value.decode().split("\n")[:n], [ms[i] for i in range(n)]))


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise RuntimeError(f"{what} failed ({rc}): {load().regt_last_error().decode()}")
