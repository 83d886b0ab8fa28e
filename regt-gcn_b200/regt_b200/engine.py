"""Host side of the cell + head: packs raw device pointers into ``regt_args`` and calls the
C-ABI (include/regt_b200.h).  PyTorch is used for device memory, streams and autograd
bookkeeping only; every arithmetic op of the path runs inside libregt_b200.so.
There is no CPU / eager fallback: non-CUDA tensors raise."""
from __future__ import annotations

import ctypes as C
import math
from typing import Dict, Optional, Sequence

import torch

from . import _lib
from .plan import GraphPlanTensors

F_IN = 8         # the kernels' feature width (REGT_F): node_features may be 1..F_IN
HEAD_HID = 128

# canonical order of the parameter tensors handed to the autograd Function
CELL_KEYS = ["conv_w0", "conv_b0", "lin_w0", "lin_b0", "conv_w1", "conv_b1", "lin_w1", "lin_b1",
             "conv_w2", "conv_b2", "lin_w2", "lin_b2"]
CHEB_KEYS = ["attention", "cheb_w0", "cheb_w1", "cheb_b"]
COMB_KEYS = ["comb_w", "comb_b"]
HEAD_KEYS = ["head_w1", "head_b1", "head_w2", "head_b2"]


def keys_for(mode: int, head: bool):
    k = list(CELL_KEYS)
    if mode != _lib.MODE_TGCN:
        k += CHEB_KEYS
    if mode == _lib.MODE_REGIONAL:
        k += COMB_KEYS
    if head:
        k += HEAD_KEYS
    return k


def _check(t: torch.Tensor, name: str, device, align: int = 16) -> torch.Tensor:
    if not t.is_cuda:
        raise RuntimeError(f"regt_b200: {name} must be a CUDA tensor (no CPU fallback exists); got {t.device}")
    if t.device != device:
        raise RuntimeError(f"regt_b200: {name} is on {t.device}, expected {device}")
    if t.dtype != torch.float32:
        raise TypeError(f"regt_b200: {name} must be float32, got {t.dtype}")
    if not t.is_contiguous() or t.data_ptr() % align:
        raise RuntimeError(f"regt_b200: {name} must be contiguous and {align}-byte aligned")
    return t


def check_features(F: int, param_width: int) -> None:
    """x's feature count F against the kernels' range and the [H, F] parameters' width."""
    if not 1 <= F <= F_IN:
        raise ValueError(f"regt_b200: node_features must be 1..{F_IN} (the kernels' feature width is {F_IN}), got {F}")
    if F != param_width:
        raise ValueError(f"regt_b200: x has {F} features per node, the model's parameters were built for {param_width}")


def _fill_params(dst: _lib.Params, tensors: Dict[str, Optional[torch.Tensor]]) -> None:
    def p(k):
        t = tensors.get(k)
        return None if t is None else t.data_ptr()
    dst.attention = p("attention")
    for g in range(3):
        dst.conv_w[g] = p(f"conv_w{g}")
        dst.conv_b[g] = p(f"conv_b{g}")
        dst.lin_w[g] = p(f"lin_w{g}")
        dst.lin_b[g] = p(f"lin_b{g}")
    for k in ("cheb_w0", "cheb_w1", "cheb_b", "comb_w", "comb_b", "head_w1", "head_b1", "head_w2", "head_b2"):
        setattr(dst, k, p(k))


class StepState:
    """everything one forward leaves behind for its backward (args struct + live tensors)."""

    def __init__(self):
        self.args = _lib.Args()
        self.keep = []          # tensors whose storage the args point into


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def build_state(mode: int, precision: int, plan: GraphPlanTensors, x: torch.Tensor, H: int, O: int,
                params: Dict[str, torch.Tensor], y: Optional[torch.Tensor] = None,
                h_ext: Optional[torch.Tensor] = None, head: bool = True,
                workspace: Optional[torch.Tensor] = None, fuse_head: bool = False,
                loss_nodes: Optional[int] = None, inference: bool = False, loss_kind: int = _lib.LOSS_MSE,
                null_value: Optional[float] = None, loss_count: Optional[torch.Tensor] = None,
                out_hidden: Optional[torch.Tensor] = None) -> StepState:
    """x [B,N,F,T] float32 CUDA.  Allocates outputs + workspace and fills ``regt_args``.
    Region shards (shard.py): x is [B,x_rows,F,T] with x_rows >= plan.N -- the plan's N owned rows
    followed by halo rows that only the plan's column indices address -- and ``loss_nodes`` is the
    node count of the full graph, so the per-rank losses and gradients add up to the unsharded ones.
    ``loss_kind`` / ``null_value`` pick the loss of the fused step (``check_loss``); ``loss_count`` [B] holds the valid
    targets of each snapshot over the full graph (region shards), else the library counts them in ``y``.
    ``out_hidden``: a caller's [B,N,H] buffer for the cell output (else one is allocated)."""
    lib = _lib.load()
    dev = x.device
    B, x_rows, Fx, T = x.shape
    # F < F_IN: the kernels read x with scalar loads, and a micro-batch slice of x need not start on 16 bytes
    _check(x, "x", dev, 16 if Fx == F_IN else 4)
    N = plan.N
    check_features(Fx, params["conv_w0"].shape[1])
    if x_rows < N or (x_rows != N and x_rows != N + getattr(plan, "n_halo", 0)):
        raise ValueError(f"regt_b200: x has {x_rows} nodes, graph plan has {N} (+{getattr(plan, 'n_halo', 0)} halo)")
    st = StepState()
    a = st.args
    a.B, a.N, a.T, a.H, a.O = B, N, T, H, O
    a.mode, a.precision, a.accumulate = mode, precision, 0
    a.fuse_head = 1 if (fuse_head and head and y is not None) else 0
    a.inference = 1 if inference else 0
    a.x_rows = x_rows
    a.F = Fx
    a.loss_nodes = int(loss_nodes) if loss_nodes else 0
    a.loss_kind = loss_kind
    if null_value is not None:
        a.loss_masked, a.loss_null = 1, float(null_value)
        if loss_count is not None:
            _check(loss_count, "loss_count", dev, 4)
            if tuple(loss_count.shape) != (B,):
                raise ValueError(f"regt_b200: loss_count must be [B]=({B},), got {tuple(loss_count.shape)}")
            a.loss_count = loss_count.data_ptr()
            st.keep.append(loss_count)
    a.plan = plan.c_struct()
    a.x = x.data_ptr()
    for k in keys_for(mode, head):
        _check(params[k], k, dev)
    _fill_params(a.p, params)
    st.keep += [x, plan, params]
    if y is not None:
        _check(y, "y", dev)
        if tuple(y.shape) != (B, N, O):
            raise ValueError(f"regt_b200: y must be [B,N,O]={B, N, O}, got {tuple(y.shape)}")
        a.y = y.data_ptr()
        st.keep.append(y)
    if h_ext is not None:
        _check(h_ext, "H", dev)
        a.h_ext = h_ext.data_ptr()
        st.keep.append(h_ext)
    if out_hidden is not None:
        _check(out_hidden, "out_hidden", dev)
        if tuple(out_hidden.shape) != (B, N, H):
            raise ValueError(f"regt_b200: out_hidden must be [B,N,H]={B, N, H}, got {tuple(out_hidden.shape)}")
    st.out_hidden = torch.empty(B, N, H, device=dev, dtype=torch.float32) if out_hidden is None else out_hidden
    a.out_hidden = st.out_hidden.data_ptr()
    if head:
        st.out = torch.empty(B, N, O, device=dev, dtype=torch.float32)
        a.out = st.out.data_ptr()
        if y is not None:
            st.loss = torch.empty(1, device=dev, dtype=torch.float32)
            st.d_out = torch.empty(B, N, O, device=dev, dtype=torch.float32)
            a.loss, a.d_out = st.loss.data_ptr(), st.d_out.data_ptr()
    nbytes = lib.regt_workspace_bytes(C.byref(a))
    if workspace is None or workspace.numel() < nbytes:
        workspace = torch.empty(nbytes, device=dev, dtype=torch.uint8)
    st.workspace = workspace
    a.workspace, a.workspace_bytes = workspace.data_ptr(), workspace.numel()
    return st


def _head_args(mode: int, precision: int, plan: GraphPlanTensors, B: int, T: int, H: int, O: int, F: int) -> _lib.Args:
    a = _lib.Args()
    a.B, a.N, a.T, a.H, a.O = B, plan.N, T, H, O
    a.mode, a.precision, a.x_rows, a.F = mode, precision, plan.N, F
    a.head_only = 1
    a.plan = plan.c_struct()
    return a


def head_workspace_bytes(mode: int, precision: int, plan: GraphPlanTensors, B: int, T: int, H: int, O: int, F: int = F_IN) -> int:
    """bytes of a head-only workspace that holds every head-only call over at most B snapshots: the training call (targets,
    fused head) is the largest, since the head-only layout takes the same buffers whichever head the route picks"""
    a = _head_args(mode, precision, plan, B, T, H, O, F)
    a.fuse_head, a.y, a.out, a.d_out, a.loss = 1, 1, 1, 1, 1     # sizes only: never dereferenced
    return int(_lib.load().regt_workspace_bytes(C.byref(a)))


def build_head_state(mode: int, precision: int, plan: GraphPlanTensors, hid: torch.Tensor, T: int, O: int,
                     params: Dict[str, torch.Tensor], out: torch.Tensor, workspace: torch.Tensor, y: Optional[torch.Tensor] = None,
                     loss: Optional[torch.Tensor] = None, d_out: Optional[torch.Tensor] = None, train: bool = False,
                     loss_kind: int = _lib.LOSS_MSE, null_value: Optional[float] = None) -> StepState:
    """``head_only`` args: the decoder head (and, with y, the loss) on a given out_hidden ``hid`` [B,N,H], with no cell; T is
    the model's period count (it sizes nothing).  ``train``: the fused head of a training step (needs y, loss, d_out); its
    regt_head_backward leaves the gradient wrt ``hid`` at the start of ``workspace``.  All buffers are the caller's."""
    lib = _lib.load()
    dev = hid.device
    B, N, H = hid.shape
    F = params["conv_w0"].shape[1]
    st = StepState()
    a = st.args = _head_args(mode, precision, plan, B, T, H, O, F)
    a.fuse_head = 1 if train else 0
    a.inference = 0 if train else 1
    a.loss_kind = loss_kind
    if null_value is not None:
        a.loss_masked, a.loss_null = 1, float(null_value)
    for k in HEAD_KEYS:
        _check(params[k], k, dev)
    _fill_params(a.p, params)
    st.out_hidden, st.out = _check(hid, "out_hidden", dev), _check(out, "out", dev)
    a.out_hidden, a.out = hid.data_ptr(), out.data_ptr()
    st.keep += [params, plan, hid, out]
    if y is not None:
        _check(y, "y", dev)
        if tuple(y.shape) != (B, N, O) or tuple(out.shape) != (B, N, O):
            raise ValueError(f"regt_b200: y and out must be [B,N,O]={B, N, O}, got {tuple(y.shape)}, {tuple(out.shape)}")
        a.y, a.loss, a.d_out = y.data_ptr(), loss.data_ptr(), d_out.data_ptr()
        st.y, st.loss, st.d_out = y, loss, d_out
    nbytes = lib.regt_workspace_bytes(C.byref(a))
    if workspace.numel() < nbytes:
        raise RuntimeError(f"regt_b200: head workspace of {workspace.numel()} bytes, the call needs {nbytes}")
    st.workspace = workspace
    a.workspace, a.workspace_bytes = workspace.data_ptr(), workspace.numel()
    return st


def run_head(st: StepState, grads: Optional[Dict[str, torch.Tensor]] = None) -> None:
    """regt_head_forward on head-only args; with ``grads`` (the head's .grad views) also regt_head_backward, which
    accumulates into them and leaves the gradient wrt out_hidden at the start of the workspace"""
    lib = _lib.load()
    a = st.args
    with torch.cuda.device(st.out.device):
        a.stream = _stream()
        _lib.check(lib.regt_head_forward(C.byref(a)), "regt_head_forward")
        if grads is not None:
            a.accumulate = 1
            _fill_params(a.g, {k: grads[k] for k in HEAD_KEYS})
            st.keep.append(grads)
            _lib.check(lib.regt_head_backward(C.byref(a)), "regt_head_backward")


def check_loss(loss: str, null_value) -> int:
    """``loss`` ("mse" or "mae") -> its ``REGT_LOSS_*`` code; ``null_value`` must be None (no mask) or a float (targets equal to
    it, or NaN, are missing; ``float("nan")`` marks only NaNs)."""
    if loss not in _lib.LOSSES:
        raise ValueError(f"regt_b200: loss must be one of {sorted(_lib.LOSSES)}, got {loss!r}")
    if null_value is not None and (isinstance(null_value, bool) or not isinstance(null_value, (int, float))):
        raise ValueError(f"regt_b200: null_value must be None (no mask) or a float, got {null_value!r}")
    return _lib.LOSSES[loss]


def loss_counts(y: torch.Tensor, null_value: float) -> torch.Tensor:
    """valid targets of each snapshot of ``y [B,N,O]`` (neither ``null_value`` nor NaN) as float32 [B]: the ``loss_count`` a
    region shard passes, taken from the full graph's targets."""
    missing = torch.isnan(y) if math.isnan(null_value) else (torch.isnan(y) | (y == null_value))
    return (~missing).sum(dim=(1, 2)).to(torch.float32)


def workspace_bytes(mode: int, precision: int, plan: GraphPlanTensors, B: int, x_rows: int, T: int, H: int, O: int,
                    F: int = F_IN, inference: bool = False) -> int:
    """bytes ``build_state`` will ask for at batch B (saved planes scale with B*N*T*H): used to size micro-batches."""
    a = _lib.Args()
    a.B, a.N, a.T, a.H, a.O = B, plan.N, T, H, O
    a.mode, a.precision, a.x_rows, a.F = mode, precision, x_rows, F
    a.fuse_head = 1
    a.inference = 1 if inference else 0
    a.plan = plan.c_struct()
    return int(_lib.load().regt_workspace_bytes(C.byref(a)))


def auto_micro_batch(mode: int, precision: int, plan: GraphPlanTensors, B: int, x_rows: int, T: int, H: int, O: int,
                     have: int = 0, F: int = F_IN) -> int:
    """largest divisor of B whose workspace fits 70 % of the free device memory (plus what a cached workspace of
    ``have`` bytes already holds); SURVEY 8d: cfg 4/5 save 63 / 157 GB of planes at full B, so they micro-batch inside the step."""
    free, _ = torch.cuda.mem_get_info()
    budget = int(0.7 * (free + have))
    for mb in sorted({d for d in range(1, B + 1) if B % d == 0}, reverse=True):
        if workspace_bytes(mode, precision, plan, mb, x_rows, T, H, O, F) <= budget:
            return mb
    return 1


def run_forward(st: StepState, head: bool = True) -> None:
    lib = _lib.load()
    with torch.cuda.device(st.out_hidden.device):     # the model may live on a device that is not the current one
        st.args.stream = _stream()
        _lib.check(lib.regt_cell_forward(C.byref(st.args)), "regt_cell_forward")
        if head:
            _lib.check(lib.regt_head_forward(C.byref(st.args)), "regt_head_forward")


def run_backward(st: StepState, grads: Dict[str, Optional[torch.Tensor]], d_out: Optional[torch.Tensor],
                 d_hidden: Optional[torch.Tensor], accumulate: bool, head: bool = True,
                 d_h_ext: Optional[torch.Tensor] = None) -> None:
    lib = _lib.load()
    a = st.args
    a.accumulate = 1 if accumulate else 0
    _fill_params(a.g, grads)
    a.d_out = None if d_out is None else d_out.data_ptr()
    a.d_hidden = None if d_hidden is None else d_hidden.data_ptr()
    a.d_h_ext = None if d_h_ext is None else d_h_ext.data_ptr()
    st.keep += [grads, d_out, d_hidden, d_h_ext]
    with torch.cuda.device(st.out_hidden.device):
        a.stream = _stream()
        # the head backward also seeds the cell gradient (G = d out_hidden) inside the workspace
        _lib.check(lib.regt_head_backward(C.byref(a)), "regt_head_backward")
        _lib.check(lib.regt_cell_backward(C.byref(a)), "regt_cell_backward")


def run_backward_x(st: StepState) -> torch.Tensor:
    """gradient wrt x [B,N,F,T] of the loss whose gradients the preceding ``run_backward`` on ``st`` consumed."""
    lib = _lib.load()
    a = st.args
    plan = st.keep[1]
    x = st.keep[0]
    with torch.cuda.device(x.device):
        xp = plan.xgrad_struct()
        nbytes = lib.regt_cell_backward_x_scratch_bytes(C.byref(a), C.byref(xp))
        scratch = torch.empty(nbytes, device=x.device, dtype=torch.uint8)
        d_x = torch.empty_like(x)
        a.stream = _stream()
        _lib.check(lib.regt_cell_backward_x(C.byref(a), C.byref(xp), d_x.data_ptr(), scratch.data_ptr(), nbytes),
                   "regt_cell_backward_x")
    return d_x


def _check_input_grad(precision: int, plan: GraphPlanTensors, x: torch.Tensor) -> None:
    """refuse, at the forward, an x that requires grad where the kernels cannot differentiate through it."""
    if precision == _lib.PREC_BF16:
        raise RuntimeError("regt_b200: the gradient wrt x is not available in precision bf16 (its kernels keep no "
                           "gate-gradient plane); use precision fp32 or tf32x3")
    if x.shape[1] != plan.N:
        raise RuntimeError("regt_b200: the gradient wrt x is not available on region shards (x has halo rows owned by "
                           "other ranks)")


class _ModelFn(torch.autograd.Function):
    """(x, *params) -> (out, out_hidden); everything runs in the C-ABI kernels."""

    @staticmethod
    def forward(ctx, mode, precision, plan, H, O, keys, x, h_ext, *tensors):
        params = dict(zip(keys, tensors))
        head = "head_w1" in params
        st = build_state(mode, precision, plan, x, H, O, params, None, h_ext, head)
        run_forward(st, head)
        ctx.st, ctx.keys, ctx.head, ctx.mode = st, keys, head, mode
        ctx.h_ext_grad = h_ext is not None and h_ext.requires_grad
        ctx.set_materialize_grads(False)
        if head:
            return st.out, st.out_hidden
        return st.out_hidden

    @staticmethod
    def backward(ctx, *gouts):
        st = ctx.st
        if ctx.head:
            d_out, d_hidden = gouts
        else:
            d_out, d_hidden = None, gouts[0]
        d_out = None if d_out is None else d_out.contiguous()
        d_hidden = None if d_hidden is None else d_hidden.contiguous()
        params = st.keep[2]
        grads = {k: torch.empty_like(params[k]) for k in ctx.keys}
        if d_out is None:
            for k in HEAD_KEYS:
                if k in grads:
                    grads[k].zero_()
        d_h_ext = None
        if ctx.h_ext_grad:
            d_h_ext = torch.empty(st.args.B, st.args.N, st.args.T, st.args.H, device=st.out_hidden.device)
        run_backward(st, grads, d_out, d_hidden, False, ctx.head, d_h_ext)
        d_x = run_backward_x(st) if ctx.needs_input_grad[6] else None
        ctx.st = None
        return (None, None, None, None, None, None, d_x, d_h_ext) + tuple(grads[k] for k in ctx.keys)


def model_apply(mode: int, precision: int, plan: GraphPlanTensors, H: int, O: int, x: torch.Tensor,
                params: Dict[str, torch.Tensor], h_ext: Optional[torch.Tensor] = None, head: bool = True):
    keys = keys_for(mode, head)
    x_grad = torch.is_grad_enabled() and x.requires_grad
    if x_grad:
        _check_input_grad(precision, plan, x)
    needs_grad = x_grad or torch.is_grad_enabled() and (any(params[k].requires_grad for k in keys) or
                                                        (h_ext is not None and h_ext.requires_grad))
    if not needs_grad:
        # run.py:208-216 / predict.py:151-172 (torch.no_grad()): forward only -- the fused kernels keep no activations
        st = build_state(mode, precision, plan, x, H, O, params, None, h_ext, head, inference=True)
        run_forward(st, head)
        return (st.out, st.out_hidden) if head else st.out_hidden
    return _ModelFn.apply(mode, precision, plan, H, O, keys, x, h_ext, *[params[k] for k in keys])
