"""Static-graph plan: edge_index -> CSR + normalised values, built ONCE per static graph by
the K1 kernels (csrc/plan.cu) and cached.  The reference rebuilds the same normalisation
3*T + R*T times per sample (models/utils.py:169-181, models/RegionalTemporalGCN.py:136-140)."""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import torch

from . import _lib


def _stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


class GraphPlanTensors:
    """owns the device arrays behind a ``regt_graph_plan``."""

    def __init__(self, device: torch.device, N: int):
        self.device, self.N = device, N
        self.R = 1
        self.nnz_gcn = self.nnz_cheb = self.nseg = 0
        self.t = {}
        self.xg = None          # transposed operator of the input gradient (xgrad_struct), built on first use

    def c_struct(self) -> _lib.GraphPlan:
        p = _lib.GraphPlan()
        p.N, p.nnz_gcn, p.nnz_cheb, p.nseg, p.R = self.N, self.nnz_gcn, self.nnz_cheb, self.nseg, self.R
        for k in ("g_rowptr", "g_col", "g_val", "c_rowptr", "c_col", "c_val", "c_reg", "seg_ptr", "seg_eptr",
                  "seg_reg", "seg_node", "rseg_ptr", "rseg_list"):
            setattr(p, k, _ptr(self.t.get(k)))
        return p

    def xgrad_struct(self) -> _lib.XgradPlan:
        """the ``regt_xgrad_plan`` of this graph (A_hat^T and the regional operators transposed, one CSR by input node).
        Built on the first backward that asks for the gradient wrt x and kept with the plan, so the identity and the
        content entries of the plan cache both reach it."""
        if self.xg is None:
            if torch.cuda.is_current_stream_capturing():
                raise RuntimeError("regt_b200: the transposed graph operator of the input gradient is built on the first "
                                   "backward that needs it; run one such backward outside CUDA-graph capture first")
            lib = _lib.load()
            ps = self.c_struct()
            n = self.N + self.nnz_gcn + self.nnz_cheb
            dev = self.device
            rowptr = torch.empty(self.N + 1, device=dev, dtype=torch.int32)
            col = torch.empty(n, device=dev, dtype=torch.int32)
            val = torch.empty(n, device=dev, dtype=torch.float32)
            wsb = lib.regt_xgrad_plan_workspace_bytes(C.byref(ps))
            with torch.cuda.device(dev):
                ws = torch.empty(wsb, device=dev, dtype=torch.uint8)
                rc = lib.regt_xgrad_plan_build(C.byref(ps), rowptr.data_ptr(), col.data_ptr(), val.data_ptr(), ws.data_ptr(),
                                               wsb, _stream_ptr())
                _lib.check(rc, "regt_xgrad_plan_build")
            self.xg = dict(nnz=n, n_src=2 * self.N + self.nseg, rowptr=rowptr, col=col, val=val)
        p = _lib.XgradPlan()
        p.N, p.nnz, p.n_src = self.N, self.xg["nnz"], self.xg["n_src"]
        p.rowptr, p.col, p.val = (self.xg[k].data_ptr() for k in ("rowptr", "col", "val"))
        return p


def build_gcn(plan: GraphPlanTensors, edge_index: torch.Tensor, edge_weight: Optional[torch.Tensor]) -> None:
    lib = _lib.load()
    dev, N = plan.device, plan.N
    ei = edge_index.to(device=dev, dtype=torch.int64).contiguous()
    ew = None if edge_weight is None else edge_weight.to(device=dev, dtype=torch.float32).contiguous()
    E = int(ei.shape[1])
    if E and (int(ei.min()) < 0 or int(ei.max()) >= N):
        raise IndexError(f"edge_index out of range for {N} nodes")
    i32 = dict(device=dev, dtype=torch.int32)
    rowptr = torch.empty(N + 1, **i32)
    col = torch.empty(E + N, **i32)
    eid = torch.empty(E + N, **i32)
    val = torch.empty(E + N, device=dev, dtype=torch.float32)
    wsb = lib.regt_plan_workspace_bytes(N, E)
    ws = torch.empty(wsb, device=dev, dtype=torch.uint8)
    nnz = C.c_int32(0)
    with torch.cuda.device(dev):
        rc = lib.regt_gcn_plan_build(ei.data_ptr(), _ptr(ew), E, N, rowptr.data_ptr(), col.data_ptr(), val.data_ptr(),
                                     eid.data_ptr(), C.byref(nnz), ws.data_ptr(), wsb, _stream_ptr())
    _lib.check(rc, "regt_gcn_plan_build")
    plan.nnz_gcn = nnz.value
    plan.t.update(g_rowptr=rowptr, g_col=col[:nnz.value], g_val=val[:nnz.value], g_eid=eid[:nnz.value])


def build_cheb(plan: GraphPlanTensors, edge_lists: Sequence[torch.Tensor],
               weight_lists: Sequence[Optional[torch.Tensor]]) -> None:
    lib = _lib.load()
    dev, N = plan.device, plan.N
    R = len(edge_lists)
    assert R >= 1
    eis = [e.to(device=dev, dtype=torch.int64).reshape(2, -1) for e in edge_lists]
    ei = torch.cat(eis, dim=1).contiguous()
    if all(w is None for w in weight_lists):
        ew = None
    else:
        ws_ = [torch.ones(e.shape[1], device=dev) if w is None else w.to(device=dev, dtype=torch.float32).reshape(-1)
               for e, w in zip(eis, weight_lists)]
        ew = torch.cat(ws_).contiguous()
    E = int(ei.shape[1])
    if E and (int(ei.min()) < 0 or int(ei.max()) >= N):
        raise IndexError(f"regional edge_index out of range for {N} nodes")
    lp = [0]
    for e in eis:
        lp.append(lp[-1] + int(e.shape[1]))
    list_ptr = (C.c_int64 * (R + 1))(*lp)
    i32 = dict(device=dev, dtype=torch.int32)
    names = ["c_rowptr", "c_col", "c_val", "c_reg", "c_eid", "seg_ptr", "seg_eptr", "seg_reg", "seg_node",
             "rseg_ptr", "rseg_list", "region_of"]
    sizes = [N + 1, E + 1, E + 1, E + 1, E + 1, N + 1, E + 2, E + 1, E + 1, R + 1, E + 1, N]
    t = {n: (torch.zeros(s, device=dev, dtype=torch.float32) if n == "c_val" else torch.zeros(s, **i32))
         for n, s in zip(names, sizes)}
    wsb = lib.regt_plan_workspace_bytes(N, E + R + 8)
    ws = torch.empty(wsb, device=dev, dtype=torch.uint8)
    counts = (C.c_int32 * 2)(0, 0)
    with torch.cuda.device(dev):
        rc = lib.regt_cheb_plan_build(ei.data_ptr(), _ptr(ew), list_ptr, R, E, N, *[t[n].data_ptr() for n in names],
                                      counts, ws.data_ptr(), wsb, _stream_ptr())
    _lib.check(rc, "regt_cheb_plan_build")
    nnz, nseg = counts[0], counts[1]
    plan.R, plan.nnz_cheb, plan.nseg = R, nnz, nseg
    plan.t.update(c_rowptr=t["c_rowptr"], c_col=t["c_col"][:max(nnz, 1)], c_val=t["c_val"][:max(nnz, 1)],
                  c_reg=t["c_reg"][:max(nnz, 1)], c_eid=t["c_eid"][:nnz], seg_ptr=t["seg_ptr"],
                  seg_eptr=t["seg_eptr"][:nseg + 1], seg_reg=t["seg_reg"][:max(nseg, 1)],
                  seg_node=t["seg_node"][:max(nseg, 1)], rseg_ptr=t["rseg_ptr"],
                  rseg_list=t["rseg_list"][:max(nseg, 1)], region_of=t["region_of"])


# ---- plan cache (the graph is static across snapshots) ----
# Level 1: identity of the graph tensors (no device work, no sync) -- loops that pass the same tensors every step.
# Level 2: CONTENT of the graph tensors.  The reference's loop does ``batch.to(device)`` per snapshot (run.py:172), which
# makes a NEW edge_index tensor every time: identity never hits there.  On an identity miss the lists are hashed on the
# device (two position-weighted int64 sums per tensor, one small D2H read) and the plan is looked up by that; K1 itself
# runs once per distinct graph.
_CACHE: dict = {}
_CONTENT: dict = {}


def _key(t: Optional[torch.Tensor]):
    return None if t is None else (t.data_ptr(), tuple(t.shape), t._version, str(t.device))


def _content_key(tensors) -> tuple:
    parts, shapes = [], []
    for t in tensors:
        if t is None:
            shapes.append(None)
            continue
        shapes.append((tuple(t.shape), str(t.dtype)))
        if t.numel():
            v = t.reshape(-1)
            parts.append(v.view(torch.int32).to(torch.int64) if v.dtype == torch.float32 else v.to(torch.int64))
    if not parts:
        return (tuple(shapes), ())
    bits = torch.cat(parts)          # shapes are part of the key, so the concatenation is unambiguous
    w = torch.arange(1, bits.numel() + 1, device=bits.device, dtype=torch.int64)
    # two position-weighted wrap-around int64 sums = a 128-bit fingerprint, one small D2H read
    fp = torch.stack([(bits * w).sum(), ((bits + w * 2654435761) * (bits ^ (w << 17))).sum()])
    return (tuple(shapes), tuple(fp.cpu().tolist()))


def get_plan(N: int, device: torch.device, edge_index: torch.Tensor, edge_weight: Optional[torch.Tensor],
             reg_edge_index: Sequence[torch.Tensor], reg_edge_weight: Sequence[Optional[torch.Tensor]],
             need_cheb: bool = True) -> GraphPlanTensors:
    """gcn plan from (edge_index, edge_weight); cheb plan from the regional lists."""
    if torch.device(device).type != "cuda":
        raise RuntimeError(f"regt_b200 runs on CUDA devices only (no CPU fallback exists); tensors are on {device}")
    key = (N, str(device), _key(edge_index), _key(edge_weight), tuple(_key(e) for e in reg_edge_index),
           tuple(_key(w) for w in reg_edge_weight), need_cheb)
    hit = _CACHE.get(key)
    if hit is not None:
        return hit[0]
    ckey = None
    if not torch.cuda.is_current_stream_capturing():
        with torch.cuda.device(device):
            ckey = (N, str(device), need_cheb,
                    _content_key([edge_index, edge_weight, *reg_edge_index, *reg_edge_weight]))
        plan = _CONTENT.get(ckey)
        if plan is not None:
            # also by identity: a CUDA-graph capture of a step with these tensors must find the plan without the device
            # work of hashing (or building) it, even when their content was first seen through other tensors
            _remember(key, plan, edge_index, edge_weight, reg_edge_index, reg_edge_weight)
            return plan
    plan = GraphPlanTensors(device, N)
    build_gcn(plan, edge_index, edge_weight)
    if need_cheb:
        build_cheb(plan, reg_edge_index, reg_edge_weight)
    _remember(key, plan, edge_index, edge_weight, reg_edge_index, reg_edge_weight)
    if len(_CONTENT) > 16:
        _CONTENT.clear()
    if ckey is not None:
        _CONTENT[ckey] = plan
    return plan


def _remember(key, plan, edge_index, edge_weight, reg_edge_index, reg_edge_weight) -> None:
    if len(_CACHE) > 64:
        _CACHE.clear()
    # keep the key tensors alive so data_ptr() cannot be recycled while the entry lives
    _CACHE[key] = (plan, edge_index, edge_weight, list(reg_edge_index), list(reg_edge_weight))


_PARTS: dict = {}     # (rowptr ptr, col ptr, versions, N, width) -> (rowptr, col, blk_ptr, nblk): the staged SpMM's row partition


def spmm_partition(rowptr: torch.Tensor, col: torch.Tensor, N: int, width: int):
    """(blk_ptr, nblk) of regt_spmm_partition for this CSR, built once per static graph (None, 0 when the rows are too
    wide for the staged kernel)."""
    lib = _lib.load()
    key = (rowptr.data_ptr(), col.data_ptr(), rowptr._version, col._version, int(N), int(width))
    hit = _PARTS.get(key)
    if hit is not None:
        return hit[2], hit[3]
    cap = lib.regt_spmm_partition_capacity(int(N), int(width))
    blk, nblk = None, 0
    if cap > 0:
        import ctypes as C
        blk = torch.empty(cap, dtype=torch.int32, device=rowptr.device)
        n = C.c_int32(0)
        with torch.cuda.device(rowptr.device):
            rc = lib.regt_spmm_partition(rowptr.data_ptr(), col.data_ptr(), int(N), int(width), blk.data_ptr(), C.byref(n), _stream_ptr())
        _lib.check(rc, "regt_spmm_partition")
        nblk = int(n.value)
        blk = blk[: nblk + 1]
    if len(_PARTS) > 16:
        _PARTS.clear()
    _PARTS[key] = (rowptr, col, blk, nblk)      # the key tensors stay alive: their data_ptr() cannot be recycled
    return blk, nblk


def spmm_f8(rowptr: torch.Tensor, col: torch.Tensor, val: torch.Tensor, x: torch.Tensor, partition: bool = True) -> torch.Tensor:
    """y[b,n,:] = sum_e val[e] x[b,col[e],:] over rows of F*T floats (x [B,N,F,T] or [B,N,W]).  With ``partition`` the row
    blocks of the staged kernel come from regt_spmm_partition (cached per CSR); the sums are bit-identical either way."""
    lib = _lib.load()
    assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous()
    B, N = x.shape[0], x.shape[1]
    width = x[0, 0].numel()
    y = torch.empty_like(x)
    blk, nblk = (None, 0)
    if partition and width % 4 == 0 and B * N >= 4096 and x.data_ptr() % 16 == 0:
        blk, nblk = spmm_partition(rowptr, col, N, width)
    with torch.cuda.device(x.device):
        if nblk > 0:
            rc = lib.regt_spmm_f8_blocked(rowptr.data_ptr(), col.data_ptr(), val.data_ptr(), x.data_ptr(), y.data_ptr(), B, N, width,
                                          blk.data_ptr(), nblk, _stream_ptr())
        else:
            rc = lib.regt_spmm_f8(rowptr.data_ptr(), col.data_ptr(), val.data_ptr(), x.data_ptr(), y.data_ptr(), B, N, width,
                                  _stream_ptr())
    _lib.check(rc, "regt_spmm_f8")
    return y
