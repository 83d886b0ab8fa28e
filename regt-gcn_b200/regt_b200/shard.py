"""Region sharding of the hot path across GPUs (SURVEY.md 8(e); one process per GPU).

The reference is single-device (run.py:73).  What makes the path shard: every output row depends
only on the 1-hop in-neighbourhood of the raw input ``x`` (the hidden state is not recurrent and is
never propagated over the graph), and the regional edge lists are disjoint subgraphs.  So

  * regions -> ranks by longest-processing-time bin packing on node counts (deterministic,
    bit-exact: ``lpt_partition``); a rank owns the nodes of its regions;
  * a rank's input is ``x[:, own | halo]``: its owned rows followed by the halo rows -- sources of
    full-graph in-edges of owned nodes that live on other ranks.  ``x`` is input data, so the halo
    is read from the rank's own copy of the input: NO activation exchange;
  * the rank's static-graph plan is the owned ROWS of the global gcn_norm CSR (the normalisation
    needs global degrees, so the global plan is built once by K1 and sliced) with columns renumbered
    into the local [own | halo] order, plus the Chebyshev plan of the owned regional lists;
  * the exchange step: ONE sum all-reduce of the flat shared-weight gradient buffer (+ the scalar
    loss) per step, and -- only when the caller wants full-N outputs -- an all-gather of the
    per-rank ``[B, n_own, H+O]`` outputs, scattered back into global node order.

Host logic (partition, halo, CSR slicing, reassembly) is plain numpy/torch and runs on CPU tensors
too, which is how tests/test_shard_cpu.py covers it with world_size-2 gloo groups."""
from __future__ import annotations

import os
import sys
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from .plan import GraphPlanTensors, build_cheb, build_gcn


# ------------------------------------------------------------------------------------------
# partition (host, integer, bit-exact)
# ------------------------------------------------------------------------------------------
def region_of_nodes(reg_edge_index: Sequence, N: int) -> np.ndarray:
    """int32 [N]: regional list that touches node n (as source or target), -1 if none, -2 if more
    than one list does (then the decomposition is not regional: models/RegionalTemporalGCN.py's
    ``random`` decomposition, load_dataset.py:324-329)."""
    ro = np.full(N, -1, dtype=np.int32)
    for r, ei in enumerate(reg_edge_index):
        e = ei.detach().cpu().numpy() if isinstance(ei, torch.Tensor) else np.asarray(ei)
        if e.size == 0:
            continue
        nodes = np.unique(e.reshape(2, -1))
        clash = (ro[nodes] != -1) & (ro[nodes] != r)
        ro[nodes[clash]] = -2
        ro[nodes[~clash]] = r
    return ro


def lpt_partition(sizes: Sequence[int], world: int) -> np.ndarray:
    """items -> ranks, longest processing time first: items sorted by (-size, id); each goes to the
    least-loaded rank, ties -> lowest rank id.  Returns int32 owner[item]."""
    sizes = [int(s) for s in sizes]
    order = sorted(range(len(sizes)), key=lambda r: (-sizes[r], r))
    load = [0] * world
    owner = np.zeros(len(sizes), dtype=np.int32)
    for r in order:
        k = min(range(world), key=lambda i: (load[i], i))
        owner[r] = k
        load[k] += sizes[r]
    return owner


@dataclass
class RegionShard:
    rank: int
    world: int
    N: int                    # nodes of the full graph
    region_owner: np.ndarray  # int32 [R]   rank of every regional list
    node_owner: np.ndarray    # int32 [N]   rank of every node
    own: np.ndarray           # int64 [n_own]  owned global node ids, ascending
    halo: np.ndarray          # int64 [n_halo] halo global node ids, ascending
    counts: np.ndarray        # int64 [world]  n_own of every rank

    @property
    def n_own(self) -> int:
        return int(self.own.size)

    @property
    def n_halo(self) -> int:
        return int(self.halo.size)

    @property
    def perm(self) -> np.ndarray:
        """global ids in local row order: owned rows first, then halo rows."""
        return np.concatenate([self.own, self.halo])


def make_shard(N: int, edge_index, reg_edge_index: Sequence, rank: int, world: int) -> RegionShard:
    """deterministic on every rank (no communication): same inputs -> same partition."""
    if not (0 <= rank < world):
        raise ValueError(f"rank {rank} outside world of {world}")
    ro = region_of_nodes(reg_edge_index, N)
    if (ro == -2).any():
        raise ValueError("region sharding needs a regional decomposition (every node in at most one regional "
                         f"edge list); {int((ro == -2).sum())} nodes appear in several lists -- shard by batch instead")
    R = len(reg_edge_index)
    sizes = np.bincount(ro[ro >= 0], minlength=R)
    # nodes that no regional list touches are singleton items after the regions, in id order
    orphans = np.nonzero(ro == -1)[0]
    owner_all = lpt_partition(list(sizes) + [1] * len(orphans), world)
    region_owner = owner_all[:R].astype(np.int32)
    node_owner = np.empty(N, dtype=np.int32)
    node_owner[ro >= 0] = region_owner[ro[ro >= 0]]
    node_owner[orphans] = owner_all[R:]
    own = np.nonzero(node_owner == rank)[0].astype(np.int64)
    e = edge_index.detach().cpu().numpy() if isinstance(edge_index, torch.Tensor) else np.asarray(edge_index)
    src, dst = e[0], e[1]
    m = (node_owner[dst] == rank) & (node_owner[src] != rank)
    halo = np.unique(src[m]).astype(np.int64)
    counts = np.bincount(node_owner, minlength=world).astype(np.int64)
    return RegionShard(rank, world, N, region_owner, node_owner, own, halo, counts)


# ------------------------------------------------------------------------------------------
# local plan = owned rows of the global plan (torch ops: CPU or CUDA tensors)
# ------------------------------------------------------------------------------------------
def slice_csr(rowptr: torch.Tensor, col: torch.Tensor, val: torch.Tensor, own: torch.Tensor,
              lut: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """rows ``own`` of a CSR, in that order, columns renumbered through ``lut`` (global -> local id).
    Entry order inside a row is preserved (the canonical order is part of the bit-exact contract)."""
    rp = rowptr.to(torch.int64)
    start, cnt = rp[own], rp[own + 1] - rp[own]
    local_rp = torch.zeros(own.numel() + 1, dtype=torch.int64, device=rowptr.device)
    local_rp[1:] = torch.cumsum(cnt, 0)
    nnz = int(local_rp[-1])
    pos = torch.arange(nnz, device=rowptr.device, dtype=torch.int64)
    row_of = torch.repeat_interleave(torch.arange(own.numel(), device=rowptr.device), cnt, output_size=nnz)
    src = pos - local_rp[row_of] + start[row_of]
    lc = lut[col[src].to(torch.int64)]
    if nnz and int(lc.min()) < 0:
        raise RuntimeError("slice_csr: a column of an owned row is neither owned nor in the halo")
    return local_rp.to(torch.int32), lc.to(torch.int32), val[src].contiguous()


def local_lut(shard: RegionShard, device) -> torch.Tensor:
    lut = torch.full((shard.N,), -1, dtype=torch.int64)
    perm = torch.from_numpy(shard.perm)
    lut[perm] = torch.arange(perm.numel(), dtype=torch.int64)
    return lut.to(device)


def build_local_plan(shard: RegionShard, device: torch.device, edge_index: torch.Tensor,
                     edge_weight: Optional[torch.Tensor], reg_edge_index: Sequence[torch.Tensor],
                     reg_edge_weight: Sequence[Optional[torch.Tensor]]) -> GraphPlanTensors:
    """K1 on the full graph (global degrees), sliced to the owned rows; Chebyshev plan of the owned
    regional lists (the lists of other ranks are passed EMPTY so that region ids -- and with them
    the per-region weight blocks -- stay global)."""
    gplan = GraphPlanTensors(device, shard.N)
    build_gcn(gplan, edge_index, edge_weight)
    lut = local_lut(shard, device)
    own = torch.from_numpy(shard.own).to(device)
    rp, col, val = slice_csr(gplan.t["g_rowptr"], gplan.t["g_col"], gplan.t["g_val"], own, lut)
    plan = GraphPlanTensors(device, shard.n_own)
    plan.n_halo = shard.n_halo
    plan.nnz_gcn = int(col.numel())
    plan.t.update(g_rowptr=rp, g_col=col, g_val=val)
    eis, eas = [], []
    for r, (ei, ea) in enumerate(zip(reg_edge_index, reg_edge_weight)):
        if shard.region_owner[r] == shard.rank:
            le = lut[ei.to(device=device, dtype=torch.int64)]
            if le.numel() and (int(le.min()) < 0 or int(le.max()) >= shard.n_own):
                raise RuntimeError(f"regional list {r} has an endpoint outside its own region")
            eis.append(le)
            eas.append(ea)
        else:
            eis.append(torch.zeros(2, 0, dtype=torch.int64, device=device))
            eas.append(None if ea is None else torch.zeros(0, dtype=torch.float32, device=device))
    build_cheb(plan, eis, eas)
    return plan


# ------------------------------------------------------------------------------------------
# K4 row gather / scatter through the C-ABI (CUDA) -- index_select / index_copy on CPU tensors
# ------------------------------------------------------------------------------------------
def gather_rows(src: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    """dst[b, i] = src[b, idx[i]] for src [B, n_src, ...]."""
    if not src.is_cuda:
        return src.index_select(1, idx)
    src = src.contiguous()
    B, n_src = src.shape[0], src.shape[1]
    width = src[0, 0].numel()
    dst = torch.empty((B, idx.numel()) + tuple(src.shape[2:]), device=src.device, dtype=src.dtype)
    rc = _lib.load().regt_gather_rows(src.data_ptr(), idx.data_ptr(), dst.data_ptr(), B, n_src, idx.numel(), width,
                                      torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "regt_gather_rows")
    return dst


def scatter_rows(src: torch.Tensor, idx: torch.Tensor, dst: torch.Tensor) -> torch.Tensor:
    """dst[b, idx[i]] = src[b, i] for src [B, n_idx, ...], dst [B, n_dst, ...] (in place)."""
    if not src.is_cuda:
        dst.index_copy_(1, idx, src)
        return dst
    src = src.contiguous()
    assert dst.is_contiguous()
    width = src[0, 0].numel()
    rc = _lib.load().regt_scatter_rows(src.data_ptr(), idx.data_ptr(), dst.data_ptr(), src.shape[0], idx.numel(),
                                       dst.shape[1], width, torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "regt_scatter_rows")
    return dst


# ------------------------------------------------------------------------------------------
# the exchange step (torch.distributed: NCCL over NVLink on GPUs, gloo in the CPU tests)
# ------------------------------------------------------------------------------------------
def _flat_layout(params: Sequence[torch.nn.Parameter]):
    offs, tot = [], 0
    for p in params:
        offs.append(tot)
        tot += (p.numel() + 3) // 4 * 4
    return offs, tot + 4      # last 4: loss slot


def flatten_grads(params: Sequence[torch.nn.Parameter], flat: Optional[torch.Tensor] = None) -> torch.Tensor:
    """one flat buffer (fp32 in the product; the CPU tests use fp64 oracle modules) behind every ``.grad`` so that ONE all-reduce covers all shared weights."""
    offs, tot = _flat_layout(params)
    if flat is None:
        flat = torch.zeros(tot, device=params[0].device, dtype=params[0].dtype)
    for p, o in zip(params, offs):
        p.grad = flat[o:o + p.numel()].view_as(p)
    return flat


PEER_PUSH_MAX_FLOATS = 1 << 18     # csrc/peer.cu PEER_LL_MAX


class _DeviceSpan:
    """zero-copy torch view of device memory owned by libregt_b200 (``__cuda_array_interface__``)."""

    def __init__(self, ptr: int, n_floats: int):
        self.__cuda_array_interface__ = {"shape": (n_floats,), "typestr": "<f4", "data": (ptr, False), "version": 2}


class PeerRegion:
    """one rank's NVLink communication region (include/regt_b200.h, csrc/peer.cu): ``[flags | data | scratch]`` in one
    cudaMalloc block, mapped into every other rank of the node through CUDA IPC.  ``data`` is exposed as a torch
    tensor (the flat gradient buffer); ``allreduce()`` is ONE kernel launch on the current stream."""

    def __init__(self, n_floats: int, device: torch.device, rank: int, world: int, group=None):
        import ctypes as C
        import torch.distributed as dist
        from . import _lib
        self.lib, self.rank, self.world, self.n = _lib.load(), rank, world, n_floats
        lib = self.lib
        torch.cuda.set_device(device)
        self.base = C.c_void_p()
        _lib.check(lib.regt_comm_alloc(lib.regt_comm_region_bytes(n_floats), C.byref(self.base)), "regt_comm_alloc")
        handle = (C.c_ubyte * 64)()
        _lib.check(lib.regt_comm_export(self.base, handle), "regt_comm_export")
        mine = torch.tensor(list(handle), dtype=torch.uint8, device=device)
        every = torch.empty(world * 64, dtype=torch.uint8, device=device)
        dist.all_gather_into_tensor(every, mine, group=group)
        every = every.cpu().view(world, 64)
        self.peers = []
        regions = []
        for r in range(world):
            if r == rank:
                regions.append(self.base.value)
                continue
            h = (C.c_ubyte * 64)(*every[r].tolist())
            ptr = C.c_void_p()
            _lib.check(lib.regt_comm_import(h, C.byref(ptr)), "regt_comm_import")
            self.peers.append(ptr)
            regions.append(ptr.value)
        self.regions = (C.c_void_p * world)(*regions)
        self.data = torch.as_tensor(_DeviceSpan(self.base.value + lib.regt_comm_data_offset(), n_floats), device=device)
        dist.barrier(group=group)      # every rank has mapped every region before the first all-reduce

    def allreduce(self, last_in: Optional[torch.Tensor] = None, last_out: Optional[torch.Tensor] = None) -> None:
        """in-place sum over the ranks of ``data``.  Push path only (``n <= regt_peer_push_max_floats()``): ``last_in`` (one
        float) is added to this rank's loss slot ``data[-4]`` first; ``last_out`` receives the reduced slot, which is cleared."""
        from . import _lib
        _lib.check(self.lib.regt_peer_allreduce_f32(self.regions, self.rank, self.world, self.n,
                                                    None if last_in is None else last_in.data_ptr(),
                                                    None if last_out is None else last_out.data_ptr(),
                                                    torch.cuda.current_stream().cuda_stream), "regt_peer_allreduce_f32")

    @property
    def push(self) -> bool:
        return self.n <= int(self.lib.regt_peer_push_max_floats()) and os.environ.get("REGT_PEER_PULL", "0") != "1"

    def error(self) -> int:
        """non-zero once a kernel of this region gave up waiting for a peer (a rank stalled past the spin limit): the sums
        of that call are not trustworthy.  Reading the flag synchronises with the device."""
        return int(self.lib.regt_comm_error(self.base))

    def close(self) -> None:
        """unmap the peers' regions and free this rank's (call after the last all-reduce has completed on every rank)."""
        if getattr(self, "base", None) is None:
            return
        try:
            torch.cuda.synchronize()
            for ptr in self.peers:
                self.lib.regt_comm_unimport(ptr)
            self.lib.regt_comm_free(self.base)
        finally:
            self.peers, self.base, self.data = [], None, None



class GradExchange:
    """the per-step exchange of a sharded job: every ``.grad`` of ``params`` is a view into ONE flat
    fp32 buffer (so the wgrad kernels write straight into the communication buffer), whose last
    slots carry the loss; ``sync()`` is one sum all-reduce of that buffer.

    ``transport``: ``"peer"`` = the one-kernel all-reduce over NVLink peer memory (csrc/peer.cu; the buffer then lives in
    a CUDA-IPC region), ``"nccl"`` = ``torch.distributed.all_reduce``; ``None`` picks ``"peer"`` on CUDA with world > 1
    when every rank can map every region (env ``REGT_EXCHANGE=nccl`` forces NCCL), otherwise the process group's backend
    (gloo in the CPU tests)."""

    def __init__(self, params: Sequence[torch.nn.Parameter], world: int, group=None, transport: Optional[str] = None,
                 rank: Optional[int] = None):
        self.params, self.world, self.group = list(params), world, group
        self.region = None
        dev = self.params[0].device
        # transport None: the peer-memory kernels (8 GPUs: 9.4 us vs NCCL 32.7 us for 37 k floats through the push path,
        # 84.5 us vs 103.9 us for 4.4 M floats through the two-stage push); env REGT_EXCHANGE=nccl forces NCCL
        _, tot = _flat_layout(self.params)
        env = os.environ.get("REGT_EXCHANGE", "auto")
        want_peer = transport == "peer" or (transport is None and env in ("peer", "auto"))
        import torch.distributed as dist
        if world > 1 and dev.type == "cuda" and self.params[0].dtype == torch.float32 and want_peer and dist.is_available() \
                and dist.is_initialized():
            rank = dist.get_rank(group) if rank is None else rank
            ok = torch.ones(1, device=dev)
            try:
                self.region = PeerRegion(tot, dev, rank, world, group)
            except Exception as e:  # noqa: BLE001  (no P2P / IPC between these devices: every rank falls back together)
                print(f"[rank {rank}] peer-memory exchange unavailable ({e}); using the process group's all_reduce", file=sys.stderr)
                ok.zero_()
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
            if not bool(ok.item()):
                self.region = None
        self.transport = "peer" if self.region is not None else ("nccl" if dev.type == "cuda" else "gloo")
        self.flat = flatten_grads(self.params, None if self.region is None else self.region.data)
        self._offs, _ = _flat_layout(self.params)
        self._syncs = 0
        self.check_every = int(os.environ.get("REGT_EXCHANGE_CHECK_EVERY", "64"))
        for p in self.params:            # module_base._fused_step re-attaches a detached .grad through this
            p._regt_grad_owner = self

    def attach(self, p: torch.nn.Parameter) -> None:
        """``optimizer.zero_grad()`` (set_to_none, run.py:195) drops ``p.grad``: bind it to its slice of the flat buffer
        again (zeroed), so the next backward writes into the exchange buffer and not into a stray tensor."""
        for q, o in zip(self.params, self._offs):
            if q is p:
                view = self.flat[o:o + p.numel()].view_as(p)
                view.zero_()
                p.grad = view
                return
        raise RuntimeError("regt_b200: parameter is not part of this exchange")

    def _assert_owned(self) -> None:
        lo = self.flat.data_ptr()
        hi = lo + self.flat.numel() * self.flat.element_size()
        for i, p in enumerate(self.params):
            g = p.grad
            # None is fine: nothing was accumulated since zero_grad(set_to_none=True); fused_step re-attaches before it writes
            if g is not None and not (lo <= g.data_ptr() < hi):
                raise RuntimeError(
                    f"regt_b200: the gradient of parameter #{i} {tuple(p.shape)} is not a view of the exchange buffer any more "
                    "(optimizer.zero_grad(set_to_none=True) or another flat optimizer rebound .grad): the all-reduce would sum a "
                    "stale buffer.  Use exchange.zero() / zero_grad(set_to_none=False), or FlatRMSprop(..., flat_grad=exchange.flat)")

    def check_peers(self) -> None:
        """raises if a peer-memory kernel of this exchange timed out waiting for another rank (device sync)."""
        if self.region is not None and self.region.error():
            raise RuntimeError("regt_b200: a peer all-reduce kernel gave up waiting for another rank (a rank stalled past the spin "
                               "limit); the gradients of that step are not the global sums")

    def add_loss(self, loss: torch.Tensor) -> None:
        self.flat[-4:-3].add_(loss.reshape(1).to(self.flat.dtype))

    def sync(self) -> torch.Tensor:
        """returns the global loss accumulated since the last sync and clears the slot."""
        self._assert_owned()
        self._syncs += 1
        if (self.region is not None and self.check_every > 0 and self._syncs % self.check_every == 0
                and not torch.cuda.is_current_stream_capturing()):
            self.check_peers()      # the error flag of the PREVIOUS calls (one device sync every check_every steps)
        if self.world > 1:
            if self.region is not None and self.region.push:
                loss = torch.empty(1, device=self.flat.device)     # the kernel hands back the reduced loss and clears its slot
                self.region.allreduce(None, loss)
                return loss
            if self.region is not None:
                self.region.allreduce()
            else:
                import torch.distributed as dist
                dist.all_reduce(self.flat, group=self.group)
        loss = self.flat[-4:-3].clone()
        self.flat[-4:].zero_()
        return loss

    def zero(self) -> None:
        self.flat.zero_()

    def close(self) -> None:
        """collective: every rank has finished its last all-reduce (barrier), then the peer mappings and the region go.
        Not done from ``__del__``: a peer may still be writing into a region whose owner is being garbage-collected."""
        if self.region is not None:
            import torch.distributed as dist
            self.check_peers()
            dist.barrier(group=self.group)
            for p in self.params:
                p.grad = None
            self.flat = None
            self.region.close()
            self.region = None


def all_gather_nodes(local: torch.Tensor, shard: RegionShard, group=None) -> torch.Tensor:
    """per-rank [B, n_own, W] -> full [B, N, W] in global node order on every rank.  Ranks own
    different node counts: pad to the largest, all-gather, scatter each rank's rows to its ids."""
    import torch.distributed as dist
    B, W = local.shape[0], local.shape[2]
    nmax = int(shard.counts.max())
    pad = torch.zeros(B, nmax, W, device=local.device, dtype=local.dtype)
    pad[:, :shard.n_own] = local
    buf = torch.empty(shard.world, B, nmax, W, device=local.device, dtype=local.dtype)
    dist.all_gather_into_tensor(buf.view(-1), pad.view(-1), group=group)
    full = torch.empty(B, shard.N, W, device=local.device, dtype=local.dtype)
    for r in range(shard.world):
        ids = torch.from_numpy(np.nonzero(shard.node_owner == r)[0].astype(np.int64)).to(local.device)
        scatter_rows(buf[r, :, :ids.numel()].contiguous(), ids, full)
    return full


class RegionShardedModel:
    """wraps a ``models.RegionalTemporalGCN`` for one rank of a region-sharded job.

    ``fused_step(x, y)`` takes the FULL ``x [B,N,F,T]`` / ``y [B,N,O]`` (every rank sees every
    snapshot; input data is replicated or loaded per rank), runs forward + loss + backward on the
    rank's rows, then all-reduces the flat gradient buffer and the loss.  After it returns,
    ``.grad`` of every parameter and the loss equal the single-GPU values (up to summation order)."""

    def __init__(self, model, edge_index: torch.Tensor, reg_edge_index: Sequence[torch.Tensor],
                 reg_edge_weight: Sequence[Optional[torch.Tensor]], rank: int, world: int, group=None):
        self.model, self.group = model, group
        dev = next(model.parameters()).device
        N = model.tgnn.num_nodes
        self.shard = make_shard(N, edge_index, reg_edge_index, rank, world)
        self.plan = build_local_plan(self.shard, dev, edge_index, None, reg_edge_index, reg_edge_weight)
        self.perm = torch.from_numpy(self.shard.perm).to(dev)
        self.own = torch.from_numpy(self.shard.own).to(dev)
        self.exchange = GradExchange([p for p in model.parameters() if p.requires_grad], world, group)
        self.flat = self.exchange.flat

    def local_inputs(self, x: torch.Tensor, y: Optional[torch.Tensor]):
        """K4 gather: owned + halo rows of x, owned rows of y."""
        return gather_rows(x, self.perm), (None if y is None else gather_rows(y, self.own))

    def fused_step(self, x: torch.Tensor, y: torch.Tensor, micro_batch: Optional[int] = None,
                   gather_outputs: bool = False, local_inputs=None, sync: bool = True):
        """forward + loss + backward on this rank's rows; gradients ACCUMULATE into the flat buffer
        behind ``.grad`` (run.py:190).  ``sync=True`` all-reduces that buffer in place right away, so
        it is for loops that zero the gradients every step; loops that accumulate over many
        snapshots and step once (the reference's epoch, run.py:190-195) pass ``sync=False`` and call
        ``sync_gradients()`` once before ``optimizer.step()`` -- the sum is linear, one all-reduce
        per optimizer step is enough.  The loss rides in a slot of the same buffer."""
        xl, yl = local_inputs if local_inputs is not None else self.local_inputs(x, y)
        loss, out, hid = self.model._fused_step(xl, yl, self.plan, micro_batch, loss_nodes=self.shard.N)
        self.exchange.add_loss(loss)
        if sync:
            loss = self.sync_gradients()
        if gather_outputs and self.shard.world > 1:
            both = all_gather_nodes(torch.cat([out, hid], dim=2), self.shard, self.group)
            out, hid = both[..., :out.shape[2]].contiguous(), both[..., out.shape[2]:].contiguous()
        return loss, out, hid

    def sync_gradients(self) -> torch.Tensor:
        """the exchange step: one sum all-reduce of every shared-weight gradient + the loss slot.
        Returns the (global) loss accumulated since the last call and clears the slot."""
        return self.exchange.sync()

    def zero_grad(self) -> None:
        self.exchange.zero()

    @torch.no_grad()
    def forward(self, x: torch.Tensor):
        """inference: full-N ``(out, out_hidden)`` on every rank (all-gather of the regional outputs)."""
        from . import engine
        xl, _ = self.local_inputs(x, None)
        out, hid = engine.model_apply(self.model._mode, self.model._prec(xl.shape[3]), self.plan, self.model._hidden,
                                      self.model.output_dim, xl, self.model._param_dict(), None, True)
        if self.shard.world > 1:
            both = all_gather_nodes(torch.cat([out, hid], dim=2), self.shard, self.group)
            out, hid = both[..., :out.shape[2]].contiguous(), both[..., out.shape[2]:].contiguous()
        return out, hid
