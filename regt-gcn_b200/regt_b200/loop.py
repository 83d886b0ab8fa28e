"""The callers on either side of the hot path, kept on the device (SURVEY 8f.1 / 8f.2; csrc/loop.cu):

* ``SlidingWindows``  -- ``load_dataset.py:451-457`` materialises every window of ``node_data [N, F, T_total]`` on the host and
  ``run.py:172`` ships one per step; here ``node_data`` stays resident and a batch of windows is gathered by one kernel.
* ``train_epoch``     -- ``run.py:163-199``: every snapshot's loss is back-propagated into the SAME gradients, ONE
  ``RMSprop`` step per epoch; no per-snapshot ``loss.cpu()`` (the losses stay on the device, one read at the end).
* ``evaluate``        -- ``predict.py:142-194``: MAE, RMSE, MAPE normalised by each snapshot's 95th percentile, reduced on the
  device (``regt_eval_metrics``), one small D2H read per batch instead of three tensors per snapshot.

Both take a ``null_value`` for series that mark a missing reading (METR-LA / PEMS-BAY: 0): the loss and the metrics then
run over the valid targets only.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional, Sequence, Tuple

import torch

from . import _lib


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


class SlidingWindows:
    """device-resident ``node_data [N, F, T_total]`` (fp32); window ``i`` = features ``node_data[:, :, i:i+T_in]`` and targets
    ``node_data[:, target_feature, i+T_in:i+T_in+T_out]`` (``load_dataset.py:451-457``: the LAST feature is the target)."""

    def __init__(self, node_data: torch.Tensor, t_in: int, t_out: int, target_feature: int = -1):
        if node_data.dim() != 3 or node_data.dtype != torch.float32 or not node_data.is_cuda:
            raise ValueError("regt_b200: node_data must be a CUDA float32 tensor [N, F, T_total]")
        self.data = node_data.contiguous()
        self.N, self.F, self.T_total = self.data.shape
        self.t_in, self.t_out = int(t_in), int(t_out)
        self.target = target_feature % self.F
        self.count = self.T_total - (self.t_in + self.t_out) + 1
        if self.count <= 0:
            raise ValueError("regt_b200: series shorter than one window")

    def __len__(self) -> int:
        return self.count

    def gather(self, starts: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """starts: int64 CUDA tensor [B] of window indices -> (x [B,N,F,T_in], y [B,N,T_out])"""
        lib = _lib.load()
        starts = starts.to(device=self.data.device, dtype=torch.int64).contiguous()
        B = starts.numel()
        x = torch.empty(B, self.N, self.F, self.t_in, device=self.data.device)
        y = torch.empty(B, self.N, self.t_out, device=self.data.device)
        with torch.cuda.device(self.data.device):
            _lib.check(lib.regt_window_gather(self.data.data_ptr(), starts.data_ptr(), B, self.N, self.F, self.T_total, self.t_in,
                                              self.t_out, self.target, x.data_ptr(), y.data_ptr(), _stream()), "regt_window_gather")
        return x, y


class FlatRMSprop:
    """``torch.optim.RMSprop(params, lr, alpha=0.99, eps=1e-8, weight_decay)`` (run.py:145) over ONE flat buffer: parameters and
    gradients become views of two flat fp32 tensors, the step is a single kernel launch.

    ``skip``: parameters that never receive a gradient (the reference's dead ``_weight_att*`` / ``_bias_att*`` / A3TGCN
    ``linear``; ``model.dead_parameters()``).  ``torch.optim.RMSprop`` leaves a parameter whose ``.grad`` is None untouched --
    weight decay included -- so these are laid out BEHIND the stepped range and never move.
    ``exchange``: a ``shard.GradExchange`` whose flat buffer already backs every ``.grad`` (multi-GPU): the optimizer then
    steps out of that buffer instead of rebinding ``.grad`` to a buffer of its own (which would detach the all-reduce)."""

    def __init__(self, params: Sequence[torch.nn.Parameter], lr: float = 1e-3, alpha: float = 0.99, eps: float = 1e-8,
                 weight_decay: float = 0.0, skip: Sequence[torch.nn.Parameter] = (), exchange=None):
        skip_ids = {id(p) for p in skip}
        params = [p for p in params if p.requires_grad]
        self.exchange = exchange
        if exchange is not None:
            if [id(p) for p in exchange.params] != [id(p) for p in params]:
                raise ValueError("regt_b200: FlatRMSprop(exchange=...) needs the exchange's parameter list, in its order")
            self.params = params           # layout dictated by the exchange buffer; skipped ranges are masked by segments
        else:
            self.params = [p for p in params if id(p) not in skip_ids] + [p for p in params if id(p) in skip_ids]
        self.lr, self.alpha, self.eps, self.wd = lr, alpha, eps, weight_decay
        dev = self.params[0].device
        offs, tot = [], 0
        for p in self.params:
            offs.append(tot)
            tot += (p.numel() + 3) // 4 * 4
        self._offs = offs
        self.flat_p = torch.zeros(tot, device=dev)
        self.square_avg = torch.zeros(tot, device=dev)
        if exchange is not None:
            self.flat_g = exchange.flat[:tot]
        else:
            self.flat_g = torch.zeros(tot, device=dev)
        # contiguous runs [lo, hi) of stepped (live) elements
        self.segments = []
        for p, o in zip(self.params, offs):
            if id(p) in skip_ids:
                continue
            hi = o + (p.numel() + 3) // 4 * 4
            if self.segments and self.segments[-1][1] == o:
                self.segments[-1][1] = hi
            else:
                self.segments.append([o, hi])
        with torch.no_grad():
            for p, o in zip(self.params, offs):
                self.flat_p[o:o + p.numel()].copy_(p.reshape(-1))
                p.data = self.flat_p[o:o + p.numel()].view_as(p)
                if exchange is None:
                    p.grad = self.flat_g[o:o + p.numel()].view_as(p)
                    p._regt_grad_owner = self

    def attach(self, p: torch.nn.Parameter) -> None:
        """re-bind a ``.grad`` dropped by ``zero_grad(set_to_none=True)`` to its (zeroed) slice of the flat buffer."""
        for q, o in zip(self.params, self._offs):
            if q is p:
                view = self.flat_g[o:o + p.numel()].view_as(p)
                view.zero_()
                p.grad = view
                return
        raise RuntimeError("regt_b200: parameter is not owned by this optimizer")

    def zero_grad(self) -> None:
        if self.exchange is not None:
            self.exchange.zero()
        else:
            self.flat_g.zero_()

    def step(self) -> None:
        lib = _lib.load()
        lo_g, hi_g = self.flat_g.data_ptr(), self.flat_g.data_ptr() + self.flat_g.numel() * 4
        for p in self.params:
            if p.grad is not None and not (lo_g <= p.grad.data_ptr() < hi_g):
                raise RuntimeError("regt_b200: a parameter's .grad is no longer a view of the optimizer's flat gradient buffer "
                                   "(something rebound it): the step would use stale gradients")
        with torch.cuda.device(self.flat_p.device):
            for lo, hi in self.segments:
                _lib.check(lib.regt_rmsprop_step(self.flat_p.data_ptr() + 4 * lo, self.flat_g.data_ptr() + 4 * lo,
                                                 self.square_avg.data_ptr() + 4 * lo, hi - lo,
                                                 self.lr, self.alpha, self.eps, self.wd, _stream()), "regt_rmsprop_step")


def train_epoch(model, windows: SlidingWindows, graph_args: Sequence, optimizer, first: int = 0, last: Optional[int] = None,
                batch: int = 64, micro_batch: Optional[int] = None, loss: str = "mse", null_value: Optional[float] = None):
    """one epoch of run.py:163-199 over windows [first, last): gradients of every snapshot accumulate, ONE optimizer step.
    Returns (last snapshot's loss -- what run.py:197 returns --, sum of the snapshot losses); both are device tensors.
    ``loss`` / ``null_value``: the loss of ``model.fused_step``."""
    last = len(windows) if last is None else last
    optimizer.zero_grad()
    total = torch.zeros(1, device=windows.data.device)
    last_loss = None
    for s0 in range(first, last, batch):
        s1 = min(last, s0 + batch)
        # fused_step returns the SUM of its snapshots' losses; the final snapshot of the epoch runs alone because its loss is
        # what run.py:197 returns
        tail = 1 if s1 == last else 0
        if s1 - tail > s0:
            x, y = windows.gather(torch.arange(s0, s1 - tail, device=windows.data.device))
            total += model.fused_step(x, y, *graph_args, micro_batch=micro_batch, loss=loss, null_value=null_value)[0]
        if tail:
            x, y = windows.gather(torch.arange(s1 - 1, s1, device=windows.data.device))
            last_loss = model.fused_step(x, y, *graph_args, loss=loss, null_value=null_value)[0]
            total += last_loss
    optimizer.step()
    return last_loss, total


@torch.no_grad()
def evaluate(model, windows: SlidingWindows, graph_args: Sequence, first: int = 0, last: Optional[int] = None, batch: int = 64,
             q: float = 95.0, null_value: Optional[float] = None):
    """predict.py:142-194 -> (MAE, RMSE, MAPE %) over windows [first, last).  ``null_value`` (a float): targets equal to it,
    or NaN, are missing and left out of every metric and of the percentile (``regt_eval_metrics_masked``)."""
    lib = _lib.load()
    last = len(windows) if last is None else last
    dev = windows.data.device
    sums = []
    n = 0
    for s0 in range(first, last, batch):
        s1 = min(last, s0 + batch)
        x, y = windows.gather(torch.arange(s0, s1, device=dev))
        out = model(x, *graph_args)[0].contiguous()
        n = out[0].numel()
        part = torch.empty(s1 - s0, 4 if null_value is None else 5, device=dev, dtype=torch.float64)
        with torch.cuda.device(dev):
            if null_value is None:
                _lib.check(lib.regt_eval_metrics(out.data_ptr(), y.contiguous().data_ptr(), s1 - s0, n, q, part.data_ptr(),
                                                 _stream()), "regt_eval_metrics")
            else:
                _lib.check(lib.regt_eval_metrics_masked(out.data_ptr(), y.contiguous().data_ptr(), s1 - s0, n, q, float(null_value),
                                                        part.data_ptr(), _stream()), "regt_eval_metrics_masked")
        sums.append(part)
    return reduce_metrics(torch.cat(sums).cpu(), n)


def reduce_metrics(sums: torch.Tensor, n: int):
    """per-snapshot [sum|e|, sum e^2, p95, sum|e|/p95] -> predict.py's return values: snapshots whose normalised errors
    contain an inf (p95 == 0) are left out of the MAPE only (predict.py:167-169).  Masked sums [count, sum|e|, sum e^2, p95,
    sum|e|/p95] (5 columns) are divided by the valid counts; snapshots without a valid target drop out."""
    if sums.shape[1] == 5:
        sums = sums[sums[:, 0] > 0]
        cnt = float(sums[:, 0].sum())
        if cnt == 0:
            return float("nan"), float("nan"), float("nan")
        keep = ~torch.isinf(sums[:, 4])
        mape = float(sums[keep, 4].sum()) / float(sums[keep, 0].sum()) * 100 if bool(keep.any()) else float("nan")
        return float(sums[:, 1].sum()) / cnt, math.sqrt(float(sums[:, 2].sum()) / cnt), mape
    S = sums.shape[0]
    mae = float(sums[:, 0].sum()) / (S * n)
    rmse = math.sqrt(float(sums[:, 1].sum()) / (S * n))
    keep = ~torch.isinf(sums[:, 3])
    mape = float(sums[keep, 3].sum()) / (int(keep.sum()) * n) * 100 if bool(keep.any()) else float("nan")
    return mae, rmse, mape
