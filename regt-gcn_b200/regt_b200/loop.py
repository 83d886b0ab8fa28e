"""The callers on either side of the hot path, kept on the device (SURVEY 8f.1 / 8f.2; csrc/loop.cu):

* ``SlidingWindows``  -- ``load_dataset.py:451-457`` materialises every window of ``node_data [N, F, T_total]`` on the host and
  ``run.py:172`` ships one per step; here ``node_data`` stays resident and a batch of windows is gathered by one kernel.
* ``train_epoch``     -- ``run.py:163-199``: every snapshot's loss is back-propagated into the SAME gradients, ONE
  ``RMSprop`` step per epoch; no per-snapshot ``loss.cpu()`` (the losses stay on the device, one read at the end).
* ``evaluate``        -- ``predict.py:142-194``: MAE, RMSE, MAPE normalised by each snapshot's 95th percentile, reduced on the
  device (``regt_eval_metrics``), one small D2H read per batch instead of three tensors per snapshot.

Both take a ``null_value`` for series that mark a missing reading (METR-LA / PEMS-BAY: 0): the loss and the metrics then
run over the valid targets only.

Both take ``share_periods=True`` (opt-in): the cell output of a period depends on that period's input alone, so a pass over
C consecutive windows runs the cell once per time step (C + T - 1 steps instead of C * T periods) and combines the steps
into each window's out_hidden with the attention weights (``regt_combine_forward`` / ``regt_combine_backward``).  It is
exact in real arithmetic; floating-point sums run in another order, so the default keeps the windowed path.
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

    def _gather_into(self, starts: torch.Tensor, t_in: int, t_out: int, x: torch.Tensor, y: Optional[torch.Tensor]) -> None:
        lib = _lib.load()
        with torch.cuda.device(self.data.device):
            _lib.check(lib.regt_window_gather(self.data.data_ptr(), starts.data_ptr(), starts.numel(), self.N, self.F, self.T_total,
                                              t_in, t_out, self.target, x.data_ptr(), None if y is None else y.data_ptr(),
                                              _stream()), "regt_window_gather")

    def gather_steps(self, t0: int, x: torch.Tensor) -> None:
        """x [S,N,F,1] <- the inputs of time steps t0 .. t0+S-1 (period t of window w is time step w + t)"""
        starts = torch.arange(t0, t0 + x.shape[0], device=self.data.device)
        self._gather_into(starts, 1, 0, x, None)

    def gather_targets(self, w0: int, y: torch.Tensor, scratch_x: torch.Tensor) -> None:
        """y [C,N,T_out] <- the targets of windows w0 .. w0+C-1 (scratch_x [>=C,N,F,1] receives their last input step)"""
        starts = torch.arange(w0 + self.t_in - 1, w0 + self.t_in - 1 + y.shape[0], device=self.data.device)
        self._gather_into(starts, 1, self.t_out, scratch_x, y)

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


# ---- time steps shared across the windows of a pass (share_periods=True) -------------------------------------------------

_COMBINE_MAX_T = 256   # periods the combine kernels take (csrc/combine.cu); a longer window runs the windowed epoch


def _shared_budget(have: int = 0) -> int:
    """bytes a pass may hold: 70 % of the free device memory plus the ``have`` bytes of buffers being replaced, which the
    caching allocator still holds (as auto_micro_batch)"""
    free, _ = torch.cuda.mem_get_info()
    return int(0.7 * (free + have))


class _SharedPlan:
    """what every pass of a shared-period epoch uses: the model's step configuration, the pass size, and the buffers,
    allocated once per shape and cached on the model (a shorter last pass takes views)"""

    def __init__(self, model, windows: SlidingWindows, graph_args: Sequence, batch: int, n_windows: int, train: bool = True):
        from .module_base import RegTModelBase
        if not isinstance(model, RegTModelBase) or not hasattr(model, "step_plan") or model._mode == _lib.MODE_TGCN:
            raise TypeError(f"regt_b200: share_periods needs a RegionalTemporalGCN or TemporalGCN trained by its own fused_step; "
                            f"{type(model).__name__} has no sliding windows with period attention to share (region shards: "
                            f"their halo rows follow the windowed path only)")
        from . import engine
        self.engine = engine
        T = self.T = windows.t_in
        self.prec = model._prec(T)
        if self.prec != _lib.PREC_FP32 and T > 64:
            name = {v: k for k, v in _lib.PRECISIONS.items()}[self.prec]
            raise RuntimeError(f"regt_b200: precision {name} supports up to 64 periods (got {T})")
        if windows.t_out != model.output_dim:
            raise ValueError(f"regt_b200: windows have {windows.t_out} targets, the model {model.output_dim} outputs")
        self.model, self.windows = model, windows
        self.mode, self.H, self.O, self.N, self.F = model._mode, model._hidden, model.output_dim, windows.N, windows.F
        dev = windows.data.device
        probe = torch.empty(1, self.N, self.F, 1, device=dev)
        self.plan = model.step_plan(probe, *graph_args)
        cache = getattr(model, "_shared_bufs", None)
        key = (self.N, self.F, T, self.H, self.O, self.prec, id(self.plan))
        want = max(1, min(batch, n_windows))
        # the step workspace of an evaluation holds no planes (inference = 1): a training epoch needs a larger one
        self.train = train
        if (cache is not None and cache["key"] == key and (cache["train"] or not train)
                and (cache["C"] >= want or cache["want"] == want)):
            self.C, self.bufs = min(want, cache["C"]), cache
            return
        have = 0 if cache is None else sum(t.numel() * t.element_size() for t in cache.values() if isinstance(t, torch.Tensor))
        model._shared_bufs = cache = None                     # release the old buffers before sizing the new ones
        C = want
        while C > 1 and self._bytes(C) > _shared_budget(have):
            C = (C + 1) // 2
        self.C = C
        self.bufs = model._shared_bufs = self._alloc(C, key)
        self.bufs["want"], self.bufs["train"] = want, train

    def _bytes(self, C: int) -> int:
        e, S = self.engine, C + self.T - 1
        N, H, O, F = self.N, self.H, self.O, self.F
        ws = e.workspace_bytes(self.mode, self.prec, self.plan, S, N, 1, H, O, F, inference=not self.train)
        hw = e.head_workspace_bytes(self.mode, self.prec, self.plan, C, self.T, H, O, F)
        return ws + hw + 4 * N * (2 * S * H + C * H + S * F + C * F + 3 * C * O)

    def _alloc(self, C: int, key) -> dict:
        e, S, dev = self.engine, C + self.T - 1, self.windows.data.device
        N, H, O, F = self.N, self.H, self.O, self.F
        lib = _lib.load()
        f32 = dict(device=dev, dtype=torch.float32)
        return {"key": key, "C": C,
                "step_ws": torch.empty(e.workspace_bytes(self.mode, self.prec, self.plan, S, N, 1, H, O, F, inference=not self.train),
                                       device=dev, dtype=torch.uint8),
                "head_ws": torch.empty(e.head_workspace_bytes(self.mode, self.prec, self.plan, C, self.T, H, O, F), device=dev,
                                       dtype=torch.uint8),
                "xs": torch.empty(S, N, F, 1, **f32), "xw": torch.empty(C, N, F, 1, **f32), "y": torch.empty(C, N, O, **f32),
                "Hs": torch.empty(S, N, H, **f32), "Gs": torch.empty(S, N, H, **f32), "hid": torch.empty(C, N, H, **f32),
                "out": torch.empty(C, N, O, **f32), "d_out": torch.empty(C, N, O, **f32), "loss": torch.empty(2, **f32),
                "y1": torch.empty(1, N, O, **f32), "out1": torch.empty(1, N, O, **f32), "d_out1": torch.empty(1, N, O, **f32),
                "att0": torch.zeros(1, **f32),
                "scratch": torch.empty(lib.regt_combine_scratch_bytes(self.T), device=dev, dtype=torch.uint8)}

    def run_pass(self, w0: int, w1: int, train: bool, loss_kind: int = _lib.LOSS_MSE, null_value: Optional[float] = None,
                 last_alone: bool = False):
        """windows [w0, w1) (w1 - w0 <= self.C): the cell once per time step, the combine, the head over the windows and, when
        training (a plan built with train=True), the backward into .grad.  Returns (out [C,N,O], y [C,N,O], sum of the losses, loss of window w1 - 1 or
        None); the tensors are views of the cached buffers."""
        e, b, lib = self.engine, self.bufs, _lib.load()
        C, T = w1 - w0, self.T
        S, width = C + T - 1, self.N * self.H
        xs, Hs, Gs, hid = b["xs"][:S], b["Hs"][:S], b["Gs"][:S], b["hid"][:C]
        y, out, d_out = b["y"][:C], b["out"][:C], b["d_out"][:C]
        self.windows.gather_steps(w0, xs)
        self.windows.gather_targets(w0, y, b["xw"])
        params = self.model._param_dict()
        step_params = dict(params, attention=b["att0"])      # one period per step: softmax([0]) = 1, out_hidden = H'
        st = e.build_state(self.mode, self.prec, self.plan, xs, self.H, self.O, step_params, None, None, head=False,
                           workspace=b["step_ws"], inference=not train, out_hidden=Hs)
        e.run_forward(st, head=False)
        att = params["attention"]
        with torch.cuda.device(hid.device):
            _lib.check(lib.regt_combine_forward(att.data_ptr(), Hs.data_ptr(), S, C, T, width, hid.data_ptr(), _stream()),
                       "regt_combine_forward")
        hs = e.build_head_state(self.mode, self.prec, self.plan, hid, T, self.O, params, out, b["head_ws"], y if train else None,
                                b["loss"][:1], d_out, train=train, loss_kind=loss_kind, null_value=null_value)
        if not train:
            e.run_head(hs)
            return out, y, None, None
        grads = self.model._grad_views(params)
        e.run_head(hs, grads)
        with torch.cuda.device(hid.device):
            g_att = grads["attention"]
            _lib.check(lib.regt_combine_backward(att.data_ptr(), Hs.data_ptr(), b["head_ws"].data_ptr(), S, C, T, width, Gs.data_ptr(),
                                                 g_att.data_ptr(), b["scratch"].data_ptr(), b["scratch"].numel(), _stream()),
                       "regt_combine_backward")
        total = b["loss"][:1].clone()
        last_loss = None
        if last_alone:   # the final window's own loss (what run.py:197 returns), from the same out_hidden
            y1 = b["y1"]
            self.windows.gather_targets(w1 - 1, y1, b["xw"])
            ls = e.build_head_state(self.mode, self.prec, self.plan, hid[C - 1:], T, self.O, params, b["out1"], b["head_ws"], y1,
                                    b["loss"][1:], b["d_out1"], train=False, loss_kind=loss_kind, null_value=null_value)
            e.run_head(ls)
            last_loss = b["loss"][1:].clone()
        step_grads = {k: (None if k == "attention" else g) for k, g in grads.items() if k not in e.HEAD_KEYS}
        e.run_backward(st, step_grads, None, Gs, True, head=False)
        return out, y, total, last_loss


def _train_epoch_shared(model, windows, graph_args, optimizer, first, last, batch, loss, null_value):
    from . import engine
    loss_kind = engine.check_loss(loss, null_value)
    sp = _SharedPlan(model, windows, graph_args, batch, last - first)
    optimizer.zero_grad()
    total = torch.zeros(1, device=windows.data.device)
    last_loss = None
    for w0 in range(first, last, sp.C):
        w1 = min(last, w0 + sp.C)
        _, _, part, ll = sp.run_pass(w0, w1, True, loss_kind, null_value, last_alone=w1 == last)
        total += part
        if ll is not None:
            last_loss = ll
    optimizer.step()
    return last_loss, total


def train_epoch(model, windows: SlidingWindows, graph_args: Sequence, optimizer, first: int = 0, last: Optional[int] = None,
                batch: int = 64, micro_batch: Optional[int] = None, loss: str = "mse", null_value: Optional[float] = None,
                share_periods: bool = False):
    """one epoch of run.py:163-199 over windows [first, last): gradients of every snapshot accumulate, ONE optimizer step.
    Returns (last snapshot's loss -- what run.py:197 returns --, sum of the snapshot losses); both are device tensors.
    ``loss`` / ``null_value``: the loss of ``model.fused_step``.
    ``share_periods``: run the cell once per time step of a pass of ``batch`` windows and share it across the windows
    (module docstring); a pass shrinks when its buffers do not fit the free device memory, ``micro_batch`` does not apply.
    Windows of more than 256 periods (precision fp32 only) run the windowed epoch: the combine kernels keep up to 256
    periods per column on chip."""
    last = len(windows) if last is None else last
    if share_periods and windows.t_in <= _COMBINE_MAX_T:
        return _train_epoch_shared(model, windows, graph_args, optimizer, first, last, batch, loss, null_value)
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
             q: float = 95.0, null_value: Optional[float] = None, share_periods: bool = False):
    """predict.py:142-194 -> (MAE, RMSE, MAPE %) over windows [first, last).  ``null_value`` (a float): targets equal to it,
    or NaN, are missing and left out of every metric and of the percentile (``regt_eval_metrics_masked``).
    ``share_periods``: the forward of ``train_epoch(share_periods=True)``, one cell evaluation per time step of a pass
    (windows of more than 256 periods run windowed, as there)."""
    lib = _lib.load()
    last = len(windows) if last is None else last
    dev = windows.data.device
    sums = []
    n = 0
    share_periods = share_periods and windows.t_in <= _COMBINE_MAX_T
    sp = _SharedPlan(model, windows, graph_args, batch, last - first, train=False) if share_periods else None
    step = sp.C if share_periods else batch
    for s0 in range(first, last, step):
        s1 = min(last, s0 + step)
        if share_periods:
            out, y, _, _ = sp.run_pass(s0, s1, False)
        else:
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
