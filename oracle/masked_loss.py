"""TEST INFRASTRUCTURE: the masked losses of a batch, for data that marks a missing reading with a null value or NaN
(METR-LA / PEMS-BAY style inputs), restated in torch so that the same code is the fp64 oracle, its fp32 twin and, on
``model(x)``'s output, the autograd path's loss.

  loss = sum_b [c_b > 0] * sum_{n,o} m * l(out - y) / c_b        c_b = sum_{n,o} m      (run.py:180 over valid targets)
  l = (out - y)^2 (``"mse"``) or |out - y| (``"mae"``); m = 0 where y == null_value or y is NaN, 1 elsewhere;
  null_value None: m = 1 everywhere (a NaN in y propagates); null_value NaN: only NaNs are missing.
A snapshot without a valid target adds 0 and no gradient.  torch.where passes no gradient (and no NaN) to the masked
entries, and |.|'s backward gives sign(0) = 0 at ties."""
import math
from typing import Optional

import torch


def valid_mask(y: torch.Tensor, null_value: Optional[float]) -> torch.Tensor:
    if null_value is None:
        return torch.ones_like(y, dtype=torch.bool)
    m = ~torch.isnan(y)
    if not math.isnan(null_value):
        m &= y != null_value
    return m


def masked_loss(out: torch.Tensor, y: torch.Tensor, loss: str = "mse", null_value: Optional[float] = None) -> torch.Tensor:
    """out, y [B,N,O] (or [N,O], one snapshot) -> the summed per-snapshot masked mean (a 0-d tensor, differentiable)."""
    if out.dim() == 2:
        out, y = out.unsqueeze(0), y.unsqueeze(0)
    m = valid_mask(y, null_value)
    d = torch.where(m, out - y, torch.zeros_like(out)) if null_value is not None else out - y
    ell = d * d if loss == "mse" else d.abs()
    c = m.sum(dim=(1, 2)).to(out.dtype)
    per = ell.sum(dim=(1, 2)) / c.clamp(min=1)
    return per.sum()


def masked_batched_step(model, x: torch.Tensor, y: torch.Tensor, graph_args: tuple, loss: str = "mse",
                        null_value: Optional[float] = None):
    """regt_oracle.batched_step with the masked loss: x [B,N,F,T], y [B,N,O] -> (out, out_hidden, loss_sum); the
    parameters' .grad hold the summed gradient (one backward per snapshot, run.py:190)."""
    outs, hids, total = [], [], 0.0
    for b in range(x.size(0)):
        out, hid = model(x[b], *graph_args)
        outs.append(out.detach())
        hids.append(hid.detach())
        lb = masked_loss(out, y[b], loss, null_value)
        if lb.requires_grad:
            lb.backward()
        total += float(lb.detach())
    return torch.stack(outs), torch.stack(hids), total
