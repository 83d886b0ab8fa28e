"""nn.Module plumbing shared by the drop-in classes in ``models/``: parameter holders with the
reference's state_dict key names, the graph-plan lookup, and the fused training step."""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence

import torch
import torch.nn as nn

from . import _lib, engine
from .plan import get_plan


def check_node_features(F: int) -> None:
    """constructor check: the kernels work at ``engine.F_IN`` features per node and take any narrower input."""
    if not 1 <= F <= engine.F_IN:
        raise ValueError(f"node_features must be an int in 1..{engine.F_IN} (the kernels' feature width is "
                         f"{engine.F_IN}), got {F!r}")


def _glorot(rows: int, cols: int) -> nn.Parameter:
    a = math.sqrt(6.0 / (rows + cols))
    return nn.Parameter(torch.empty(rows, cols).uniform_(-a, a))


class _LinWeight(nn.Module):
    """holder for PyG ``Linear(bias=False)``: state_dict key ``<name>.weight`` [out,in]."""

    def __init__(self, cin: int, cout: int):
        super().__init__()
        self.weight = _glorot(cout, cin)


class GCNConvParams(nn.Module):
    """parameters of a PyG GCNConv (``lin.weight`` [H,F] glorot, ``bias`` [H] zeros); the
    arithmetic runs in the fused kernels, so this module has no forward."""

    def __init__(self, cin: int, cout: int):
        super().__init__()
        self.bias = nn.Parameter(torch.zeros(cout))
        self.lin = _LinWeight(cin, cout)


class ChebConvParams(nn.Module):
    """parameters of a PyG ChebConv(K=2): ``lins.{0,1}.weight`` [H,F], ``bias`` [H]."""

    def __init__(self, cin: int, cout: int, K: int = 2):
        super().__init__()
        if K != 2:
            raise NotImplementedError("only ChebConv K=2 is on the RegT-GCN hot path")
        self.bias = nn.Parameter(torch.zeros(cout))
        self.lins = nn.ModuleList([_LinWeight(cin, cout) for _ in range(K)])


def tgcn_param_dict(tgcn: nn.Module) -> Dict[str, torch.Tensor]:
    d = {}
    for g, name in enumerate("zrh"):
        conv, lin = getattr(tgcn, f"conv_{name}"), getattr(tgcn, f"linear_{name}")
        d[f"conv_w{g}"], d[f"conv_b{g}"] = conv.lin.weight, conv.bias
        d[f"lin_w{g}"], d[f"lin_b{g}"] = lin.weight, lin.bias
    return d


class RegTModelBase(nn.Module):
    """common forward / fused-step logic.  Subclasses define ``_mode``, ``_hidden``,
    ``output_dim``, ``precision`` and ``_param_dict()``."""

    _mode = _lib.MODE_A3TGCN

    def _param_dict(self) -> Dict[str, torch.Tensor]:
        raise NotImplementedError

    def _prec(self, T: Optional[int] = None) -> int:
        """``precision="auto"`` (the default): fp32-equivalent arithmetic on the fastest path that offers it -- the 3xTF32
        tensor-core kernels when the hidden width allows (hidden % 32 == 0; the reference's 256 does) and the input has at
        most 64 periods (``T``, the tf32x3 kernels' limit), else the FFMA kernels, which take any period count.
        Both meet the same 1e-5 parity bound; ``bf16`` (stated tolerance) is opt-in only.  An explicit precision is
        used as given: tf32x3 with T > 64 is refused by the kernels."""
        prec = self.precision
        if prec == "auto":
            fits = self._hidden % 32 == 0 and self._mode != _lib.MODE_TGCN and (T is None or T <= 64)
            prec = "tf32x3" if fits else "fp32"
        try:
            return _lib.PRECISIONS[prec]
        except KeyError:
            raise ValueError(f"precision must be 'auto' or one of {sorted(_lib.PRECISIONS)}, got {self.precision!r}")

    def dead_parameters(self):
        """parameters the reference never trains (``attention()`` is never called, models/RegionalTemporalGCN.py:91-111;
        ``A3TGCN.linear``, models/TemporalGCN.py:70): they exist for checkpoint compatibility and get no gradient, so an
        optimizer must leave them alone (``FlatRMSprop(skip=model.dead_parameters())``)."""
        dead = []
        for name, p in self.named_parameters():
            leaf = name.split(".")[-1]
            if leaf in ("_weight_att1", "_weight_att2", "_bias_att1", "_bias_att2"):
                dead.append(p)
            elif self._mode == _lib.MODE_A3TGCN and name.startswith("tgnn.linear."):
                dead.append(p)
        return dead

    @staticmethod
    def _as_batched(x: torch.Tensor):
        if x.dim() == 3:
            return x.unsqueeze(0), False
        if x.dim() == 4:
            return x, True
        raise ValueError(f"x must be [N,F,T] (reference) or [B,N,F,T] (batched), got {tuple(x.shape)}")

    def _run(self, x: torch.Tensor, plan):
        xb, batched = self._as_batched(x)
        xb = xb.to(torch.float32).contiguous()
        out, hid = engine.model_apply(self._mode, self._prec(xb.shape[3]), plan, self._hidden, self.output_dim, xb,
                                      self._param_dict(), None, True)
        if not batched:
            out, hid = out[0], hid[0]
        return out, hid

    # ---- fused training step: forward + loss + backward in one pass, no autograd graph ----
    def _fused_step(self, x: torch.Tensor, y: torch.Tensor, plan, micro_batch: Optional[int] = None,
                    loss_nodes: Optional[int] = None):
        """run.py:170-192 for a whole batch of snapshots: loss = sum_b mean((out_b-y_b)^2);
        gradients are ACCUMULATED into ``.grad`` (the reference accumulates over the epoch and
        steps once, run.py:190-195).  Returns (loss [1] device tensor, out, out_hidden)."""
        xb, batched = self._as_batched(x)
        yb = y if batched else y.unsqueeze(0)
        xb = xb.to(torch.float32).contiguous()
        yb = yb.to(torch.float32).contiguous()
        params = self._param_dict()
        grads = {}
        for k, p in params.items():
            if p.grad is None:
                owner = getattr(p, "_regt_grad_owner", None)   # a GradExchange / FlatRMSprop owns the flat buffer behind .grad
                if owner is not None:
                    owner.attach(p)
                else:
                    p.grad = torch.zeros_like(p)
            grads[k] = p.grad
        B = xb.shape[0]
        prec = self._prec(xb.shape[3])
        if micro_batch:
            mb = min(B, micro_batch)
        else:   # whole batch if its saved planes fit, else the largest divisor of B that does (decided once per shape)
            key = (B, xb.shape[1], xb.shape[3])
            if getattr(self, "_mb_key", None) != key:
                ws = getattr(self, "_ws", None)
                self._mb = engine.auto_micro_batch(self._mode, prec, plan, B, xb.shape[1], xb.shape[3], self._hidden,
                                                   self.output_dim, 0 if ws is None else ws.numel(), xb.shape[2])
                self._mb_key = key
            mb = self._mb
        loss = None
        outs, hids = [], []
        for b0 in range(0, B, mb):
            st = engine.build_state(self._mode, prec, plan, xb[b0:b0 + mb], self._hidden, self.output_dim,
                                    params, yb[b0:b0 + mb], None, True, getattr(self, "_ws", None), fuse_head=True,
                                    loss_nodes=loss_nodes)
            self._ws = st.workspace
            engine.run_forward(st, True)
            engine.run_backward(st, grads, st.d_out, None, True, True)
            loss = st.loss if loss is None else loss + st.loss
            outs.append(st.out)
            hids.append(st.out_hidden)
        out = outs[0] if len(outs) == 1 else torch.cat(outs)
        hid = hids[0] if len(hids) == 1 else torch.cat(hids)
        if not batched:
            out, hid = out[0], hid[0]
        return loss, out, hid


def split_regional_args(regional: Sequence, R: int):
    """accepts the reference's positional form (R edge_index tensors then R edge_attr
    tensors) or two lists."""
    regional = [r for r in regional if r is not None]
    if len(regional) == 2 and isinstance(regional[0], (list, tuple)):
        eis, eas = list(regional[0]), list(regional[1])
    else:
        if len(regional) != 2 * R:
            raise TypeError(f"expected {R} regional edge_index tensors followed by {R} edge_attr tensors, "
                            f"got {len(regional)} tensors")
        eis, eas = list(regional[:R]), list(regional[R:])
    if len(eis) != R or len(eas) != R:
        raise TypeError(f"model was built for {R} regions, got {len(eis)} edge lists / {len(eas)} weight lists")
    return eis, eas
