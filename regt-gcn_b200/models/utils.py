"""``models.utils.TGCN`` of the reference (models/utils.py:69-203) over the B200 kernels.

Same constructor, same ``forward(X, edge_index, edge_weight=None, H=None) -> H'`` and the same
state_dict keys (``conv_{z,r,h}.lin.weight``, ``conv_{z,r,h}.bias``, ``linear_{z,r,h}.{weight,bias}``).
The three GCNConv + three Linear(2H,H) + GRU blend of the reference are one fused pass
(csrc/cell.cu); only ``baseblock="gcn"`` is on the accelerated path."""
from typing import Optional

import torch
import torch.nn as nn

from regt_b200 import _lib, engine
from regt_b200.module_base import GCNConvParams, check_node_features, tgcn_param_dict
from regt_b200.plan import get_plan


class TGCN(nn.Module):
    def __init__(self, in_channels: int, out_channels: int, baseblock: str = "gcn", improved: bool = False,
                 cached: bool = False, add_self_loops: bool = True, precision: str = "fp32"):
        super().__init__()
        if baseblock in ("gat", "graphsage"):
            raise NotImplementedError("baseblock %s is outside the B200 hot path (only 'gcn' is built)" % baseblock)
        if baseblock != "gcn":
            raise NotImplementedError("Current baseblock %s is not supported." % (baseblock))
        if improved or not add_self_loops:
            raise NotImplementedError("only improved=False, add_self_loops=True (the reference's use) is built")
        check_node_features(in_channels)
        self.in_channels, self.out_channels = in_channels, out_channels
        self.improved, self.cached, self.add_self_loops, self.baseblock = improved, cached, add_self_loops, baseblock
        self.precision = precision
        for g in "zrh":
            setattr(self, f"conv_{g}", GCNConvParams(in_channels, out_channels))
            setattr(self, f"linear_{g}", nn.Linear(2 * out_channels, out_channels))

    def forward(self, X: torch.Tensor, edge_index: torch.Tensor, edge_weight: Optional[torch.Tensor] = None,
                H: Optional[torch.Tensor] = None) -> torch.Tensor:
        if X.dim() != 2:
            raise ValueError("TGCN.forward expects X of shape [num_nodes, in_channels]")
        N = X.shape[0]
        plan = get_plan(N, X.device, edge_index, edge_weight, [], [], need_cheb=False)
        x4 = X.to(torch.float32).contiguous().view(1, N, self.in_channels, 1)
        h_ext = None
        if H is not None:  # H=None -> zeros (models/utils.py:163-166)
            h_ext = H.to(torch.float32).contiguous().view(1, N, 1, self.out_channels)
        out = engine.model_apply(_lib.MODE_TGCN, _lib.PRECISIONS["fp32" if self.precision == "auto" else self.precision], plan, self.out_channels, 1, x4,
                                 tgcn_param_dict(self), h_ext, head=False)
        return out[0]
