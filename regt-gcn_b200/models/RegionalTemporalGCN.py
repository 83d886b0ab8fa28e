"""``RegionalTemporalGCN`` / ``RegionalA3TGCN`` of the reference
(models/RegionalTemporalGCN.py:9-149) over the B200 kernels.

Same constructor ``RegionalTemporalGCN(node_features, num_nodes, periods, output_dim)``, same
12-tensor positional ``forward`` returning ``(h, out_hidden)`` (call sites run.py:178,214), same 26
state_dict keys -- the reference's shipped checkpoints load with ``strict=True``.  Additive keyword
arguments: ``hidden`` (reference 256), ``n_regions`` (reference 5) and ``precision``.
For R != 5 pass two lists: ``forward(x, edge_index, [ei_0..ei_R-1], [ea_0..ea_R-1])``.
x may be [N,F,T] (reference) or [B,N,F,T] (B independent snapshots on the same static graph)."""
import torch
import torch.nn as nn

from regt_b200 import _lib
from regt_b200.module_base import (ChebConvParams, RegTModelBase, check_node_features, split_regional_args,
                                   tgcn_param_dict)
from regt_b200.plan import get_plan
from models.utils import TGCN


class RegionalA3TGCN(nn.Module):
    """parameter container with the reference's key names (models/RegionalTemporalGCN.py:47-88).
    ``_weight_att{1,2}`` / ``_bias_att{1,2}`` are dead in the reference (``attention()`` :91-111 is
    never called); they exist for checkpoint compatibility and never receive gradients."""

    def __init__(self, in_channels: int, out_channels: int, num_nodes: int, periods: int, improved: bool = False,
                 cached: bool = False, add_self_loops: bool = True, n_regions: int = 5):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.num_nodes, self.periods, self.n_regions = num_nodes, periods, n_regions
        self._base_tgcn = TGCN(in_channels, out_channels, improved=improved, cached=cached,
                               add_self_loops=add_self_loops)
        self.conv = ChebConvParams(in_channels, out_channels, K=2)
        self.linear = nn.Linear(out_channels * n_regions, out_channels)
        self._attention = nn.Parameter(torch.empty(periods).uniform_())
        self._weight_att1 = nn.Parameter(torch.normal(0.0, 0.1, size=(out_channels, 1)))
        self._weight_att2 = nn.Parameter(torch.normal(0.0, 0.1, size=(num_nodes, 1)))
        self._bias_att1 = nn.Parameter(torch.normal(0.0, 1.0, size=(1, 1)))
        self._bias_att2 = nn.Parameter(torch.normal(0.0, 1.0, size=(1, 1)))


class RegionalTemporalGCN(RegTModelBase):
    _mode = _lib.MODE_REGIONAL

    def __init__(self, node_features, num_nodes, periods, output_dim, hidden: int = 256, n_regions: int = 5,
                 precision: str = "auto"):
        super().__init__()
        check_node_features(node_features)
        self.tgnn = RegionalA3TGCN(in_channels=node_features, out_channels=hidden, num_nodes=num_nodes,
                                   periods=periods, n_regions=n_regions)
        self.output_dim = output_dim
        self._hidden, self._n_regions, self.precision = hidden, n_regions, precision
        self.linear1 = nn.Linear(hidden, 128)
        self.linear2 = nn.Linear(128, output_dim)
        self.relu = nn.ReLU()

    def _param_dict(self):
        d = tgcn_param_dict(self.tgnn._base_tgcn)
        d.update(attention=self.tgnn._attention, cheb_w0=self.tgnn.conv.lins[0].weight,
                 cheb_w1=self.tgnn.conv.lins[1].weight, cheb_b=self.tgnn.conv.bias,
                 comb_w=self.tgnn.linear.weight, comb_b=self.tgnn.linear.bias,
                 head_w1=self.linear1.weight, head_b1=self.linear1.bias,
                 head_w2=self.linear2.weight, head_b2=self.linear2.bias)
        return d

    def _plan(self, x, edge_index, regional):
        eis, eas = split_regional_args(regional, self._n_regions)
        N = x.shape[-3]
        # the wrapper never forwards edge_weight: the full-graph TGCN sees None (unit weights),
        # the regional ChebConvs see the raw distances (RegionalTemporalGCN.py:128,136-148)
        return get_plan(N, x.device, edge_index, None, eis, eas)

    def step_plan(self, x, edge_index, *regional):
        """the graph plan ``fused_step`` runs on for these graph arguments (``loop.train_epoch(share_periods=True)``)"""
        return self._plan(x, edge_index, regional)

    def forward(self, x, edge_index, IAedge_index=None, KSedge_index=None, KYedge_index=None, OHedge_index=None,
                WIedge_index=None, IAedge_attr=None, KSedge_attr=None, KYedge_attr=None, OHedge_attr=None,
                WIedge_attr=None, *more):
        """x = node features for T time steps, edge_index = full graph; then the regional edge
        lists and their weights.  Returns (h [.,N,O], out_hidden [.,N,H])."""
        regional = (IAedge_index, KSedge_index, KYedge_index, OHedge_index, WIedge_index, IAedge_attr, KSedge_attr,
                    KYedge_attr, OHedge_attr, WIedge_attr) + tuple(more)
        return self._run(x, self._plan(x, edge_index, regional))

    def fused_step(self, x, y, edge_index, *regional, micro_batch=None, loss="mse", null_value=None):
        """forward + MSE loss + backward in one pass (run.py:178-190); grads accumulate in .grad.
        ``loss="mae"``: mean absolute error; ``null_value``: targets equal to it (or NaN) are missing and left out."""
        return self._fused_step(x, y, self._plan(x, edge_index, regional), micro_batch, loss=loss, null_value=null_value)
