"""``TemporalGCN`` / ``A3TGCN`` of the reference (models/TemporalGCN.py:7-91) over the B200 kernels.

Same constructor ``TemporalGCN(node_features, periods, output_dim)``, same
``forward(x, edge_index, edge_attr) -> (h, out_hidden)`` (keyword call at run.py:188), same
state_dict keys.  Additive keyword arguments: ``hidden`` (reference: 256) and ``precision``.
x may be [N,F,T] (reference) or [B,N,F,T] (B independent snapshots on the same static graph)."""
import torch
import torch.nn as nn

from regt_b200 import _lib
from regt_b200.module_base import ChebConvParams, RegTModelBase, check_node_features, tgcn_param_dict
from regt_b200.plan import get_plan
from models.utils import TGCN


class A3TGCN(nn.Module):
    """parameter container with the reference's key names (models/TemporalGCN.py:35-73)."""

    def __init__(self, in_channels: int, out_channels: int, periods: int, improved: bool = False,
                 cached: bool = False, add_self_loops: bool = True):
        super().__init__()
        self.in_channels, self.out_channels, self.periods = in_channels, out_channels, periods
        self._base_tgcn = TGCN(in_channels, out_channels, baseblock="gcn")
        self.conv = ChebConvParams(in_channels, out_channels, K=2)
        self.linear = nn.Linear(64, out_channels)  # dead in the reference too (TemporalGCN.py:70); kept for keys
        self._attention = nn.Parameter(torch.empty(periods).uniform_())


class TemporalGCN(RegTModelBase):
    _mode = _lib.MODE_A3TGCN

    def __init__(self, node_features, periods, output_dim, hidden: int = 256, precision: str = "auto"):
        super().__init__()
        check_node_features(node_features)
        self.tgnn = A3TGCN(in_channels=node_features, out_channels=hidden, periods=periods)
        self.output_dim = output_dim
        self._hidden, self.precision = hidden, precision
        self.linear1 = nn.Linear(hidden, 128)
        self.linear2 = nn.Linear(128, output_dim)
        self.relu = nn.ReLU()

    def _param_dict(self):
        d = tgcn_param_dict(self.tgnn._base_tgcn)
        d.update(attention=self.tgnn._attention, cheb_w0=self.tgnn.conv.lins[0].weight,
                 cheb_w1=self.tgnn.conv.lins[1].weight, cheb_b=self.tgnn.conv.bias,
                 head_w1=self.linear1.weight, head_b1=self.linear1.bias,
                 head_w2=self.linear2.weight, head_b2=self.linear2.bias)
        return d

    def _plan(self, x, edge_index, edge_attr):
        N = x.shape[-3]
        # edge_attr reaches BOTH the ChebConv and the gcn_norm of the TGCN (TemporalGCN.py:88-90)
        return get_plan(N, x.device, edge_index, edge_attr, [edge_index], [edge_attr])

    def forward(self, x, edge_index, edge_attr=None):
        """x = node features for T time steps; returns (h [.,N,O], out_hidden [.,N,H])."""
        return self._run(x, self._plan(x, edge_index, edge_attr))

    def fused_step(self, x, y, edge_index, edge_attr=None, micro_batch=None):
        """forward + MSE loss + backward in one pass (run.py:188-190); grads accumulate in .grad."""
        return self._fused_step(x, y, self._plan(x, edge_index, edge_attr), micro_batch)
