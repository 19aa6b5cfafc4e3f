"""``gaddconv`` / ``gmulconv`` — the design-space attention layers (ref: graphgym/contrib/layer/attconv.py:14-240) on the
primitives the GAT layers already use (SURVEY §8f item 4).

GeneralAddAttConvLayer (attconv.py:14-112): h = linear_msg(x); additive attention leaky_relu_{0.2}(att . [h_i || h_j])
soft-maxed over the edges that share a target; out_i = sum alpha_ij h_j (+ bias).  Unlike GATConv it does NOT edit self
loops: the attention runs on the edge list as given.  -> ``functional.gat_aggregate`` on the LOOPS_KEEP layout.
GeneralMulAttConvLayer (attconv.py:115-214): logits (<h_i, h_j> + sum(bias_att)) / sqrt(out_channels); the additive
constant cancels in the softmax (its gradient is zero, as autograd finds in the reference up to rounding), so the layer is
scaled dot-product attention with Q = K = V = h.  -> the SDDMM / segment-softmax / SpMM passes of contrib/layer/tfg.py.
``cfg.gnn.agg`` picks the reduction over a target's in-edges (the edge list as given, duplicates counted):
  'add'   the sum above (GraphGym's default).
  'mean'  the sum divided by the in-degree (0 without in-edges), then + bias -> ``functional.gat_aggregate(agg='mean')``
          on every path the sum takes (fused sliced-ELL, merge-path, row) / ``spmm(MEAN)`` with the alpha weights.
  'max'   per column the largest message alpha_ij h_j (0 without in-edges), then + bias; torch_scatter's scatter_max:
          the gradient goes to the first in-edge in edge order that reaches the maximum, and through it to h_j and to
          alpha_ij (the softmax, att and the scores).  The weighted max of csrc/spmm_max.cu (sliced ELL for heads = 1,
          a warp-per-row kernel with one weight per (edge, head) otherwise) and the winner SDDMM of csrc/attn_agg.cu.
``cfg.gnn.normalize_adj = True`` is not on the accelerated path.
"""
import math

import torch
import torch.nn as nn
from torch.nn import Parameter

from graphgym_b200 import functional as F_
from graphgym_b200 import ops
from graphgym_b200.config import cfg
from graphgym_b200.contrib.layer.idconv import glorot_, zeros_
from graphgym_b200.contrib.layer.tfg import _DotAttention
from graphgym_b200.graph import get_layout
from graphgym_b200.register import register_layer


def _check_cfg(name):
    if cfg.gnn.normalize_adj or cfg.gnn.agg not in ('add', 'mean', 'max'):
        raise NotImplementedError(f"{name}: cfg.gnn.normalize_adj / agg {cfg.gnn.agg!r} are not on the accelerated path")
    return cfg.gnn.agg


class GeneralAddAttConvLayer(nn.Module):
    def __init__(self, in_channels, out_channels, improved=False, cached=False, bias=True, **kwargs):
        super().__init__()
        self.agg = _check_cfg('gaddconv')
        self.heads = int(cfg.gnn.get('att_heads', 1))
        self.in_channels = in_channels // self.heads * self.heads
        self.out_channels = out_channels // self.heads * self.heads
        self.negative_slope = 0.2
        self.head_channels = out_channels // self.heads
        self.linear_msg = nn.Linear(in_channels, out_channels, bias=False)
        self.att = Parameter(torch.empty(1, self.heads, 2 * self.head_channels))
        if bias:
            self.bias = Parameter(torch.empty(out_channels))
        else:
            self.register_parameter('bias', None)
        self.reset_parameters()

    def reset_parameters(self):
        glorot_(self.att)
        zeros_(self.bias)

    def forward(self, x, edge_index, edge_weight=None):
        if edge_weight is not None:
            raise NotImplementedError('edge_weight is never passed by GeneralAddAttConv')
        h = F_.linear(x, self.linear_msg.weight, None)
        layout = get_layout(edge_index, x.size(0), ops.LOOPS_KEEP)
        return F_.gat_aggregate(h, self.att, self.bias, layout, self.heads, self.negative_slope, self.agg)

    def __repr__(self):
        return '{}({}, {}, {})'.format(self.__class__.__name__, self.in_channels, self.out_channels, self.heads)


class GeneralMulAttConvLayer(nn.Module):
    def __init__(self, in_channels, out_channels, improved=False, cached=False, bias=True, **kwargs):
        super().__init__()
        self.agg = _check_cfg('gmulconv')
        if int(cfg.gnn.get('att_heads', 1)) != 1:
            raise NotImplementedError('gmulconv: "currently only for single head attention" (attconv.py:134)')
        self.in_channels, self.out_channels = in_channels, out_channels
        self.linear_msg = nn.Linear(in_channels, out_channels, bias=False)
        self.bias_att = Parameter(torch.zeros(out_channels))      # cancels in the softmax: gradient identically zero
        if bias:
            self.bias = Parameter(torch.zeros(out_channels))
        else:
            self.register_parameter('bias', None)

    def forward(self, x, edge_index, edge_weight=None):
        if edge_weight is not None:
            raise NotImplementedError('edge_weight is never passed by GeneralMulAttConv')
        h = F_.linear(x, self.linear_msg.weight, None)
        layout = get_layout(edge_index, x.size(0), ops.LOOPS_KEEP)
        # 1 / scaler = 1 / sqrt(out_channels); _DotAttention scales by 1 / sqrt(q.size(1)) = the same
        if self.agg == 'add':
            return _DotAttention.apply(h, h, h, self.bias, layout)
        return F_.dot_attention_aggregate(h, self.bias, layout, self.agg)

    def __repr__(self):
        return '{}({}, {}, 1)'.format(self.__class__.__name__, self.in_channels, self.out_channels)


class GeneralAddAttConv(nn.Module):
    def __init__(self, dim_in, dim_out, bias=False, **kwargs):
        super().__init__()
        self.model = GeneralAddAttConvLayer(dim_in, dim_out, bias=bias)

    def forward(self, batch):
        batch.node_feature = self.model(batch.node_feature, batch.edge_index)
        return batch


class GeneralMulAttConv(nn.Module):
    def __init__(self, dim_in, dim_out, bias=False, **kwargs):
        super().__init__()
        self.model = GeneralMulAttConvLayer(dim_in, dim_out, bias=bias)

    def forward(self, batch):
        batch.node_feature = self.model(batch.node_feature, batch.edge_index)
        return batch


register_layer('gaddconv', GeneralAddAttConv)
register_layer('gmulconv', GeneralMulAttConv)
