"""``generalconv`` and ``sageinitconv`` — the remaining design-space layers that are re-parameterisations of the hot-path
primitives (SURVEY §8f item 4).

GeneralConvLayer (ref: graphgym/contrib/layer/generalconv.py:12-113): h = x W; optional GCN normalisation
(``cfg.gnn.normalize_adj``: remaining self loops, degree over edge_index[0]); aggregate with ``cfg.gnn.agg``; then the self
message ``cfg.gnn.self_msg``: 'none' | 'add' (+ h) | 'concat' (+ x W_self); + bias.  ``agg = 'max'``: torch_scatter's
scatter_max (empty rows 0), the gradient to the first in-edge that reaches each column's maximum.
SAGEConvLayer (ref: graphgym/contrib/layer/sageinitconv.py:12-102, used with concat=True by ``sageinitconv``):
[x || mean_j x_j] W + bias, no self loops.
"""
import torch
import torch.nn as nn
from torch.nn import Parameter

from graphgym_b200 import functional as F_
from graphgym_b200 import ops
from graphgym_b200.config import cfg
from graphgym_b200.contrib.layer.idconv import glorot_, zeros_
from graphgym_b200.graph import get_layout
from graphgym_b200.register import register_layer


class GeneralConvLayer(nn.Module):
    def __init__(self, in_channels, out_channels, improved=False, cached=False, bias=True, **kwargs):
        super().__init__()
        if cfg.gnn.agg not in ('add', 'mean', 'max'):
            raise NotImplementedError("cfg.gnn.agg = {!r}: 'add', 'mean' and 'max' are on the accelerated path".format(
                cfg.gnn.agg))
        if improved:
            raise NotImplementedError('improved=True is never set by the GraphGym wrappers (ref: layer.py:189-191)')
        self.in_channels, self.out_channels = in_channels, out_channels
        self.aggr, self.normalize = cfg.gnn.agg, cfg.gnn.normalize_adj
        self.self_msg = cfg.gnn.get('self_msg', 'concat')
        if self.self_msg not in ('none', 'add', 'concat'):
            raise ValueError('self_msg {} not defined'.format(self.self_msg))
        self.weight = Parameter(torch.empty(in_channels, out_channels))
        if self.self_msg == 'concat':
            self.weight_self = Parameter(torch.empty(in_channels, out_channels))
        if bias:
            self.bias = Parameter(torch.empty(out_channels))
        else:
            self.register_parameter('bias', None)
        self.reset_parameters()

    def reset_parameters(self):
        glorot_(self.weight)
        if self.self_msg == 'concat':
            glorot_(self.weight_self)
        zeros_(self.bias)

    def forward(self, x, edge_index, edge_weight=None, edge_feature=None):
        if edge_weight is not None or edge_feature is not None:
            raise NotImplementedError('edge_weight / edge_feature are not on the accelerated path (GeneralConv passes neither)')
        n = x.size(0)
        h = F_.seg_linear([x], [self.weight], [(0, 0, False)])
        if self.normalize:
            layout = get_layout(edge_index, n, ops.LOOPS_ADD_REMAINING)
            kind = {'add': 'gcn_src', 'mean': 'gcn_src_mean', 'max': 'gcn_src_max'}[self.aggr]
        else:
            layout, kind = get_layout(edge_index, n, ops.LOOPS_KEEP), {'add': 'sum', 'mean': 'mean', 'max': 'max'}[self.aggr]
        if self.self_msg == 'none':
            return F_.aggregate(h, layout, kind, 0.0, self.bias)
        if self.self_msg == 'add':       # x_msg (+ bias, added in update) + x, x = the transformed features
            return F_.aggregate(h, layout, kind, 1.0, self.bias)
        x_self = F_.seg_linear([x], [self.weight_self], [(0, 0, False)])
        return F_.aggregate(h, layout, kind, 0.0, self.bias, residual=x_self)

    def __repr__(self):
        return '{}({}, {})'.format(self.__class__.__name__, self.in_channels, self.out_channels)


class GeneralConv(nn.Module):
    """ref: graphgym/models/layer.py:188-196 (a built-in of the reference's layer_dict)."""

    def __init__(self, dim_in, dim_out, bias=False, **kwargs):
        super().__init__()
        self.model = GeneralConvLayer(dim_in, dim_out, bias=bias)

    def forward(self, batch):
        batch.node_feature = self.model(batch.node_feature, batch.edge_index)
        return batch


class SAGEConvLayer(nn.Module):
    def __init__(self, in_channels, out_channels, normalize=False, concat=False, bias=True, **kwargs):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.normalize, self.concat = normalize, concat
        self.weight = Parameter(torch.empty(2 * in_channels if concat else in_channels, out_channels))
        if bias:
            self.bias = Parameter(torch.empty(out_channels))
        else:
            self.register_parameter('bias', None)
        self.reset_parameters()

    def reset_parameters(self):
        glorot_(self.weight)
        zeros_(self.bias)

    def forward(self, x, edge_index, edge_weight=None, size=None, res_n_id=None):
        if edge_weight is not None or size is not None or res_n_id is not None:
            raise NotImplementedError('edge_weight / bipartite inputs are not on the accelerated path')
        n, k = x.size(0), self.in_channels
        if self.concat:
            mean = F_.aggregate(x, get_layout(edge_index, n, ops.LOOPS_KEEP), 'mean')
            out = F_.seg_linear([x, mean], [self.weight], [(0, 0, False), (1, 0, False)], None, self.bias,
                                w_rows=((0, k), (k, 2 * k)))
        else:
            mean = F_.aggregate(x, get_layout(edge_index, n, ops.LOOPS_ADD_REMAINING), 'mean')
            out = F_.seg_linear([mean], [self.weight], [(0, 0, False)], None, self.bias)
        if self.normalize:
            out = F_.post_ops(out, None, self.training, ops.ACT_NONE, 0.0, True)
        return out

    def __repr__(self):
        return '{}({}, {})'.format(self.__class__.__name__, self.in_channels, self.out_channels)


class SAGEinitConv(nn.Module):
    """ref: sageinitconv.py:105-115."""

    def __init__(self, dim_in, dim_out, bias=False, **kwargs):
        super().__init__()
        self.model = SAGEConvLayer(dim_in, dim_out, bias=bias, concat=True)

    def forward(self, batch):
        batch.node_feature = self.model(batch.node_feature, batch.edge_index)
        return batch


register_layer('sageinitconv', SAGEinitConv)
