"""``generalconv`` and ``sageinitconv`` — the remaining design-space layers that are re-parameterisations of the hot-path
primitives (SURVEY §8f item 4).

GeneralConvLayer (ref: graphgym/contrib/layer/generalconv.py:12-113): h = x W; optional GCN normalisation
(``cfg.gnn.normalize_adj``: remaining self loops, degree over edge_index[0]); aggregate with ``cfg.gnn.agg``; then the self
message ``cfg.gnn.self_msg``: 'none' | 'add' (+ h) | 'concat' (+ x W_self); + bias.  ``agg = 'max'``: torch_scatter's
scatter_max (empty rows 0), the gradient to the first in-edge that reaches each column's maximum.
GeneralEdgeConvLayer (ref: graphgym/contrib/layer/generalconv.py, GeneralEdgeConvLayer): the message on edge (j -> i)
is linear_msg([x_j | a_e]) or, with ``cfg.gnn.msg_direction = 'both'``, linear_msg([x_i | x_j | a_e]), a = edge_feature;
aggregated with ``cfg.gnn.agg``; + bias; then the self message.  ``generaledgeconv`` / ``generalsampleedgeconv`` (the
latter on the edges kept by rand(E) < cfg.gnn.keep_edge).
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


class GeneralEdgeConvLayer(nn.Module):
    """ref: graphgym/contrib/layer/generalconv.py, GeneralEdgeConvLayer.  The message on edge e = (j -> i) is
    linear_msg([x_j | a_e]) (``cfg.gnn.msg_direction = 'single'``) or linear_msg([x_i | x_j | a_e]) ('both'), a the edge
    features; aggregated with ``cfg.gnn.agg``; + bias; + the self message ('add': + x, 'concat': + linear_self(x)).

    linear_msg.weight is split by column blocks into W_i, W_j, W_a: h_j = x W_j^T (and h_i = x W_i^T) are node-level
    GEMMs, and ``functional.edge_aggregate`` adds the edge term without forming a per-edge tensor."""

    def __init__(self, in_channels, out_channels, improved=False, cached=False, bias=True, **kwargs):
        super().__init__()
        if cfg.gnn.agg not in ('add', 'mean', 'max'):
            raise NotImplementedError("cfg.gnn.agg = {!r}: 'add', 'mean' and 'max' are on the accelerated path".format(
                cfg.gnn.agg))
        if improved:
            raise NotImplementedError('improved=True is never set by the GraphGym wrappers')
        if cfg.gnn.normalize_adj:
            # the reference adds self loops to edge_index but not to edge_feature, so its message concatenation fails
            raise NotImplementedError('generaledgeconv with cfg.gnn.normalize_adj = True is not defined by the reference')
        self.in_channels, self.out_channels = in_channels, out_channels
        self.aggr = cfg.gnn.agg
        self.edge_dim = int(cfg.dataset.edge_dim)
        self.msg_direction = cfg.gnn.msg_direction
        if self.msg_direction not in ('single', 'both'):
            raise ValueError('msg_direction {} not defined'.format(self.msg_direction))
        self.self_msg = cfg.gnn.get('self_msg', 'concat')
        if self.self_msg not in ('none', 'add', 'concat'):
            raise ValueError('self_msg {} not defined'.format(self.self_msg))
        if self.self_msg == 'add' and in_channels != out_channels:
            raise ValueError("self_msg 'add' needs in_channels == out_channels (got {} and {})".format(
                in_channels, out_channels))
        if self.aggr == 'max' and self.edge_dim > ops.EDGE_MAX_KD:
            raise NotImplementedError('generaledgeconv: agg max needs cfg.dataset.edge_dim <= {} (got {})'.format(
                ops.EDGE_MAX_KD, self.edge_dim))
        k = (2 if self.msg_direction == 'both' else 1) * in_channels + self.edge_dim
        self.linear_msg = nn.Linear(k, out_channels, bias=False)
        if self.self_msg == 'concat':
            self.linear_self = nn.Linear(in_channels, out_channels, bias=False)
        if bias:
            self.bias = Parameter(torch.zeros(out_channels))
        else:
            self.register_parameter('bias', None)

    def forward(self, x, edge_index, edge_weight=None, edge_feature=None):
        if edge_weight is not None:
            raise NotImplementedError('edge_weight is not on the accelerated path (GeneralEdgeConv passes none)')
        e = edge_index.size(1)
        if (edge_feature is None or edge_feature.dim() != 2 or edge_feature.dtype != torch.float32
                or tuple(edge_feature.shape) != (e, self.edge_dim)):
            got = None if edge_feature is None else '{} {}'.format(tuple(edge_feature.shape), edge_feature.dtype)
            raise ValueError('edge_feature: expected a [{}, {}] float32 tensor (cfg.dataset.edge_dim = {}), got {}'.format(
                e, self.edge_dim, self.edge_dim, got))
        if cfg.b200.gather_dtype == 'bf16':
            raise NotImplementedError("cfg.b200.gather_dtype = 'bf16' has no edge-feature aggregation")
        fin = self.in_channels
        w = self.linear_msg.weight
        if self.msg_direction == 'both':
            h_i = F_.linear(x, w[:, :fin])
            h_j = F_.linear(x, w[:, fin:2 * fin])
            w_a = w[:, 2 * fin:]
        else:
            h_i = None
            h_j = F_.linear(x, w[:, :fin])
            w_a = w[:, fin:]
        if self.self_msg == 'concat':
            residual = F_.linear(x, self.linear_self.weight)
        elif self.self_msg == 'add':
            residual = x
        else:
            residual = None
        layout = get_layout(edge_index, x.size(0), ops.LOOPS_KEEP)
        return F_.edge_aggregate(h_j, h_i, edge_feature, w_a, layout, self.aggr, self.bias, residual)

    def __repr__(self):
        return '{}({}, {})'.format(self.__class__.__name__, self.in_channels, self.out_channels)


class GeneralEdgeConv(nn.Module):
    """ref: graphgym/models/layer.py, GeneralEdgeConv (a built-in of the reference's layer_dict)."""

    def __init__(self, dim_in, dim_out, bias=False, **kwargs):
        super().__init__()
        self.model = GeneralEdgeConvLayer(dim_in, dim_out, bias=bias)

    def forward(self, batch):
        batch.node_feature = self.model(batch.node_feature, batch.edge_index, edge_feature=batch.edge_feature)
        return batch


def sample_edges(edge_index, edge_feature, keep):
    """(edge_index, edge_feature) of the edges kept by rand(E) < keep, drawn on the device (torch's CUDA generator)."""
    if edge_feature is None:
        raise ValueError('edge_feature: generalsampleedgeconv needs batch.edge_feature')
    mask = torch.rand(edge_index.size(1), device=edge_index.device) < keep
    return edge_index[:, mask], edge_feature[mask, :]


class GeneralSampleEdgeConv(nn.Module):
    """ref: graphgym/models/layer.py, GeneralSampleEdgeConv: GeneralEdgeConvLayer on the edges kept by
    rand(E) < cfg.gnn.keep_edge, drawn on every forward (training and eval, as the reference)."""

    def __init__(self, dim_in, dim_out, bias=False, **kwargs):
        super().__init__()
        self.model = GeneralEdgeConvLayer(dim_in, dim_out, bias=bias)

    def forward(self, batch):
        edge_index, edge_feature = sample_edges(batch.edge_index, batch.edge_feature, cfg.gnn.keep_edge)
        batch.node_feature = self.model(batch.node_feature, edge_index, edge_feature=edge_feature)
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
