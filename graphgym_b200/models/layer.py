"""The reference's built-in message-passing layers and the ``layer_dict`` they are served from
(ref: graphgym/models/layer.py:16-47,135-174,224-238).

``gcnconv / sageconv / ginconv / gatconv`` wrap ``pyg.nn.*Conv`` in the reference; torch_geometric is
neither vendored nor a dependency here, so each layer restates the PyG module's semantics
(parameters, init, self-loop policy, normalisation) over the gg_* CUDA path:

    GCNConv   add_remaining_self_loops, deg over the target, X W then propagate, + bias
    SAGEConv  lin_l(mean_j x_j) + lin_r(x_i), no self loops            (PyG >= 1.6 SAGEConv)
    GINConv   nn((1 + eps) x_i + sum_j x_j), eps = 0 buffer, loops kept
    GATConv   remove + add self loops, additive attention (slope 0.2, heads=1), edge-softmax fused
              into the aggregation (parameters weight / att / bias as in PyG <= 1.5 and idconv.py)
    SplineConv  PyG 1.6 SplineConv(dim=1, kernel_size=2): the mean over the in-edges of the degree-1 open B-spline
              weighting of the pseudo-coordinate ``edge_feature[e, 0]``, + x root + bias; loops kept, none added
"""
import math

import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.nn import Parameter

import graphgym_b200.register as register
from graphgym_b200 import functional as F_
from graphgym_b200 import ops
from graphgym_b200.config import cfg
from graphgym_b200.contrib.layer import idconv as _idconv  # registers the ID layers
from graphgym_b200.contrib.layer import generalconv as _generalconv  # registers sageinitconv; GeneralConv is a built-in
from graphgym_b200.contrib.layer import tfg as _tfg  # registers Tfg-idgcn / Tfg-idsage / Tfg-idgin / Tfg-idgat
from graphgym_b200.contrib.layer import attconv as _attconv  # registers gaddconv / gmulconv
from graphgym_b200.contrib.layer.idconv import _mlp, glorot_, zeros_
from graphgym_b200.graph import get_layout


class _GCNConvLayer(nn.Module):
    def __init__(self, in_channels, out_channels, bias=True):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.weight = Parameter(torch.empty(in_channels, out_channels))
        if bias:
            self.bias = Parameter(torch.empty(out_channels))
        else:
            self.register_parameter('bias', None)
        self.reset_parameters()

    def reset_parameters(self):
        glorot_(self.weight)
        zeros_(self.bias)

    def forward(self, x, edge_index):
        n = x.size(0)
        h = F_.seg_linear([x], [self.weight], [(0, 0, False)])
        return F_.aggregate(h, get_layout(edge_index, n, ops.LOOPS_ADD_REMAINING), 'gcn_tgt', 0.0,
                            self.bias)


class _SAGEConvLayer(nn.Module):
    def __init__(self, in_channels, out_channels, bias=True):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.lin_l = nn.Linear(in_channels, out_channels, bias=bias)
        self.lin_r = nn.Linear(in_channels, out_channels, bias=False)

    def forward(self, x, edge_index):
        mean = F_.aggregate(x, get_layout(edge_index, x.size(0), ops.LOOPS_KEEP), 'mean')
        return F_.seg_linear([mean, x], [self.lin_l.weight, self.lin_r.weight],
                             [(0, 0, False), (1, 1, False)], None, self.lin_l.bias, w_trans=True)


class _GINConvLayer(nn.Module):
    def __init__(self, nn_, eps=0.0):
        super().__init__()
        self.nn = nn_
        self.initial_eps = eps
        self.register_buffer('eps', torch.Tensor([eps]))

    def forward(self, x, edge_index):
        z = F_.aggregate(x, get_layout(edge_index, x.size(0), ops.LOOPS_KEEP), 'sum',
                         self_scale=1.0 + float(self.initial_eps))
        return _mlp(self.nn, z)


class _GATConvLayer(nn.Module):
    def __init__(self, in_channels, out_channels, heads=1, negative_slope=0.2, bias=True):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.heads, self.negative_slope = heads, negative_slope
        self.weight = Parameter(torch.empty(in_channels, heads * out_channels))
        self.att = Parameter(torch.empty(1, heads, 2 * out_channels))
        if bias:
            self.bias = Parameter(torch.empty(heads * out_channels))
        else:
            self.register_parameter('bias', None)
        self.reset_parameters()

    def reset_parameters(self):
        glorot_(self.weight)
        glorot_(self.att)
        zeros_(self.bias)

    def forward(self, x, edge_index):
        n = x.size(0)
        h = F_.seg_linear([x], [self.weight], [(0, 0, False)])
        layout = get_layout(edge_index, n, ops.LOOPS_REMOVE_ADD)
        return F_.gat_aggregate(h, self.att, self.bias, layout, self.heads, self.negative_slope)


class _SplineConvLayer(nn.Module):
    """PyG 1.6 ``SplineConv`` for dim = 1, kernel_size = 2, degree = 1, open spline, aggr 'mean', root weight: with
    t = trunc(u_e), fr = u_e - floor(u_e), edge e = (j -> i) weighs x_j by 1 - fr through kernel matrix t mod 2 and by fr
    through (t + 1) mod 2 (a non-negative mod: for u_e <= -1, where the reference indexes weight[-1], this is the
    continuation of the pattern it has for u_e > -1).  out_i = mean_e (...) + x_i root + bias; a row without in-edges gets
    x_i root + bias.  The other settings of the reference class are refused."""

    def __init__(self, in_channels, out_channels, dim=1, kernel_size=2, is_open_spline=True, degree=1, bias=True):
        super().__init__()
        if dim != 1 or kernel_size != 2 or degree != 1 or not is_open_spline:
            raise NotImplementedError('SplineConv: only dim=1, kernel_size=2, degree=1 with an open spline are on the '
                                      'accelerated path (got dim={}, kernel_size={}, degree={}, is_open_spline={})'.format(
                                          dim, kernel_size, degree, is_open_spline))
        self.in_channels, self.out_channels = in_channels, out_channels
        self.register_buffer('kernel_size', torch.tensor([kernel_size], dtype=torch.long))
        self.register_buffer('is_open_spline', torch.tensor([1], dtype=torch.uint8))
        self.weight = Parameter(torch.empty(kernel_size, in_channels, out_channels))
        self.root = Parameter(torch.empty(in_channels, out_channels))
        if bias:
            self.bias = Parameter(torch.empty(out_channels))
        else:
            self.register_parameter('bias', None)
        self.reset_parameters()

    def reset_parameters(self):
        bound = 1.0 / math.sqrt(self.weight.size(0) * self.weight.size(1))     # PyG's uniform(size, t)
        for t in (self.weight, self.root, self.bias):
            if t is not None:
                with torch.no_grad():
                    t.uniform_(-bound, bound)

    def forward(self, x, edge_index, pseudo):
        e = edge_index.size(1)
        if pseudo is None:
            raise ValueError('edge_feature: splineconv needs the pseudo-coordinates batch.edge_feature ([E] or [E, 1])')
        if pseudo.dtype != torch.float32:
            raise ValueError('edge_feature: splineconv needs float32 pseudo-coordinates, got {}'.format(pseudo.dtype))
        if pseudo.dim() == 2 and pseudo.size(1) != 1:
            raise ValueError('edge_feature: splineconv has dim=1 (one pseudo-coordinate per edge), got {}; PyG\'s dim=1 '
                             'basis would read out of bounds on a wider edge_feature'.format(tuple(pseudo.shape)))
        if pseudo.dim() not in (1, 2) or pseudo.size(0) != e:
            raise ValueError('edge_feature: expected [{}] or [{}, 1] pseudo-coordinates, got {}'.format(
                e, e, tuple(pseudo.shape)))
        if cfg.b200.gather_dtype == 'bf16':
            raise NotImplementedError("cfg.b200.gather_dtype = 'bf16' has no splineconv aggregation")
        layout = get_layout(edge_index, x.size(0), ops.LOOPS_KEEP)
        return F_.spline_aggregate(x, pseudo, self.weight, self.root, self.bias, layout,
                                   self.in_channels <= self.out_channels)

    def __repr__(self):
        return '{}({}, {}, dim=1)'.format(self.__class__.__name__, self.in_channels, self.out_channels)


class _EdgeIndexWrapper(nn.Module):
    def forward(self, batch):
        batch.node_feature = self.model(batch.node_feature, batch.edge_index)
        return batch


class GCNConv(_EdgeIndexWrapper):
    def __init__(self, dim_in, dim_out, bias=False, **kwargs):
        super().__init__()
        self.model = _GCNConvLayer(dim_in, dim_out, bias=bias)


class SAGEConv(_EdgeIndexWrapper):
    def __init__(self, dim_in, dim_out, bias=False, **kwargs):
        super().__init__()
        self.model = _SAGEConvLayer(dim_in, dim_out, bias=bias)


class GATConv(_EdgeIndexWrapper):
    def __init__(self, dim_in, dim_out, bias=False, **kwargs):
        super().__init__()
        self.model = _GATConvLayer(dim_in, dim_out, bias=bias)


class GINConv(_EdgeIndexWrapper):
    def __init__(self, dim_in, dim_out, bias=False, **kwargs):
        super().__init__()
        gin_nn = nn.Sequential(nn.Linear(dim_in, dim_out), nn.ReLU(), nn.Linear(dim_out, dim_out))
        self.model = _GINConvLayer(gin_nn)


class SplineConv(nn.Module):
    """ref: graphgym/models/layer.py, SplineConv: pyg.nn.SplineConv(dim_in, dim_out, dim=1, kernel_size=2) over
    (node_feature, edge_index, edge_feature); cfg.gnn.agg / normalize_adj are not read."""

    def __init__(self, dim_in, dim_out, bias=False, **kwargs):
        super().__init__()
        self.model = _SplineConvLayer(dim_in, dim_out, dim=1, kernel_size=2, bias=bias)

    def forward(self, batch):
        batch.node_feature = self.model(batch.node_feature, batch.edge_index, batch.edge_feature)
        return batch


_ACT = {'relu': nn.ReLU, 'selu': nn.SELU, 'prelu': nn.PReLU, 'elu': nn.ELU,
        'lrelu_01': lambda: nn.LeakyReLU(0.1), 'lrelu_025': lambda: nn.LeakyReLU(0.25),
        'lrelu_05': lambda: nn.LeakyReLU(0.5)}


_FUSED_ACT = {'relu': (ops.ACT_RELU, 0.0), 'lrelu_01': (ops.ACT_LRELU, 0.1), 'lrelu_025': (ops.ACT_LRELU, 0.25),
              'lrelu_05': (ops.ACT_LRELU, 0.5)}


class GeneralLayer(nn.Module):
    """Caller of the hot path (ref: layer.py:16-47): layer -> BN -> dropout -> act -> optional L2.

    The modules of ``post_layer`` are kept as the parameter / buffer holders (same ``state_dict`` keys as the reference);
    on CUDA tensors the post-ops run as ONE fused pass (``functional.post_ops``: BN statistics, normalise + affine +
    activation + row L2) whenever the combination is on the fused path — BatchNorm1d and/or ReLU / leaky ReLU and/or L2,
    no active dropout; anything else (PReLU / ELU / SELU, dropout > 0 while training) runs the modules one by one."""

    def __init__(self, name, dim_in, dim_out, has_act=True, has_bn=True, has_l2norm=False, **kwargs):
        super().__init__()
        self.has_l2norm = has_l2norm
        has_bn = has_bn and cfg.gnn.batchnorm
        self.layer = layer_dict[name](dim_in, dim_out, bias=not has_bn, **kwargs)
        post = []
        if has_bn:
            post.append(nn.BatchNorm1d(dim_out, eps=cfg.bn.eps, momentum=cfg.bn.mom))
        if cfg.gnn.dropout > 0:
            post.append(nn.Dropout(p=cfg.gnn.dropout, inplace=cfg.mem.inplace))
        if has_act:
            post.append(_ACT[cfg.gnn.act]())
        self.post_layer = nn.Sequential(*post)
        self._has_bn = bool(has_bn)        # post_layer[0] is the BatchNorm1d (not re-registered under a second name)
        self._drop_p = cfg.gnn.dropout
        self._act = _FUSED_ACT.get(cfg.gnn.act) if has_act else (ops.ACT_NONE, 0.0)

    def _post(self, h):
        fused = (h.is_cuda and h.dim() == 2 and h.dtype == torch.float32 and self._act is not None
                 and not (self._drop_p > 0 and self.training) and cfg.b200.fused_postops)
        if fused:
            bn = self.post_layer[0] if self._has_bn else None
            if bn is None and self._act[0] == ops.ACT_NONE and not self.has_l2norm:
                return h
            return F_.post_ops(h, bn, self.training, self._act[0], self._act[1], self.has_l2norm)
        h = self.post_layer(h)
        if self.has_l2norm:
            h = F.normalize(h, p=2, dim=1)
        return h

    def forward(self, batch):
        batch = self.layer(batch)
        if isinstance(batch, torch.Tensor):
            batch = self._post(batch)
        else:
            batch.node_feature = self._post(batch.node_feature)
        return batch


_builtin = {
    'gcnconv': GCNConv,
    'sageconv': SAGEConv,
    'gatconv': GATConv,
    'ginconv': GINConv,
    'generalconv': _generalconv.GeneralConv,
    'generaledgeconv': _generalconv.GeneralEdgeConv,
    'generalsampleedgeconv': _generalconv.GeneralSampleEdgeConv,
    'splineconv': SplineConv,
}

# built-ins win on a name clash, contrib registrations fill the rest (ref: layer.py:238)
layer_dict = {**register.layer_dict, **_builtin}

# main_zd.py names (ref: main_zd.py:299-308).  The four ID layers of TfgIDLayer.py are registered with THEIR semantics
# (contrib/layer/tfg.py: 'Tfg-idgcn', 'Tfg-idsage', 'Tfg-idgin', 'Tfg-idgat').  The plain Tfg-* layers are tf_geometric's
# own (un-vendored third party, not in the reference tree): those names select the PyG-semantics operators.
TFG_ALIASES = {
    'Tfg-gcnconv': 'gcnconv', 'Tfg-sageconv': 'sageconv', 'Tfg-ginconv': 'ginconv', 'Tfg-gatconv': 'gatconv',
}


def resolve_layer(name):
    """``layer_dict`` lookup that also accepts the ``Tfg-*`` names of ``config/*_tf``."""
    return layer_dict[TFG_ALIASES.get(name, name)]


class Batch:
    """Minimal stand-in for a DeepSNAP batch: the attributes the layers touch (``edge_feature``: [E, edge_dim] rows in
    edge_index order, read by the edge-feature layers)."""

    def __init__(self, node_feature, edge_index, node_id_index=None, edge_feature=None):
        self.node_feature = node_feature
        self.edge_index = edge_index
        self.node_id_index = node_id_index
        self.edge_feature = edge_feature
