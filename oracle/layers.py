"""CPU restatement of the hot-path layers (TEST INFRASTRUCTURE ONLY — see oracle/__init__.py).

Every function follows the reference's op sequence — dense transform, index_select gather, per-edge
scale, index_add_ scatter — in plain torch on the CPU, in whatever dtype its inputs carry (fp32 to
time "the reference's CPU path", fp64 to arbitrate).  Parameters are passed explicitly so the same
tensors can be loaded into the CUDA layers.  Gradients come from torch autograd over these ops,
which is exactly how the reference obtains them (train.py:24).
"""
import torch
import torch.nn.functional as F

from . import pyg_utils as U


def id_transform(x, ids, weight, weight_id):
    """ref: idconv.py:64-67,152-155,307-310 — X W, then index_add_ of X[id] W_id."""
    x_id = torch.index_select(x, 0, ids) @ weight_id
    h = x @ weight
    return h.index_add(0, ids, x_id)


def gcn_norm_src(edge_index, num_nodes, dtype, improved=False):
    """ref: idconv.py:132-148 / identity.py:7-22 — remaining self loops, degree over edge_index[0]."""
    w = torch.ones(edge_index.size(1), dtype=dtype, device=edge_index.device)
    edge_index, w = U.add_remaining_self_loops(edge_index, w, 2 if improved else 1, num_nodes)
    row, col = edge_index
    deg = U.scatter_add(w, row, 0, num_nodes)
    dis = deg.pow(-0.5)
    dis[dis == float('inf')] = 0
    return edge_index, dis[row] * w * dis[col]


def gcn_norm_tgt(edge_index, num_nodes, dtype):
    """PyG >= 1.6 ``gcn_norm`` (used by pyg.nn.GCNConv, ref: layer.py:138): degree over edge_index[1]."""
    w = torch.ones(edge_index.size(1), dtype=dtype, device=edge_index.device)
    edge_index, w = U.add_remaining_self_loops(edge_index, w, 1, num_nodes)
    row, col = edge_index
    deg = U.scatter_add(w, col, 0, num_nodes)
    dis = deg.pow(-0.5)
    dis.masked_fill_(dis == float('inf'), 0)
    return edge_index, dis[row] * w * dis[col]


def _prop(edge_index, x, num_nodes, aggr='add', norm=None):
    """gather x_j = x[edge_index[0]], optional per-edge scale, scatter to edge_index[1]."""
    x_j = x.index_select(0, edge_index[0])
    if norm is not None:
        x_j = norm.view(-1, 1) * x_j
    return U.propagate(edge_index, x_j, num_nodes, aggr)


# ---- built-in layers (ref: layer.py:135-174 -> pyg.nn.*) --------------------------------------
def gcnconv(x, edge_index, weight, bias=None):
    n = x.size(0)
    ei, norm = gcn_norm_tgt(edge_index, n, x.dtype)
    out = _prop(ei, x @ weight, n, 'add', norm)
    return out if bias is None else out + bias


def sageconv(x, edge_index, w_l, b_l, w_r):
    """PyG >= 1.6 SAGEConv: lin_l(mean_j x_j) + lin_r(x_i); weights are nn.Linear [out,in]."""
    mean = _prop(edge_index, x, x.size(0), 'mean')
    out = F.linear(mean, w_l, b_l)
    return out + F.linear(x, w_r)


def _gin_mlp(z, p, gate=None, tap=None, key='pre'):
    """Linear -> ReLU -> Linear (ref: layer.py:168-169, idconv.py:432-435).  ``gate`` (a 0/1 tensor)
    replaces the ReLU's own gate so that gradients can be compared under the gates the implementation
    under test actually took (a pre-activation within rounding of zero may gate either way); ``tap``
    collects the pre-activation for the caller's tolerance check."""
    pre = F.linear(z, p[0], p[1])
    if tap is not None:
        tap[key] = pre.detach()
    h = F.relu(pre) if gate is None else pre * gate.to(pre.dtype)
    return F.linear(h, p[2], p[3])


def ginconv(x, edge_index, w1, b1, w2, b2, eps=0.0, gate=None, tap=None):
    z = (1 + eps) * x + _prop(edge_index, x, x.size(0), 'add')
    return _gin_mlp(z, (w1, b1, w2, b2), gate, tap)


def _gat_core(h, edge_index, att, heads, out_channels, negative_slope, bias, concat=True):
    """ref: idconv.py:317-342 (same message/update as pyg GATConv, heads concat)."""
    n = h.size(0)
    ei, _ = U.remove_self_loops(edge_index)
    ei, _ = U.add_self_loops(ei, num_nodes=n)
    x_j = h.index_select(0, ei[0]).view(-1, heads, out_channels)
    x_i = h.index_select(0, ei[1]).view(-1, heads, out_channels)
    alpha = (torch.cat([x_i, x_j], dim=-1) * att).sum(dim=-1)
    alpha = F.leaky_relu(alpha, negative_slope)
    alpha = U.softmax(alpha, ei[1], n)
    out = U.propagate(ei, x_j * alpha.view(-1, heads, 1), n, 'add')
    out = out.view(-1, heads * out_channels) if concat else out.mean(dim=1)
    return out if bias is None else out + bias


def gatconv(x, edge_index, weight, att, bias=None, heads=1, negative_slope=0.2):
    c = weight.size(1) // heads
    return _gat_core(x @ weight, edge_index, att, heads, c, negative_slope, bias)


# ---- ID-GNN layers (ref: idconv.py) ---------------------------------------------------------------
def general_idconv(x, edge_index, ids, weight, weight_id, bias=None, aggr='add', normalize=False):
    """ref: idconv.py:62-97."""
    n = x.size(0)
    h = id_transform(x, ids, weight, weight_id)
    if normalize:
        ei, norm = gcn_norm_src(edge_index, n, x.dtype)
    else:
        ei, norm = edge_index, None
    out = _prop(ei, h, n, aggr, norm)
    return out if bias is None else out + bias


def gcn_idconv(x, edge_index, ids, weight, weight_id, bias=None):
    """ref: idconv.py:150-185."""
    n = x.size(0)
    h = id_transform(x, ids, weight, weight_id)
    ei, norm = gcn_norm_src(edge_index, n, x.dtype)
    out = _prop(ei, h, n, 'add', norm)
    return out if bias is None else out + bias


def sage_idconv(x, edge_index, ids, weight, weight_id, bias=None, concat=True):
    """ref: idconv.py:221-259."""
    n = x.size(0)
    ei = edge_index
    if not concat:
        ei, _ = U.add_remaining_self_loops(edge_index, None, 1, n)
    agg = _prop(ei, x, n, 'mean')
    if concat:
        agg = torch.cat([x, agg], dim=-1)
    out = id_transform(agg, ids, weight, weight_id)
    return out if bias is None else out + bias


def gat_idconv(x, edge_index, ids, weight, weight_id, att, bias=None, heads=1, negative_slope=0.2):
    """ref: idconv.py:299-342."""
    c = weight.size(1) // heads
    return _gat_core(id_transform(x, ids, weight, weight_id), edge_index, att, heads, c,
                     negative_slope, bias)


def gin_idconv(x, edge_index, ids, p, p_id, eps=0.0, gate=None, gate_id=None, tap=None):
    """ref: idconv.py:367-376; p / p_id = (w1, b1, w2, b2) of nn / nn_id."""
    ei, _ = U.remove_self_loops(edge_index)
    z = (1 + eps) * x + _prop(ei, x, x.size(0), 'add')
    out = _gin_mlp(z, p, gate, tap, 'pre')
    z_id = z.index_select(0, ids)
    out_id = _gin_mlp(z_id, p_id, gate_id, tap, 'pre_id')
    return out.index_add(0, ids, out_id)
