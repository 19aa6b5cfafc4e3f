"""Restated torch_geometric / torch_scatter helpers (PyG 1.x semantics; un-vendored upstream).

Call sites in the reference: idconv.py:5-10,52-56,140-144,232-233,302-304,327,370; identity.py:4-5.
"""
import math

import torch


def maybe_num_nodes(edge_index, num_nodes=None):
    return int(edge_index.max()) + 1 if num_nodes is None else int(num_nodes)


def scatter_add(src, index, dim=0, dim_size=None):
    """torch_scatter.scatter_add along dim 0."""
    assert dim == 0
    n = int(index.max()) + 1 if dim_size is None else int(dim_size)
    out = torch.zeros((n,) + tuple(src.shape[1:]), dtype=src.dtype, device=src.device)
    return out.index_add_(0, index, src)


def remove_self_loops(edge_index, edge_attr=None):
    mask = edge_index[0] != edge_index[1]
    return edge_index[:, mask], (None if edge_attr is None else edge_attr[mask])


def add_self_loops(edge_index, edge_weight=None, fill_value=1, num_nodes=None):
    n = maybe_num_nodes(edge_index, num_nodes)
    loop = torch.arange(n, dtype=torch.long, device=edge_index.device).unsqueeze(0).repeat(2, 1)
    if edge_weight is not None:
        edge_weight = torch.cat([edge_weight, edge_weight.new_full((n,), fill_value)])
    return torch.cat([edge_index, loop], dim=1), edge_weight


def add_remaining_self_loops(edge_index, edge_weight=None, fill_value=1, num_nodes=None):
    """Drop existing (i,i) edges, append one (i,i) per node at the end; an existing loop's weight is
    kept (the last one if several), otherwise ``fill_value``."""
    n = maybe_num_nodes(edge_index, num_nodes)
    row, col = edge_index
    mask = row != col
    loop = torch.arange(n, dtype=torch.long, device=edge_index.device).unsqueeze(0).repeat(2, 1)
    if edge_weight is not None:
        loop_weight = edge_weight.new_full((n,), fill_value)
        inv = ~mask
        for e in torch.nonzero(inv).flatten().tolist():  # ascending e => the last loop wins
            loop_weight[row[e]] = edge_weight[e]
        edge_weight = torch.cat([edge_weight[mask], loop_weight])
    return torch.cat([edge_index[:, mask], loop], dim=1), edge_weight


def softmax(src, index, num_nodes=None):
    """PyG 1.x ``softmax``: subtract the per-segment max, exp, divide by (segment sum + 1e-16)."""
    n = maybe_num_nodes(index.unsqueeze(0), num_nodes)
    shape = (n,) + tuple(src.shape[1:])
    mx = torch.full(shape, float('-inf'), dtype=src.dtype, device=src.device)
    mx = mx.scatter_reduce(0, index.view(-1, *[1] * (src.dim() - 1)).expand_as(src), src, 'amax',
                           include_self=True)
    out = (src - mx[index]).exp()
    den = torch.zeros(shape, dtype=src.dtype, device=src.device).index_add_(0, index, out)
    return out / (den[index] + 1e-16)


def propagate(edge_index, x_j_msg, num_nodes, aggr):
    """Scatter the per-edge messages to ``edge_index[1]`` (flow source_to_target)."""
    tgt = edge_index[1]
    out = torch.zeros((num_nodes,) + tuple(x_j_msg.shape[1:]), dtype=x_j_msg.dtype, device=x_j_msg.device)
    out = out.index_add_(0, tgt, x_j_msg)
    if aggr == 'mean':
        cnt = torch.zeros(num_nodes, dtype=x_j_msg.dtype, device=tgt.device).index_add_(
            0, tgt, torch.ones(tgt.numel(), dtype=x_j_msg.dtype, device=tgt.device))
        out = out / cnt.clamp(min=1).view(-1, *[1] * (out.dim() - 1))
    elif aggr != 'add':
        raise NotImplementedError(aggr)
    return out


def glorot(tensor):
    if tensor is not None:
        stdv = math.sqrt(6.0 / (tensor.size(-2) + tensor.size(-1)))
        tensor.data.uniform_(-stdv, stdv)


def zeros(tensor):
    if tensor is not None:
        tensor.data.fill_(0)


def reset(nn):
    def _reset(item):
        if hasattr(item, 'reset_parameters'):
            item.reset_parameters()

    if nn is not None:
        if hasattr(nn, 'children') and len(list(nn.children())) > 0:
            for item in nn.children():
                _reset(item)
        else:
            _reset(nn)
