"""Max aggregation of the reference's message passing (TEST INFRASTRUCTURE ONLY — see oracle/__init__.py).

``MessagePassing(aggr='max')`` reduces with torch_scatter's ``scatter_max`` (ref: graphgym/contrib/layer/generalconv.py:12-113
with ``cfg.gnn.agg = 'max'``): per target and column the largest message, 0 for a target without in-edges, and the
gradient to one winning edge — the FIRST edge in edge order that reaches the maximum (torch_scatter's CPU kernel: a strict
`>` scan; its CUDA kernel picks an arbitrary tied edge).  ``torch.scatter_reduce('amax')``'s own backward splits a tie's
gradient evenly, so it is used for the value only: the winner is the smallest edge id among the edges whose message equals
the maximum, and the output is the winner's message gathered, so that autograd sends the gradient to the winner alone.
An explicit ``arg`` (edge ids) overrides the winner, so that gradients can be compared under the choice another
implementation made.

  scatter_argmax / gather_max / propagate   the aggregation on [E, F] messages (plain torch, autograd)
  general_conv                              generalconv with the ops of oracle.layers (autograd)
  general_conv_max_step                     the same step over edge chunks with the backward spelled out, for full size
"""
import torch

from . import layers as L
from . import pyg_utils as U


def scatter_argmax(msg, index, num_nodes):
    """[num_nodes, F] edge ids: per target and column, the FIRST edge (in edge order) whose message equals the maximum;
    -1 for a target without edges.  ``msg``: [E, F]."""
    msg = msg.detach()
    idx = index.view(-1, 1).expand_as(msg)
    shape = (num_nodes, msg.size(1))
    mx = torch.full(shape, float('-inf'), dtype=msg.dtype, device=msg.device)
    mx = mx.scatter_reduce(0, idx, msg, 'amax', include_self=True)
    e = msg.size(0)
    eid = torch.arange(e, device=msg.device).view(-1, 1).expand_as(msg)
    cand = torch.where(msg == mx[index], eid, torch.full_like(eid, e))
    arg = torch.full(shape, e, dtype=torch.long, device=msg.device).scatter_reduce(0, idx, cand, 'amin', include_self=True)
    return torch.where(arg == e, torch.full_like(arg, -1), arg)


def gather_max(msg, arg):
    """out[i,c] = msg[arg[i,c], c] (0 where arg = -1): autograd sends each gradient to the one winning edge."""
    got = msg.gather(0, arg.clamp(min=0))
    return torch.where(arg >= 0, got, torch.zeros_like(got))


def propagate(edge_index, x_j_msg, num_nodes, aggr, arg=None):
    """``pyg_utils.propagate`` with ``aggr='max'`` added (2-D messages): the maximum over the in-edges, 0 without
    in-edges, the gradient to the winner (``scatter_argmax``, or ``arg`` [num_nodes, F] edge ids when given)."""
    if aggr != 'max':
        return U.propagate(edge_index, x_j_msg, num_nodes, aggr)
    if arg is None:
        arg = scatter_argmax(x_j_msg, edge_index[1], num_nodes)
    return gather_max(x_j_msg, arg)


def general_conv(x, edge_index, weight, weight_self=None, bias=None, aggr='add', normalize=False, self_msg='concat',
                 arg=None):
    """ref: graphgym/contrib/layer/generalconv.py:12-113 — h = x W; with ``normalize`` the GCN norm over edge_index[0]
    after remaining self loops (``layers.gcn_norm_src``); aggregate with ``aggr``; + h ('add') or + x W_self ('concat');
    + bias.  ``arg``: the max aggregation's winning edges (ids into the edited edge list), see ``propagate``."""
    n = x.size(0)
    h = x @ weight
    if normalize:
        ei, norm = L.gcn_norm_src(edge_index, n, x.dtype)
    else:
        ei, norm = edge_index, None
    x_j = h.index_select(0, ei[0])
    if norm is not None:
        x_j = norm.view(-1, 1) * x_j
    out = propagate(ei, x_j, n, aggr, arg)
    if self_msg == 'add':
        out = out + h
    elif self_msg == 'concat':
        out = out + x @ weight_self
    return out if bias is None else out + bias


def _chunks(e, chunk):
    for s in range(0, e, chunk):
        yield s, min(e, s + chunk)


def general_conv_max_step(x, edge_index, weight, weight_self, bias, gy, normalize, self_msg, arg=None, chunk=1 << 22):
    """-> (out, dx, dweight, dweight_self, dbias, own_arg, gap) of ``general_conv`` with aggr='max', over edge chunks (no
    [E, F] tensor outlives its chunk; runs wherever its inputs live, in float64 on the GPU at full size).

    The max runs as scatter_reduce('amax') over edge chunks, the first edge reaching it as scatter_reduce('amin') of the
    edge ids whose message equals it (``own_arg``, ids into the edited edge list, -1 = no in-edge).  The gradients are
    taken under ``arg`` when given (the winners another implementation chose), else under ``own_arg``.  ``gap`` = the
    maximum minus the message of the edge ``arg`` names ([n, F], 0 where the two choices agree): how far a different
    choice is from a tie."""
    n = x.size(0)
    if normalize:
        ei, norm = L.gcn_norm_src(edge_index, n, x.dtype)
    else:
        ei, norm = edge_index, None
    src, tgt = ei
    h = x @ weight
    f, e = h.size(1), src.numel()

    def msg(a, b):
        m = h.index_select(0, src[a:b])
        return m if norm is None else m * norm[a:b].view(-1, 1)

    mx = torch.full_like(h, float('-inf'))
    for a, b in _chunks(e, chunk):
        mx.scatter_reduce_(0, tgt[a:b].view(-1, 1).expand(-1, f), msg(a, b), 'amax')
    own = torch.full((n, f), e, dtype=torch.long, device=h.device)
    for a, b in _chunks(e, chunk):
        m = msg(a, b)
        eid = torch.arange(a, b, device=h.device).view(-1, 1).expand(-1, f)
        cand = torch.where(m == mx.index_select(0, tgt[a:b]), eid, torch.full_like(eid, e))
        own.scatter_reduce_(0, tgt[a:b].view(-1, 1).expand(-1, f), cand, 'amin')
    own[own == e] = -1
    out = torch.where(own >= 0, mx, torch.zeros_like(mx))
    use = own if arg is None else arg
    ok = use >= 0
    win = use.clamp(min=0)
    scale = ok.to(h.dtype) if norm is None else norm[win] * ok
    gap = out - h.gather(0, src[win]) * scale
    dh = torch.zeros_like(h).scatter_add_(0, src[win], gy * scale)
    dx_extra, dws = None, None
    if self_msg == 'add':
        out = out + h
        dh = dh + gy
    elif self_msg == 'concat':
        out = out + x @ weight_self
        dws = x.t() @ gy
        dx_extra = gy @ weight_self.t()
    if bias is not None:
        out = out + bias
    dx = dh @ weight.t()
    if dx_extra is not None:
        dx = dx + dx_extra
    return out, dx, x.t() @ dh, dws, (gy.sum(0) if bias is not None else None), own, gap
