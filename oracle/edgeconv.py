"""generaledgeconv (TEST INFRASTRUCTURE ONLY — see oracle/__init__.py).

ref: graphgym/contrib/layer/generalconv.py ``GeneralEdgeConvLayer``, a MessagePassing with flow source_to_target:
  message  m_e = linear_msg([x_j | a_e])          (cfg.gnn.msg_direction = 'single')
           m_e = linear_msg([x_i | x_j | a_e])    ('both'),  e = (j -> i), j = edge_index[0, e], i = edge_index[1, e]
  aggr     cfg.gnn.agg over the in-edges of i: add, mean (duplicates counted) or max (torch_scatter's scatter_max: 0 without
           in-edges, the gradient to the first in-edge reaching each column's maximum — ``max_agg.propagate``)
  update   + bias
  self     'add': + x;  'concat': + linear_self(x);  'none'.

  general_edge_conv        the per-edge concatenation and message in plain torch (autograd)
  general_edge_conv_step   the same step over edge chunks with the backward spelled out, for full size (no [E, F] tensor
                           outlives its chunk)
"""
import torch

from . import max_agg as M


def _split(w_msg, fin, msg_direction):
    """(W_i or None, W_j, W_a): the column blocks of linear_msg.weight [out, K]."""
    if msg_direction == 'both':
        return w_msg[:, :fin], w_msg[:, fin:2 * fin], w_msg[:, 2 * fin:]
    return None, w_msg[:, :fin], w_msg[:, fin:]


def general_edge_conv(x, edge_index, edge_feature, w_msg, w_self=None, bias=None, aggr='add', msg_direction='single',
                      self_msg='concat', arg=None):
    """The layer's forward with autograd.  ``w_msg`` = linear_msg.weight [out, K], ``w_self`` = linear_self.weight;
    ``arg``: the max aggregation's winning edge ids [N, out] (see ``max_agg.propagate``)."""
    n = x.size(0)
    src, tgt = edge_index
    parts = [x.index_select(0, src), edge_feature]
    if msg_direction == 'both':
        parts = [x.index_select(0, tgt)] + parts
    msg = torch.cat(parts, dim=1) @ w_msg.t()
    out = M.propagate(edge_index, msg, n, aggr, arg)
    if bias is not None:
        out = out + bias
    if self_msg == 'add':
        out = out + x
    elif self_msg == 'concat':
        out = out + x @ w_self.t()
    return out


def _chunks(e, chunk):
    for s in range(0, e, chunk):
        yield s, min(e, s + chunk)


def general_edge_conv_step(x, edge_index, edge_feature, w_msg, w_self, bias, gy, aggr, msg_direction, self_msg, arg=None,
                           chunk=1 << 22):
    """-> (out, dx, d edge_feature, dw_msg, dw_self, dbias, own_arg, gap) of ``general_edge_conv`` over edge chunks; runs
    wherever its inputs live (float64 on the GPU at full size).

    The message of edge e is h_j[j] + h_i[i] + a_e W_a^T with h = x W^T (the column blocks of W; the same product as the
    concatenation).  Max: ``own_arg`` = the first edge reaching each maximum (-1 = no in-edge); the gradients are taken
    under ``arg`` when given, else under ``own_arg``; ``gap`` = the maximum minus the message of the edge ``arg`` names
    (0 where the two agree).  own_arg and gap are None for add / mean."""
    n, fin = x.shape
    src, tgt = edge_index
    e = src.numel()
    w_i, w_j, w_a = _split(w_msg, fin, msg_direction)
    h_j = x @ w_j.t()
    h_i = x @ w_i.t() if w_i is not None else None
    f = h_j.size(1)

    def msg(a, b):
        m = h_j.index_select(0, src[a:b]) + edge_feature[a:b] @ w_a.t()
        return m if h_i is None else m + h_i.index_select(0, tgt[a:b])

    own = gap = None
    if aggr in ('add', 'mean'):
        out = torch.zeros_like(h_j)
        for a, b in _chunks(e, chunk):
            out.index_add_(0, tgt[a:b], msg(a, b))
        deg = torch.zeros(n, dtype=x.dtype, device=x.device).index_add_(0, tgt, torch.ones_like(tgt, dtype=x.dtype))
        scale = 1.0 / deg.clamp(min=1) if aggr == 'mean' else torch.ones_like(deg)
        out = out * scale.view(-1, 1)
        g_row = gy * scale.view(-1, 1)

        def dmsg(a, b):
            return g_row.index_select(0, tgt[a:b])
    elif aggr == 'max':
        idx = lambda a, b: tgt[a:b].view(-1, 1).expand(-1, f)
        mx = torch.full_like(h_j, float('-inf'))
        for a, b in _chunks(e, chunk):
            mx.scatter_reduce_(0, idx(a, b), msg(a, b), 'amax')
        own = torch.full((n, f), e, dtype=torch.long, device=x.device)
        for a, b in _chunks(e, chunk):
            eid = torch.arange(a, b, device=x.device).view(-1, 1).expand(-1, f)
            cand = torch.where(msg(a, b) == mx.index_select(0, tgt[a:b]), eid, torch.full_like(eid, e))
            own.scatter_reduce_(0, idx(a, b), cand, 'amin')
        own[own == e] = -1
        out = torch.where(own >= 0, mx, torch.zeros_like(mx))
        use = own if arg is None else arg
        chosen = torch.zeros_like(out)
        for a, b in _chunks(e, chunk):
            inside = (use >= a) & (use < b)
            got = msg(a, b).gather(0, (use - a).clamp(0, b - a - 1))
            chosen = torch.where(inside, got, chosen)
        gap = out - chosen

        def dmsg(a, b):
            eid = torch.arange(a, b, device=x.device).view(-1, 1)
            won = use.index_select(0, tgt[a:b]) == eid
            return torch.where(won, gy.index_select(0, tgt[a:b]), torch.zeros((), dtype=gy.dtype, device=gy.device))
    else:
        raise ValueError('aggr {!r}'.format(aggr))

    dh_j = torch.zeros_like(h_j)
    dh_i = torch.zeros_like(h_j) if h_i is not None else None
    da = torch.empty_like(edge_feature)
    dw_a = torch.zeros_like(w_a)
    for a, b in _chunks(e, chunk):
        dm = dmsg(a, b)
        dh_j.index_add_(0, src[a:b], dm)
        if dh_i is not None:
            dh_i.index_add_(0, tgt[a:b], dm)
        da[a:b] = dm @ w_a
        dw_a += dm.t() @ edge_feature[a:b]
    dx = dh_j @ w_j
    dws = [x.t() @ dh_j]
    if dh_i is not None:
        dx = dx + dh_i @ w_i
        dws = [x.t() @ dh_i] + dws
    dw_msg = torch.cat([w.t() for w in dws] + [dw_a], dim=1)
    dw_self = None
    if bias is not None:
        out = out + bias
    if self_msg == 'add':
        out = out + x
        dx = dx + gy
    elif self_msg == 'concat':
        out = out + x @ w_self.t()
        dx = dx + gy @ w_self
        dw_self = gy.t() @ x
    return out, dx, da, dw_msg, dw_self, (gy.sum(0) if bias is not None else None), own, gap


def general_edge_conv_loop(x, edge_index, edge_feature, w_msg, w_self, bias, aggr, msg_direction, self_msg):
    """The forward edge by edge in Python (the definition, for tiny graphs): every message built from its own
    concatenation, each target's messages reduced in edge order."""
    n = x.size(0)
    src, tgt = edge_index.tolist()
    msgs = [[] for _ in range(n)]
    for e, (j, i) in enumerate(zip(src, tgt)):
        parts = [x[j], edge_feature[e]]
        if msg_direction == 'both':
            parts = [x[i]] + parts
        msgs[i].append(w_msg @ torch.cat(parts))
    rows = []
    for i in range(n):
        if not msgs[i]:
            r = torch.zeros(w_msg.size(0), dtype=x.dtype)
        elif aggr == 'max':
            r = torch.stack(msgs[i]).max(0).values
        else:
            r = torch.stack(msgs[i]).sum(0)
            if aggr == 'mean':
                r = r / len(msgs[i])
        if bias is not None:
            r = r + bias
        if self_msg == 'add':
            r = r + x[i]
        elif self_msg == 'concat':
            r = r + w_self @ x[i]
        rows.append(r)
    return torch.stack(rows)

