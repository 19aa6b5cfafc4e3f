"""The design-space attention layers gaddconv / gmulconv with every ``cfg.gnn.agg`` (TEST INFRASTRUCTURE ONLY — see
oracle/__init__.py).

ref: graphgym/contrib/layer/attconv.py — GeneralAddAttConvLayer (h = x W^T; logits leaky_relu_{0.2}(att . [h_i || h_j])
per head, PyG 1.x softmax over the edges sharing a target; message alpha_e[head(c)] h_j[c]) and GeneralMulAttConvLayer
(one head; logits (<h_i, h_j> + sum(bias_att)) / sqrt(out); message alpha_e h_j).  The edge list is used as given.  The
messages are reduced with ``max_agg.propagate`` ([E, H*C]): 'add' / 'mean' as ``pyg_utils.propagate``, 'max' as
torch_scatter's scatter_max (gradient to the first edge reaching the maximum, or to the edges an explicit ``arg`` names).

  gadd_conv / gmul_conv     the layers (plain torch, autograd)
  gadd_conv_step            gaddconv's forward + backward over edge chunks with the backward spelled out, for full size
"""
import math

import torch
import torch.nn.functional as F

from . import max_agg as M
from . import pyg_utils as U


def gadd_conv(x, edge_index, weight, att, bias=None, heads=1, aggr='add', arg=None, negative_slope=0.2):
    """``weight`` [out, in] (nn.Linear), ``att`` [1, heads, 2C]; ``arg``: max winners as edge ids [n, out]."""
    n = x.size(0)
    h = x @ weight.t()
    c = h.size(1) // heads
    hh = h.view(n, heads, c)
    src, tgt = edge_index
    a = att.view(heads, 2 * c)
    z = (hh.index_select(0, tgt) * a[:, :c]).sum(-1) + (hh.index_select(0, src) * a[:, c:]).sum(-1)   # [E, H]
    alpha = U.softmax(F.leaky_relu(z, negative_slope), tgt, n)
    msg = (alpha.unsqueeze(-1) * hh.index_select(0, src)).reshape(-1, heads * c)
    out = M.propagate(edge_index, msg, n, aggr, arg)
    return out if bias is None else out + bias


def gmul_conv(x, edge_index, weight, bias=None, bias_att=None, aggr='add', arg=None):
    """``weight`` [out, in]; ``bias_att`` [out] (cancels in the softmax)."""
    n = x.size(0)
    h = x @ weight.t()
    src, tgt = edge_index
    z = (h.index_select(0, tgt) * h.index_select(0, src)).sum(-1)
    if bias_att is not None:
        z = z + bias_att.sum()
    alpha = U.softmax(z / math.sqrt(h.size(1)), tgt, n)
    out = M.propagate(edge_index, alpha.view(-1, 1) * h.index_select(0, src), n, aggr, arg)
    return out if bias is None else out + bias


def _chunks(e, chunk):
    for s in range(0, e, chunk):
        yield s, min(e, s + chunk)


def gadd_conv_step(x, edge_index, weight, att, bias, gy, aggr, heads=1, arg=None, gate=None, negative_slope=0.2,
                   chunk=1 << 22):
    """-> (out, dx, dweight, datt, dbias, own_arg, gap) of ``gadd_conv``, over edge chunks: per-edge [E, H] tensors (logits,
    alpha) are kept whole, every [E, F] tensor lives for one chunk.  Runs wherever its inputs live.

    'max': the maximum is scatter_reduce('amax') over the chunks, ``own_arg`` the first edge reaching it (edge ids, -1 = no
    in-edge); the gradients are taken under ``arg`` when given, else under ``own_arg``; ``gap`` = the maximum minus the
    message of the edge ``arg`` names ([n, F], 0 where the two agree).  'add' / 'mean': ``own_arg`` and ``gap`` are None.
    ``gate`` ([E, H] bool): the leaky-ReLU branch each logit takes in the backward (True = slope 1) instead of z > 0 — the
    branches another implementation took, for logits within its rounding of zero."""
    n = x.size(0)
    src, tgt = edge_index
    e = src.numel()
    h = x @ weight.t()
    f = h.size(1)
    c = f // heads
    hh = h.view(n, heads, c)
    a = att.view(heads, 2 * c)
    a_t, a_s = a[:, :c], a[:, c:]
    s_t, s_s = (hh * a_t).sum(-1), (hh * a_s).sum(-1)                  # [n, H]
    z = s_t.index_select(0, tgt) + s_s.index_select(0, src)              # [E, H]
    alpha = U.softmax(F.leaky_relu(z, negative_slope), tgt, n)
    head = torch.arange(f, device=h.device) // c

    def msg(lo, hi):
        return (alpha[lo:hi].unsqueeze(-1) * hh.index_select(0, src[lo:hi])).reshape(-1, f)

    own = gap = None
    dalpha = torch.zeros_like(alpha)
    dh = torch.zeros_like(h)
    if aggr == 'max':
        mx = torch.full_like(h, float('-inf'))
        for lo, hi in _chunks(e, chunk):
            mx.scatter_reduce_(0, tgt[lo:hi].view(-1, 1).expand(-1, f), msg(lo, hi), 'amax')
        own = torch.full((n, f), e, dtype=torch.long, device=h.device)
        for lo, hi in _chunks(e, chunk):
            eid = torch.arange(lo, hi, device=h.device).view(-1, 1).expand(-1, f)
            cand = torch.where(msg(lo, hi) == mx.index_select(0, tgt[lo:hi]), eid, torch.full_like(eid, e))
            own.scatter_reduce_(0, tgt[lo:hi].view(-1, 1).expand(-1, f), cand, 'amin')
        own[own == e] = -1
        out = torch.where(own >= 0, mx, torch.zeros_like(mx))
        use = own if arg is None else arg
        ok = use >= 0
        win = use.clamp(min=0)
        a_win = alpha[win, head.view(1, -1).expand(n, -1)] * ok                       # [n, F]
        h_win = h.gather(0, src[win])
        gap = out - a_win * h_win
        dh.view(-1).index_add_(0, (src[win] * f + torch.arange(f, device=h.device)).view(-1), (a_win * gy).view(-1))
        dalpha.view(-1).index_add_(0, (win * heads + head).view(-1), (gy * h_win * ok).view(-1))
    else:
        out = torch.zeros_like(h)
        for lo, hi in _chunks(e, chunk):
            out.index_add_(0, tgt[lo:hi], msg(lo, hi))
        g = gy
        if aggr == 'mean':
            cnt = torch.zeros(n, dtype=h.dtype, device=h.device).index_add_(0, tgt, torch.ones_like(tgt, dtype=h.dtype))
            inv = 1.0 / cnt.clamp(min=1)
            out *= inv.view(-1, 1)
            g = gy * inv.view(-1, 1)
        for lo, hi in _chunks(e, chunk):
            g_e = g.index_select(0, tgt[lo:hi]).view(-1, heads, c)
            h_e = hh.index_select(0, src[lo:hi])
            dalpha[lo:hi] = (g_e * h_e).sum(-1)
            dh.index_add_(0, src[lo:hi], (alpha[lo:hi].unsqueeze(-1) * g_e).reshape(-1, f))
    if bias is not None:
        out = out + bias
    # softmax and leaky-ReLU backward on the [E, H] logits
    dot = torch.zeros_like(s_t).index_add_(0, tgt, alpha * dalpha)
    pos = z > 0 if gate is None else gate
    dz = alpha * (dalpha - dot.index_select(0, tgt)) * torch.where(pos, torch.ones_like(z), torch.full_like(z, negative_slope))
    ds_t = torch.zeros_like(s_t).index_add_(0, tgt, dz)
    ds_s = torch.zeros_like(s_s).index_add_(0, src, dz)
    dh += (ds_t.unsqueeze(-1) * a_t + ds_s.unsqueeze(-1) * a_s).reshape(n, f)
    datt = torch.cat([(ds_t.unsqueeze(-1) * hh).sum(0), (ds_s.unsqueeze(-1) * hh).sum(0)], dim=1).view_as(att)
    dbias = gy.sum(0) if bias is not None else None
    return out, dh @ weight, dh.t() @ x, datt, dbias, own, gap
