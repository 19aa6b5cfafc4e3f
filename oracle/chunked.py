"""Edge-chunked forward+backward steps of the built-in layers (TEST INFRASTRUCTURE ONLY — see oracle/__init__.py).

``oracle/layers.py`` restates the reference's op sequence (dense transform, index_select gather of ``x_j``, per-edge scale,
index_add_ scatter; ref: graphgym/models/layer.py:135-162 -> pyg.nn.*, graphgym/contrib/layer/idconv.py:89-92,177-180,317-342)
and lets torch autograd differentiate it, which materialises the ``[E, F]`` message tensor: 33 GB on the 62 M-edge
products-shaped graph.  SURVEY §8(d) prescribes edge chunking for that size.  The functions here run the SAME ops over
slices of the edge list and spell the backward out by hand — exactly the ops autograd would run (index_add_'s backward is
an index_select of the gradient, the scale's backward is the same scale, index_select's backward is an index_add_) — so
that no per-edge tensor outlives its chunk.  ``tests/test_oracle_golden.py`` pins them against ``oracle/layers.py`` +
autograd on small inputs.  They are the CPU arm of ``bench.py`` at full size (kind "port"), and they run wherever their
inputs live: in float64 on the GPU they are the reference of ``tests/test_fullsize_step_parity_gpu.py``.
"""
import torch
import torch.nn.functional as F

from . import layers as L
from . import pyg_utils as U


def _chunks(e, chunk):
    for s in range(0, e, chunk):
        yield s, min(e, s + chunk)


def _scatter_messages(out, h, src, tgt, w, chunk):
    """out[tgt_e] += w_e * h[src_e] over edge chunks (gather -> scale -> index_add_)."""
    for a, b in _chunks(src.numel(), chunk):
        m = h.index_select(0, src[a:b])
        if w is not None:
            m = m * w[a:b].view(-1, 1)
        out.index_add_(0, tgt[a:b], m)
    return out


def gcnconv_step(x, edge_index, weight, bias, gy, chunk=1 << 22):
    """-> (out, dx, dweight, dbias) of oracle.layers.gcnconv."""
    n = x.size(0)
    ei, norm = L.gcn_norm_tgt(edge_index, n, x.dtype)
    h = x @ weight
    out = _scatter_messages(torch.zeros_like(h), h, ei[0], ei[1], norm, chunk)
    if bias is not None:
        out += bias
    gh = _scatter_messages(torch.zeros_like(h), gy, ei[1], ei[0], norm, chunk)   # transposed graph
    return out, gh @ weight.t(), x.t() @ gh, (gy.sum(0) if bias is not None else None)


def sageconv_step(x, edge_index, w_l, b_l, w_r, gy, chunk=1 << 22):
    """-> (out, dx, dw_l, db_l, dw_r) of oracle.layers.sageconv (weights are nn.Linear [out, in])."""
    n = x.size(0)
    src, tgt = edge_index
    cnt = torch.zeros(n, dtype=x.dtype, device=x.device).index_add_(0, tgt, torch.ones(tgt.numel(), dtype=x.dtype,
                                                                             device=x.device)).clamp(min=1)
    mean = _scatter_messages(torch.zeros_like(x), x, src, tgt, None, chunk) / cnt.view(-1, 1)
    out = F.linear(mean, w_l, b_l) + F.linear(x, w_r)
    gmean = (gy @ w_l) / cnt.view(-1, 1)
    dx = _scatter_messages(gy @ w_r, gmean, tgt, src, None, chunk)
    return out, dx, gy.t() @ mean, (gy.sum(0) if b_l is not None else None), gy.t() @ x


def gatconv_step(x, edge_index, weight, att, bias, gy, negative_slope=0.2, chunk=1 << 22, return_alpha=False):
    """-> (out, dx, dweight, datt, dbias) of oracle.layers.gatconv with heads = 1; with ``return_alpha`` also alpha [E']
    over the edge list the layer aggregates (self loops removed, then one per node appended).  Per-edge SCALARS (logits,
    alpha) are kept whole ([E] floats); every [E, C] tensor is chunked.  The reference additionally materialises cat([x_i, x_j])
    [E, 2C] (idconv.py:323-326): this port is cheaper than the reference's own op sequence."""
    n, c = x.size(0), weight.size(1)
    ei, _ = U.remove_self_loops(edge_index)
    ei, _ = U.add_self_loops(ei, num_nodes=n)
    src, tgt = ei
    a_t, a_s = att.view(-1)[:c], att.view(-1)[c:]
    h = x @ weight
    s_t, s_s = h @ a_t, h @ a_s
    z = s_t[tgt] + s_s[src]
    lz = F.leaky_relu(z, negative_slope)
    alpha = U.softmax(lz, tgt, n)
    out = _scatter_messages(torch.zeros_like(h), h, src, tgt, alpha, chunk)
    if bias is not None:
        out += bias
    # backward
    dalpha = torch.empty_like(alpha)
    for a, b in _chunks(src.numel(), chunk):
        dalpha[a:b] = (gy.index_select(0, tgt[a:b]) * h.index_select(0, src[a:b])).sum(1)
    dot = torch.zeros(n, dtype=x.dtype, device=x.device).index_add_(0, tgt, alpha * dalpha)
    dlz = alpha * (dalpha - dot[tgt])
    dz = dlz * torch.where(z > 0, torch.ones_like(z), torch.full_like(z, negative_slope))
    ds_t = torch.zeros(n, dtype=x.dtype, device=x.device).index_add_(0, tgt, dz)
    ds_s = torch.zeros(n, dtype=x.dtype, device=x.device).index_add_(0, src, dz)
    dh = _scatter_messages(torch.zeros_like(h), gy, tgt, src, alpha, chunk)
    dh += ds_t.view(-1, 1) * a_t + ds_s.view(-1, 1) * a_s
    datt = torch.cat([h.t() @ ds_t, h.t() @ ds_s]).view_as(att)
    res = (out, dh @ weight.t(), x.t() @ dh, datt, (gy.sum(0) if bias is not None else None))
    return res + (alpha,) if return_alpha else res
