"""Differentiable building blocks of the layers: each one is a ``torch.autograd.Function`` whose
forward AND backward are ``gg_*`` kernels (no torch math on the path).

  aggregate    CSR SpMM forward, CSC SpMM backward            (SURVEY §8a row 4); max: arg-max forward, masked CSC sum
  seg_linear   multi-segment dense transform with ID weights  (SURVEY §8a row 9)
  gather_rows / scatter_add_rows   the M-row ID branch of GIN-ID (ref: idconv.py:372-375)
"""
import math

import torch

from . import ops


class _Aggregate(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, layout, kind, self_scale, bias, half, residual=None):
        w_fwd, _ = layout.weights(kind)
        reduce = ops.MEAN if kind.endswith("mean") else ops.SUM
        x = x.contiguous()
        gathered = ops.cast_bf16(x) if half else x        # 1e-2 mode: the gathered operand in bf16, fp32 arithmetic
        if residual is not None:      # out = A x + residual (+ bias): the residual rides in the epilogue's self term
            if self_scale != 0.0:
                raise ValueError("aggregate: residual excludes self_scale")
            out = ops.spmm(layout.csr, gathered, w_fwd, reduce, residual.contiguous(), 1.0, bias)
        else:
            out = ops.spmm(layout.csr, gathered, w_fwd, reduce, x if self_scale != 0.0 else None, self_scale, bias)
        ctx.layout, ctx.kind, ctx.self_scale, ctx.half = layout, kind, self_scale, half
        ctx.has_bias, ctx.has_residual = bias is not None, residual is not None
        return out

    @staticmethod
    def backward(ctx, g):
        g = g.contiguous()
        gx = gb = None
        if ctx.needs_input_grad[0]:
            _, w_bwd = ctx.layout.weights(ctx.kind)
            # d/dx = A^T g (+ self_scale * g): the same kernel on the transposed layout
            gathered = ops.cast_bf16(g) if ctx.half else g
            gx = ops.spmm(ctx.layout.csc, gathered, w_bwd, ops.SUM, g if ctx.self_scale != 0.0 else None,
                          ctx.self_scale, None)
        if ctx.has_bias and ctx.needs_input_grad[4]:
            gb = ops.colsum(g)
        return gx, None, None, None, gb, None, (g if ctx.has_residual else None)


class _AggregateMax(torch.autograd.Function):
    """out[i] = max_{j->i} w_ji x[j] (0 without in-edges) + self_scale * x[i] + residual[i] + bias; the gradient of the
    max goes to the first in-edge (in edge order) that reaches it, per column."""

    @staticmethod
    def forward(ctx, x, layout, kind, self_scale, bias, residual=None):
        w_fwd, _ = layout.weights(kind)
        x = x.contiguous()
        if residual is not None:
            if self_scale != 0.0:
                raise ValueError("aggregate: residual excludes self_scale")
            out, arg = ops.spmm_max(layout.csr, x, w_fwd, residual.contiguous(), 1.0, bias)
        else:
            out, arg = ops.spmm_max(layout.csr, x, w_fwd, x if self_scale != 0.0 else None, self_scale, bias)
        ctx.layout, ctx.kind, ctx.self_scale = layout, kind, self_scale
        ctx.has_bias, ctx.has_residual = bias is not None, residual is not None
        ctx.save_for_backward(arg)
        return out

    @staticmethod
    def backward(ctx, g):
        g = g.contiguous()
        gx = gb = None
        if ctx.needs_input_grad[0]:
            (arg,) = ctx.saved_tensors
            _, w_bwd = ctx.layout.weights(ctx.kind)
            gx = ops.spmm_max_bwd(ctx.layout.csc, ctx.layout.csc2csr, g, arg, w_bwd, ctx.self_scale)
        if ctx.has_bias and ctx.needs_input_grad[4]:
            gb = ops.colsum(g)
        return gx, None, None, None, gb, (g if ctx.has_residual else None)


def aggregate(x, layout, kind="sum", self_scale=0.0, bias=None, residual=None):
    """out[i] = reduce_{j->i} w_ji x[j] + self_scale * x[i] + residual[i] + bias.  ``cfg.b200.gather_dtype = 'bf16'``
    stores the gathered operand in bf16 (forward and backward) when the width allows it (f % 8 == 0, f <= 256).
    Kinds ending in 'max' reduce with a max (fp32 only)."""
    from .config import cfg
    if kind.endswith("max"):
        if cfg.b200.gather_dtype == "bf16":
            raise NotImplementedError("cfg.b200.gather_dtype = 'bf16' has no max aggregation (kind {!r})".format(kind))
        return _AggregateMax.apply(x, layout, kind, float(self_scale), bias, residual)
    half = cfg.b200.gather_dtype == "bf16" and ops.bf16_gather_ok(x.size(1))
    return _Aggregate.apply(x, layout, kind, float(self_scale), bias, half, residual)


class _EdgeAggregate(torch.autograd.Function):
    """out[i] = A h_j + r_i h_i + (S a)[i] W_a^T (+ residual[i] + bias): the add / mean aggregation of the messages
    h_j[j] (+ h_i[i]) + a_e W_a^T, which is linear, so no per-edge message is formed.  A = the sum or mean over the
    in-edges, S a = the per-target sum or mean of the edge-feature rows, r_i = indeg(i) (add) or [indeg(i) > 0] (mean)."""

    @staticmethod
    def forward(ctx, h_j, h_i, a, w_a, layout, kind, bias, residual):
        csr = layout.csr
        mean = kind == "mean"
        sa = ops.edge_row_reduce(csr, a, mean)
        t = ops.id_gemm([(sa, w_a, None)], csr.num_nodes, w_a.size(0), b_trans=True)       # (S a) W_a^T
        w_fwd, _ = layout.weights(kind)
        out = ops.spmm(csr, h_j.contiguous(), w_fwd, ops.MEAN if mean else ops.SUM, t, 1.0, bias)
        if h_i is not None or residual is not None:
            ops.edge_rows_self(csr, h_i, y=out, z=residual, mean=mean)
        ctx.layout, ctx.kind = layout, kind
        ctx.has_hi, ctx.has_bias, ctx.has_residual = h_i is not None, bias is not None, residual is not None
        ctx.save_for_backward(sa, w_a)
        return out

    @staticmethod
    def backward(ctx, g):
        sa, w_a = ctx.saved_tensors
        g = g.contiguous()
        lay = ctx.layout
        csr = lay.csr
        mean = ctx.kind == "mean"
        ghj = ghi = ga = gw = gb = None
        if ctx.needs_input_grad[0]:
            _, w_bwd = lay.weights(ctx.kind)
            ghj = ops.spmm(lay.csc, g, w_bwd, ops.SUM, None, 0.0, None)
        if ctx.has_hi and ctx.needs_input_grad[1]:
            ghi = ops.edge_rows_self(csr, g, mean=mean)
        if ctx.needs_input_grad[2]:
            # d a_e = (g W_a)[target(e)] (/ indeg for the mean), in edge order
            gwa = ops.id_gemm([(g, w_a, None)], csr.num_nodes, w_a.size(1))
            if mean:
                ops.rows_epilogue(gwa, csr, out=gwa)
            ga = ops.gather_rows(gwa, lay.edge_index[1])
        if ctx.needs_input_grad[3]:
            gw = ops.gemm_tn(g, sa)
        if ctx.has_bias and ctx.needs_input_grad[6]:
            gb = ops.colsum(g)
        return ghj, ghi, ga, gw, None, None, gb, (g if ctx.has_residual else None)


class _EdgeAggregateMax(torch.autograd.Function):
    """out[i,c] = max_{e = (j -> i)} h_j[j,c] (+ h_i[i,c]) + a_e . W_a[c] (0 without in-edges) + residual[i,c] + bias[c];
    the gradient goes to the first in-edge (in edge order) that reaches the maximum, per column.  The edge term is formed
    per edge inside the reduction (``ops.edge_max``) and never stored."""

    @staticmethod
    def forward(ctx, h_j, h_i, a, w_a, layout, bias, residual):
        out, arg = ops.edge_max(layout.csr, h_j, h_i, a, w_a, residual, 1.0 if residual is not None else 0.0, bias)
        ctx.layout = layout
        ctx.has_hi, ctx.has_bias, ctx.has_residual = h_i is not None, bias is not None, residual is not None
        ctx.save_for_backward(a, w_a, arg)
        return out

    @staticmethod
    def backward(ctx, g):
        a, w_a, arg = ctx.saved_tensors
        g = g.contiguous()
        lay = ctx.layout
        ghj = ghi = ga = gw = gb = None
        if ctx.needs_input_grad[0]:
            ghj = ops.spmm_max_bwd(lay.csc, lay.csc2csr, g, arg)
        if ctx.has_hi and ctx.needs_input_grad[1]:
            ghi = ops.max_mask(g, arg)
        if ctx.needs_input_grad[2]:
            ga = ops.edge_max_winner(lay.csr, arg, g, w_a)
        if ctx.needs_input_grad[3]:
            gw = ops.edge_max_wgrad(lay.csr, arg, g, a)
        if ctx.has_bias and ctx.needs_input_grad[5]:
            gb = ops.colsum(g)
        return ghj, ghi, ga, gw, None, gb, (g if ctx.has_residual else None)


def edge_aggregate(h_j, h_i, edge_feature, w_a, layout, agg, bias=None, residual=None):
    """Aggregation of the edge-feature messages m_e = h_j[j] (+ h_i[i]) + edge_feature[e] w_a^T over the in-edges
    e = (j -> i) of ``layout`` (edge order = the layout's edge_index), + residual + bias.  ``agg``: 'add' | 'mean' | 'max'
    (max: 0 for a row without in-edges, the gradient to the first in-edge reaching each column's maximum).  ``h_i`` may
    be None; ``w_a``: [f, edge_dim] (a column slice of nn.Linear's weight).  fp32 only."""
    from .config import cfg
    if cfg.b200.gather_dtype == "bf16":
        raise NotImplementedError("cfg.b200.gather_dtype = 'bf16' has no edge-feature aggregation")
    if agg == "max":
        return _EdgeAggregateMax.apply(h_j, h_i, edge_feature, w_a, layout, bias, residual)
    if agg not in ("add", "mean"):
        raise NotImplementedError("edge_aggregate: agg {!r}".format(agg))
    return _EdgeAggregate.apply(h_j, h_i, edge_feature, w_a, layout, "mean" if agg == "mean" else "sum", bias, residual)


class _SplineAggregate(torch.autograd.Function):
    """out[i] = mean over e = (j -> i) of (c0_e x_j W0 + c1_e x_j W1) + x_i root + bias, (c0_e, c1_e) the degree-1 open
    B-spline coefficients of u_e (kernel size 2).  No per-edge message is formed; two factorisations:
      aggregate first  [P0 | P1] = spread(x) on the CSR, out = [P0 | P1 | x] [W0; W1; root] + bias (one GEMM);
                       dX = blend([dP0 | dP1] = g [W0 | W1]^T) on the CSC + g root^T, dW_k = P_k^T g
      transform first  H = x [W0 | W1], out = blend(H) on the CSR + x root + bias;
                       [dH0 | dH1] = spread(g) on the CSC, dX = [dH0 | dH1] [W0 | W1]^T + g root^T, dW_k = x^T dH_k
    On the CSC the slots carry 1/indeg(target).  d u (only when asked for) comes from a warp-per-row pass over the CSR."""

    @staticmethod
    def forward(ctx, x, u, weight, root, bias, layout, aggregate_first):
        csr = layout.csr
        x = x.contiguous()
        uf = u.reshape(-1)
        n, (fin, fout) = x.size(0), root.shape
        if aggregate_first:
            t = ops.spline_spread(csr, x, uf, mean=True)                                    # [P0 | P1]
            w01 = weight.reshape(2 * fin, fout)                                              # [W0; W1]
            out = ops.id_gemm([(t, w01, None), (x, root, None)], n, fout, bias=bias)
        else:
            w01 = torch.cat([weight[0], weight[1]], dim=1)                                   # [W0 | W1]
            t = ops.id_gemm([(x, w01, None)], n, 2 * fout)                                   # [H0 | H1]
            r = ops.id_gemm([(x, root, None)], n, fout)
            out = ops.spline_blend(csr, t, uf, mean=True, residual=r, bias=bias)
        ctx.layout, ctx.aggregate_first, ctx.u_shape = layout, aggregate_first, u.shape
        ctx.has_bias = bias is not None
        ctx.save_for_backward(x, uf, w01, root, t)
        return out

    @staticmethod
    def backward(ctx, g):
        x, uf, w01, root, t = ctx.saved_tensors
        g = g.contiguous()
        lay = ctx.layout
        n, (fin, fout) = x.size(0), root.shape
        _, w_csc = lay.weights("mean")                                                       # 1/indeg(target) per CSC slot
        gx = gu = gw = groot = gb = None
        need_x, need_u, need_w = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.needs_input_grad[2]
        if ctx.aggregate_first:
            if need_x or need_u:
                dp = ops.id_gemm([(g, w01, None)], n, 2 * fin, b_trans=True)                 # [dP0 | dP1]
                if need_x:
                    gx = ops.spline_blend(lay.csc, dp, uf, w_csc,
                                          residual=ops.id_gemm([(g, root, None)], n, fin, b_trans=True))
                if need_u:
                    gu = ops.spline_du(lay.csr, uf, dp, fin, x, 0, fin)
            if need_w:
                gw = ops.gemm_tn(t, g).view(2, fin, fout)
        else:
            if need_x or need_w:
                dh = ops.spline_spread(lay.csc, g, uf, w_csc)                                # [dH0 | dH1]
                if need_x:
                    gx = ops.id_gemm([(dh, w01, None), (g, root, None)], n, fin, b_trans=True)
                if need_w:
                    dw = ops.gemm_tn(x, dh)
                    gw = torch.stack([dw[:, :fout], dw[:, fout:]])
            if need_u:
                gu = ops.spline_du(lay.csr, uf, g, 0, t, fout, fout)
        if ctx.needs_input_grad[3]:
            groot = ops.gemm_tn(x, g)
        if ctx.has_bias and ctx.needs_input_grad[4]:
            gb = ops.colsum(g)
        if gu is not None:
            gu = gu.view(ctx.u_shape)
        return gx, gu, gw, groot, gb, None, None


def spline_aggregate(x, pseudo, weight, root, bias, layout, aggregate_first):
    """SplineConv's mean aggregation with the root weight (dim 1, kernel size 2, degree 1, open spline): ``pseudo`` the
    [E] or [E, 1] float32 pseudo-coordinates in the edge order of ``layout``, ``weight`` [2, in, out], ``root`` [in, out].
    ``aggregate_first`` picks the factorisation (the narrower side is gathered: in <= out aggregates first)."""
    return _SplineAggregate.apply(x, pseudo, weight, root, bias, layout, bool(aggregate_first))


class _SegLinear(torch.autograd.Function):
    """out = act( sum_g diag(c_g) X_g W_g + bias ).

    ``spec``: tuple of (input index, weight index, use_id) per K-segment; inputs / weights are the
    flattened tensor arguments.  ``w_trans``: weights are [out,in] (nn.Linear) instead of [in,out].
    ``w_rows``: per segment, optional (start, stop) row slice of the weight's ``in`` dimension.
    """

    @staticmethod
    def forward(ctx, spec, w_rows, w_trans, act, id_info, n_inputs, bias, *tensors):
        xs = [t.contiguous() for t in tensors[:n_inputs]]
        ws = list(tensors[n_inputs:])
        n = xs[0].size(0)
        segs = []
        for (xi, wi, use_id), rows in zip(spec, w_rows):
            w = _w_slice(ws[wi], rows, w_trans)
            segs.append((xs[xi], w, id_info.count if use_id else None))
        f = ws[0].size(0) if w_trans else ws[0].size(1)
        out = ops.id_gemm(segs, n, f, b_trans=w_trans, bias=bias, act=act)
        ctx.spec, ctx.w_rows, ctx.w_trans, ctx.act = spec, w_rows, w_trans, act
        ctx.id_info, ctx.n_inputs = id_info, n_inputs
        ctx.has_bias = bias is not None
        ctx.save_for_backward(out if act == ops.ACT_RELU else None, *xs, *ws)
        return out

    @staticmethod
    def backward(ctx, g):
        saved = ctx.saved_tensors
        out, xs, ws = saved[0], saved[1:1 + ctx.n_inputs], saved[1 + ctx.n_inputs:]
        g = g.contiguous()
        if ctx.act == ops.ACT_RELU:
            g = ops.relu_grad(g, out)
        n = g.size(0)
        id_info = ctx.id_info
        grads_x = [None] * len(xs)
        grads_w = [None] * len(ws)
        # dX_i = sum over the segments that read X_i of diag(c) g W^T
        for xi in range(len(xs)):
            if not ctx.needs_input_grad[7 + xi]:
                continue
            segs = []
            for (sxi, wi, use_id), rows in zip(ctx.spec, ctx.w_rows):
                if sxi == xi:
                    segs.append((g, _w_slice(ws[wi], rows, ctx.w_trans),
                                 id_info.count if use_id else None))
            # forward B was [K,F] (or [F,K] transposed); the backward contracts over F
            grads_x[xi] = ops.id_gemm(segs, n, xs[xi].size(1), b_trans=not ctx.w_trans)
        # dW = X^T g over all rows, or over the centre rows for an ID weight
        for wi in range(len(ws)):
            if not ctx.needs_input_grad[7 + len(xs) + wi]:
                continue
            parts = []
            for (sxi, swi, use_id), rows in zip(ctx.spec, ctx.w_rows):
                if swi != wi:
                    continue
                ridx = id_info.ids if use_id else None
                if ctx.w_trans:
                    gw = ops.gemm_tn(g, xs[sxi], ridx)  # [out, in_slice]
                else:
                    gw = ops.gemm_tn(xs[sxi], g, ridx)  # [in_slice, out]
                parts.append((rows, gw))
            grads_w[wi] = _assemble(parts, ws[wi], ctx.w_trans)
        gb = ops.colsum(g) if (ctx.has_bias and ctx.needs_input_grad[6]) else None
        return (None, None, None, None, None, None, gb, *grads_x, *grads_w)


def _w_slice(w, rows, w_trans):
    if rows is None:
        return w
    a, b = rows
    return w[:, a:b] if w_trans else w[a:b]


def _assemble(parts, w, w_trans):
    if len(parts) == 1 and parts[0][0] is None:
        return parts[0][1]
    parts = sorted(parts, key=lambda p: p[0][0])
    return torch.cat([p[1] for p in parts], dim=1 if w_trans else 0)


def seg_linear(inputs, weights, spec, id_info=None, bias=None, act=ops.ACT_NONE, w_trans=False,
               w_rows=None):
    if w_rows is None:
        w_rows = (None,) * len(spec)
    return _SegLinear.apply(tuple(spec), tuple(w_rows), bool(w_trans), act, id_info, len(inputs), bias,
                            *inputs, *weights)


def id_linear(x, weight, weight_id, id_info, bias=None):
    """x W + onehot(id) (x W_id) in one pass (ref: idconv.py:64-67,152-155,307-310)."""
    return seg_linear([x], [weight, weight_id], [(0, 0, False), (0, 1, True)], id_info, bias)


def linear(x, weight, bias=None, act=ops.ACT_NONE, w_trans=True):
    return seg_linear([x], [weight], [(0, 0, False)], None, bias, act, w_trans)


class _GatherRows(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, ids):
        ctx.ids, ctx.n = ids, x.size(0)
        return ops.gather_rows(x.contiguous(), ids)

    @staticmethod
    def backward(ctx, g):
        gx = torch.zeros((ctx.n, g.size(1)), dtype=g.dtype, device=g.device)
        ops.scatter_add_rows_(gx, ctx.ids, g.contiguous())
        return gx, None


class _ScatterAddRows(torch.autograd.Function):
    """out = base; out[ids] += x  (index_add_, ref: idconv.py:375)."""

    @staticmethod
    def forward(ctx, base, ids, x):
        ctx.ids = ids
        out = base.clone()
        ops.scatter_add_rows_(out, ids, x.contiguous())
        return out

    @staticmethod
    def backward(ctx, g):
        g = g.contiguous()
        return g, None, ops.gather_rows(g, ctx.ids)


def gather_rows(x, ids):
    return _GatherRows.apply(x, ids)


def scatter_add_rows(base, ids, x):
    return _ScatterAddRows.apply(base, ids, x)


class _GatAggregate(torch.autograd.Function):
    """out[i] = sum_{j->i} softmax_i(leaky_relu(a_i.h_i + a_j.h_j)) h_j + bias  (ref: idconv.py:317-342)."""

    @staticmethod
    def forward(ctx, h, att, bias, layout, heads, slope):
        h = h.contiguous()
        need_grad = any(ctx.needs_input_grad[:3])
        out, alpha, a_tgt, a_src, pos = ops.gat_forward(layout.csr, h, att, heads, slope, bias, need_grad)
        ctx.layout, ctx.heads, ctx.slope = layout, heads, slope
        ctx.save_for_backward(h, att, bias, alpha, a_tgt, a_src, out, *(pos or ()))
        return out

    @staticmethod
    def backward(ctx, g):
        h, att, bias, alpha, a_tgt, a_src, out, *pos = ctx.saved_tensors
        g = g.contiguous()
        lay = ctx.layout
        dh, datt = ops.gat_backward(lay.csr, lay.csc, lay.csc2csr, h, att, ctx.heads, ctx.slope, bias, alpha,
                                    a_tgt, a_src, out, g, tuple(pos) or None)
        gb = ops.colsum(g) if (bias is not None and ctx.needs_input_grad[2]) else None
        return dh, datt.view_as(att), gb, None, None, None


class _GatAggregateMean(torch.autograd.Function):
    """out[i] = (sum_{j->i} alpha_ij h_j) / indeg(i) + bias: ``_GatAggregate``'s forward without the bias, then the row
    scale.  Its backward is the sum's backward on g / indeg, with the unscaled sum (kept from the forward, [n, f]) in
    place of out - bias."""

    @staticmethod
    def forward(ctx, h, att, bias, layout, heads, slope):
        h = h.contiguous()
        need_grad = any(ctx.needs_input_grad[:3])
        out_sum, alpha, a_tgt, a_src, pos = ops.gat_forward(layout.csr, h, att, heads, slope, None, need_grad)
        out = ops.rows_epilogue(out_sum, layout.csr, bias=bias)
        ctx.layout, ctx.heads, ctx.slope, ctx.has_bias = layout, heads, slope, bias is not None
        ctx.save_for_backward(h, att, alpha, a_tgt, a_src, out_sum, *(pos or ()))
        return out

    @staticmethod
    def backward(ctx, g):
        h, att, alpha, a_tgt, a_src, out_sum, *pos = ctx.saved_tensors
        g = g.contiguous()
        lay = ctx.layout
        g_mean = ops.rows_epilogue(g, lay.csr)
        dh, datt = ops.gat_backward(lay.csr, lay.csc, lay.csc2csr, h, att, ctx.heads, ctx.slope, None, alpha, a_tgt, a_src,
                                    out_sum, g_mean, tuple(pos) or None)
        gb = ops.colsum(g) if (ctx.has_bias and ctx.needs_input_grad[2]) else None
        return dh, datt.view_as(att), gb, None, None, None


class _GatAggregateMax(torch.autograd.Function):
    """out[i, c] = max_{j->i} alpha_ij[head(c)] h_j[c] (0 without in-edges) + bias, alpha the GAT attention; the gradient
    of the max goes to the first in-edge that reaches it, per column, and reaches h_j (scale alpha) and alpha (then the
    logits, att and h through the scores)."""

    @staticmethod
    def forward(ctx, h, att, bias, layout, heads, slope):
        h = h.contiguous()
        csr = layout.csr
        if heads == 1:
            a_tgt, a_src = ops.gat_scores(h, att.view(1, -1))
            alpha = ops.gat_alpha(csr, a_tgt, a_src, slope)
            out, arg = ops.spmm_max(csr, h, alpha, bias=bias)
        else:
            a_tgt, a_src = ops.gat_scores_heads(h, att, heads)
            alpha = ops.gat_alpha_heads(csr, a_tgt, a_src, heads, slope)
            out, arg = ops.spmm_max_heads(csr, h, alpha, heads, bias)
        ctx.layout, ctx.heads, ctx.slope, ctx.has_bias = layout, heads, slope, bias is not None
        ctx.save_for_backward(h, att, a_tgt, a_src, alpha, arg)
        return out

    @staticmethod
    def backward(ctx, g):
        h, att, a_tgt, a_src, alpha, arg = ctx.saved_tensors
        g = g.contiguous()
        lay, heads, slope = ctx.layout, ctx.heads, ctx.slope
        csr, csc, m = lay.csr, lay.csc, lay.csc2csr
        c = h.size(1) // heads
        att2 = att.view(heads, 2 * c)
        att_tgt, att_src = att2[:, :c].contiguous().view(-1), att2[:, c:].contiguous().view(-1)
        dalpha = ops.max_winner_sddmm(csr, arg, g, h, heads)
        if heads == 1:
            dz, da_tgt = ops.gat_dz(csr, a_tgt, a_src, alpha, dalpha.view(-1), slope)
            alpha_t, da_src = ops.gat_csc_gather(csc, m, alpha, dz)
            dh = ops.spmm_max_bwd(csc, m, g, arg, alpha_t)
        else:
            dz, da_tgt = ops.gat_dz_heads(csr, a_tgt, a_src, alpha, dalpha, heads, slope)
            da_src = ops.gat_src_sum_heads(csc, m, dz, heads)
            dh = ops.spmm_max_heads_bwd(csc, m, g, arg, alpha, heads)
        # + da_src att_src + da_tgt att_tgt: the scores a_src = att_src . h, a_tgt = att_tgt . h
        ops.rows_epilogue(dh, rank1=(da_src, att_src, da_tgt, att_tgt), heads=heads, out=dh)
        datt = ops.gat_att_grad(h, da_tgt, da_src, heads)
        gb = ops.colsum(g) if (ctx.has_bias and ctx.needs_input_grad[2]) else None
        return dh, datt.view_as(att), gb, None, None, None


def gat_aggregate(h, att, bias, layout, heads=1, slope=0.2, agg="add"):
    """``agg``: 'add' (sum over the in-edges), 'mean' or 'max'."""
    if agg == "mean":
        return _GatAggregateMean.apply(h, att, bias, layout, int(heads), float(slope))
    if agg == "max":
        return _GatAggregateMax.apply(h, att, bias, layout, int(heads), float(slope))
    return _GatAggregate.apply(h, att, bias, layout, int(heads), float(slope))


class _DotAttentionAgg(torch.autograd.Function):
    """out[i] = mean or max over j->i of softmax_i(<h_i, h_j> / sqrt(f)) h_j (+ bias): gmulconv's Q = K = V = h with a
    mean or max instead of the sum.  The backward sums the three gradient terms through the epilogues of the SpMMs."""

    @staticmethod
    def forward(ctx, h, bias, layout, agg):
        h = h.contiguous()
        csr = layout.csr
        scale = 1.0 / math.sqrt(h.size(1))
        z = ops.sddmm(csr, h, h)
        alpha = ops.segment_softmax(csr, z, scale)
        arg = None
        if agg == "max":
            out, arg = ops.spmm_max(csr, h, alpha, bias=bias)
        else:
            out = ops.spmm(csr, h, alpha, ops.MEAN, None, 0.0, bias)
        ctx.layout, ctx.scale, ctx.agg, ctx.has_bias = layout, scale, agg, bias is not None
        ctx.save_for_backward(h, alpha, arg)
        return out

    @staticmethod
    def backward(ctx, g):
        h, alpha, arg = ctx.saved_tensors
        lay = ctx.layout
        csr, csc, m = lay.csr, lay.csc, lay.csc2csr
        g = g.contiguous()
        if ctx.agg == "max":
            dalpha = ops.max_winner_sddmm(csr, arg, g, h).view(-1)
        else:
            g_mean = ops.rows_epilogue(g, csr)
            dalpha = ops.sddmm(csr, h, g_mean)
        dz = ops.segment_softmax_bwd(csr, alpha, dalpha, ctx.scale)
        alpha_t, _ = ops.gat_csc_gather(csc, m, alpha, dz)
        dz_t, _ = ops.gat_csc_gather(csc, m, dz, dz)
        if ctx.agg == "max":
            dv = ops.spmm_max_bwd(csc, m, g, arg, alpha_t)
        else:
            dv = ops.spmm(csc, g_mean, alpha_t)
        dq = ops.spmm(csr, h, dz, ops.SUM, dv, 1.0)          # + dv in the epilogue
        dh = ops.spmm(csc, h, dz_t, ops.SUM, dq, 1.0)        # dk + dq + dv
        gb = ops.colsum(g) if (ctx.has_bias and ctx.needs_input_grad[1]) else None
        return dh, gb, None, None


def dot_attention_aggregate(h, bias, layout, agg):
    """gmulconv's attention with ``agg`` in ('mean', 'max'); 'add' is ``tfg._DotAttention``."""
    return _DotAttentionAgg.apply(h, bias, layout, agg)


def _bn_forward(ctx, y, bn, training):
    """-> (mean, invstd) the post-op kernels normalise with (None, None without BN), updating ``bn``'s running statistics
    and num_batches_tracked as nn.BatchNorm1d would; sets ctx.train (batch statistics)."""
    mean = invstd = None
    if bn is not None:
        if training or bn.running_mean is None:
            mom = 0.0
            if training and bn.running_mean is not None:
                bn.num_batches_tracked += 1
                mom = bn.momentum if bn.momentum is not None else 1.0 / float(bn.num_batches_tracked)
            track = training and bn.running_mean is not None
            mean, invstd = ops.bn_stats(y, bn.eps, bn.running_mean if track else None,
                                        bn.running_var if track else None, mom)
            ctx.train = True
        else:
            mean = bn.running_mean
            invstd = torch.rsqrt(bn.running_var + bn.eps)   # [F]-sized, eval mode only
            ctx.train = False
    return mean, invstd


class _PostOps(torch.autograd.Function):
    """out = l2norm( act( BatchNorm1d(y) ) ) in two kernels forward (statistics, apply) and two backward
    (column sums, apply) — ref: graphgym/models/layer.py:26-46, gnn.py:79-80."""

    @staticmethod
    def forward(ctx, y, gamma, beta, bn, training, act, slope, l2norm):
        y = y.contiguous()
        mean, invstd = _bn_forward(ctx, y, bn, training)
        out, rownorm = ops.postops_fwd(y, mean, invstd, gamma, beta, act, slope, l2norm)
        ctx.act, ctx.slope, ctx.l2norm, ctx.has_bn = act, slope, l2norm, bn is not None
        ctx.save_for_backward(y, out, mean, invstd, gamma, rownorm)
        return out

    @staticmethod
    def backward(ctx, go):
        y, out, mean, invstd, gamma, rownorm = ctx.saved_tensors
        dy, dgamma, dbeta = ops.postops_bwd(go.contiguous(), out, y, mean, invstd, gamma, getattr(ctx, 'train', False),
                                            ctx.act, ctx.slope, ctx.l2norm, rownorm)
        if gamma is None:
            dgamma = dbeta = None
        return dy, dgamma, dbeta, None, None, None, None, None


def post_ops(y, bn=None, training=True, act=ops.ACT_NONE, slope=0.0, l2norm=False):
    """``bn``: an ``nn.BatchNorm1d`` (its parameters / buffers are used and updated as the module would) or None."""
    gamma = bn.weight if bn is not None else None
    beta = bn.bias if bn is not None else None
    return _PostOps.apply(y, gamma, beta, bn, bool(training), int(act), float(slope), bool(l2norm))


class _SkipPostOps(torch.autograd.Function):
    """The epilogue of a GraphGym skip block (ref: graphgym/models/gnn.py GNNSkipBlock, GNNSkipStage):
    SKIP_SUM out = l2norm( act( BatchNorm1d(y) + res ) ), SKIP_PREFIX out = l2norm( act( cat([res, BatchNorm1d(y)], 1) ) )
    in the post-op kernels, two forward (statistics, apply) and two backward (column sums, apply: dy and dres)."""

    @staticmethod
    def forward(ctx, y, res, gamma, beta, bn, training, act, slope, l2norm, mode):
        y = y.contiguous()
        mean, invstd = _bn_forward(ctx, y, bn, training)
        out, rownorm = ops.postops_skip_fwd(y, res, mode, mean, invstd, gamma, beta, act, slope, l2norm)
        ctx.act, ctx.slope, ctx.l2norm, ctx.mode = act, slope, l2norm, mode
        ctx.save_for_backward(y, out, mean, invstd, gamma, rownorm)
        return out

    @staticmethod
    def backward(ctx, go):
        y, out, mean, invstd, gamma, rownorm = ctx.saved_tensors
        dy, dres, dgamma, dbeta = ops.postops_skip_bwd(go.contiguous(), out, y, ctx.mode, mean, invstd, gamma,
                                                       getattr(ctx, 'train', False), ctx.act, ctx.slope, ctx.l2norm,
                                                       rownorm)
        if gamma is None:
            dgamma = dbeta = None
        return dy, dres, dgamma, dbeta, None, None, None, None, None, None


def skip_post_ops(y, res, mode, bn=None, training=True, act=ops.ACT_NONE, slope=0.0, l2norm=False):
    """``mode``: ops.SKIP_SUM (skipsum: + res) or ops.SKIP_PREFIX (skipconcat: res as the leading columns).
    ``bn``: an ``nn.BatchNorm1d`` on y (its parameters / buffers are used and updated as the module would) or None."""
    gamma = bn.weight if bn is not None else None
    beta = bn.bias if bn is not None else None
    return _SkipPostOps.apply(y, res, gamma, beta, bn, bool(training), int(act), float(slope), bool(l2norm), int(mode))
