"""Differentiable building blocks of the layers: each one is a ``torch.autograd.Function`` whose
forward AND backward are ``gg_*`` kernels (no torch math on the path).

  aggregate    CSR SpMM forward, CSC SpMM backward            (SURVEY §8a row 4); max: arg-max forward, masked CSC sum
  seg_linear   multi-segment dense transform with ID weights  (SURVEY §8a row 9)
  gather_rows / scatter_add_rows   the M-row ID branch of GIN-ID (ref: idconv.py:372-375)
"""
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


def gat_aggregate(h, att, bias, layout, heads=1, slope=0.2):
    return _GatAggregate.apply(h, att, bias, layout, int(heads), float(slope))


class _PostOps(torch.autograd.Function):
    """out = l2norm( act( BatchNorm1d(y) ) ) in two kernels forward (statistics, apply) and two backward
    (column sums, apply) — ref: graphgym/models/layer.py:26-46, gnn.py:79-80."""

    @staticmethod
    def forward(ctx, y, gamma, beta, bn, training, act, slope, l2norm):
        y = y.contiguous()
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
