"""splineconv (TEST INFRASTRUCTURE ONLY — see oracle/__init__.py).

ref: graphgym/models/layer.py ``SplineConv`` = pyg.nn.SplineConv(dim_in, dim_out, dim=1, kernel_size=2, bias=bias) over
(node_feature, edge_index, edge_feature).  PyG 1.6 defaults: is_open_spline, degree 1, aggr 'mean', root_weight.  The
degree-1 basis of torch_spline_conv, restated (parity unpinned: no PyG / torch_spline_conv build to run against):
  v = u (open spline, kernel size 2: u * (2 - 1)), t = (int64_t) v (trunc), fr = v - floor(v)
  basis 0: weight 1 - fr on kernel matrix t mod 2;  basis 1: weight fr on (t + 1) mod 2
  message  m_e = sum_b basis_b x_j W[index_b],  e = (j -> i), j = edge_index[0, e], i = edge_index[1, e]
  out_i    mean of m_e over the in-edges of i (0 without any), + x_i root + bias
  d u_e    sum_b d basis_b / du <g_i / indeg(i), x_j W[index_b]>, d basis_0 / du = -1, d basis_1 / du = +1
The mod is taken non-negative (t mod 2 in {0, 1}); for u <= -1 the reference indexes weight[-1].

  spline_conv        the literal basis in plain torch (autograd also through u)
  spline_conv_step   the same step over edge chunks with the backward spelled out, for full size (no [E, F] tensor
                     outlives its chunk)
  spline_conv_loop   the forward edge by edge in Python
"""
import torch


def basis(u):
    """(index0, index1, b0, b1) of torch_spline_conv's degree-1 open basis at pseudo-coordinates ``u`` [E]."""
    t = torch.trunc(u).long()
    fr = u - torch.floor(u)
    return torch.remainder(t, 2), torch.remainder(t + 1, 2), 1 - fr, fr


def coefficients(u):
    """[E, 2]: the weight of kernel matrix 0 and 1 on every edge (the two basis terms summed by matrix)."""
    i0, i1, b0, b1 = basis(u)
    c = torch.zeros(u.numel(), 2, dtype=u.dtype, device=u.device)
    c.scatter_add_(1, i0.view(-1, 1), b0.view(-1, 1))
    c.scatter_add_(1, i1.view(-1, 1), b1.view(-1, 1))
    return c


def spline_conv(x, edge_index, pseudo, weight, root, bias=None):
    """The layer's forward with autograd (through x, pseudo, weight, root, bias).  ``pseudo``: [E] or [E, 1];
    ``weight`` [2, in, out]."""
    n = x.size(0)
    src, tgt = edge_index
    u = pseudo.reshape(-1)
    i0, i1, b0, b1 = basis(u)
    xj = x.index_select(0, src)
    msg = (b0.view(-1, 1) * torch.bmm(xj.unsqueeze(1), weight[i0]).squeeze(1)
           + b1.view(-1, 1) * torch.bmm(xj.unsqueeze(1), weight[i1]).squeeze(1))
    out = torch.zeros(n, weight.size(2), dtype=x.dtype, device=x.device).index_add(0, tgt, msg)
    deg = torch.zeros(n, dtype=x.dtype, device=x.device).index_add_(0, tgt, torch.ones_like(tgt, dtype=x.dtype))
    out = out / deg.clamp(min=1).view(-1, 1) + x @ root
    return out + bias if bias is not None else out


def _chunks(e, chunk):
    for s in range(0, e, chunk):
        yield s, min(e, s + chunk)


def spline_conv_step(x, edge_index, pseudo, weight, root, bias, gy, chunk=1 << 22):
    """-> (out, dx, d pseudo (shape of ``pseudo``), dweight, droot, dbias) of ``spline_conv`` over edge chunks; runs
    wherever its inputs live (float64 on the GPU at full size).  Aggregate first: P_k = mean_e c_k,e x_j,
    out = P_0 W0 + P_1 W1 + x root + bias."""
    n = x.size(0)
    src, tgt = edge_index
    u = pseudo.reshape(-1)
    e = u.numel()
    deg = torch.zeros(n, dtype=x.dtype, device=x.device).index_add_(0, tgt, torch.ones_like(tgt, dtype=x.dtype))
    inv = (1.0 / deg.clamp(min=1)).view(-1, 1)
    p = [torch.zeros_like(x), torch.zeros_like(x)]
    for a, b in _chunks(e, chunk):
        c = coefficients(u[a:b])
        xj = x.index_select(0, src[a:b])
        for k in range(2):
            p[k].index_add_(0, tgt[a:b], c[:, k:k + 1] * xj)
    p = [pk * inv for pk in p]
    out = p[0] @ weight[0] + p[1] @ weight[1] + x @ root
    if bias is not None:
        out = out + bias
    dp = [(gy @ weight[k].t()) * inv for k in range(2)]          # d P_k / indeg, per target
    dx = gy @ root.t()
    du = torch.empty_like(u)
    for a, b in _chunks(e, chunk):
        i0, i1, _, _ = basis(u[a:b])
        c = coefficients(u[a:b])
        xj = x.index_select(0, src[a:b])
        dc = torch.stack([(dp[k].index_select(0, tgt[a:b]) * xj).sum(1) for k in range(2)], 1)
        du[a:b] = dc.gather(1, i1.view(-1, 1)).squeeze(1) - dc.gather(1, i0.view(-1, 1)).squeeze(1)
        dx.index_add_(0, src[a:b], c[:, 0:1] * dp[0].index_select(0, tgt[a:b]) + c[:, 1:2] * dp[1].index_select(0, tgt[a:b]))
    dw = torch.stack([p[k].t() @ gy for k in range(2)])
    return out, dx, du.view(pseudo.shape), dw, x.t() @ gy, (gy.sum(0) if bias is not None else None)


def spline_conv_loop(x, edge_index, pseudo, weight, root, bias=None):
    """The forward edge by edge in Python, torch_spline_conv's formula term by term (the definition, for tiny graphs)."""
    n = x.size(0)
    src, tgt = edge_index.tolist()
    u = pseudo.reshape(-1).tolist()
    msgs = [[] for _ in range(n)]
    for e, (j, i) in enumerate(zip(src, tgt)):
        v = u[e] * (2 - 1)
        t = int(v)                         # (int64_t) v
        fr = v - float(torch.floor(torch.tensor(v, dtype=torch.float64)))
        m = torch.zeros(weight.size(2), dtype=x.dtype)
        for k_mod, b in ((0, 1 - fr), (1, fr)):
            wi = (t + k_mod) % 2             # Python's % is the non-negative mod
            m = m + b * (x[j] @ weight[wi])
        msgs[i].append(m)
    rows = []
    for i in range(n):
        r = torch.stack(msgs[i]).mean(0) if msgs[i] else torch.zeros(weight.size(2), dtype=x.dtype)
        r = r + x[i] @ root
        rows.append(r + bias if bias is not None else r)
    return torch.stack(rows)
