"""gaddconv / gmulconv with cfg.gnn.agg = 'mean' / 'max' without a GPU: the oracle (oracle/attconv.py) against the
reference's own 'add' vectors and against a per-edge Python loop, its chunked full-size step against its autograd, and the
layers' configuration checks."""
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from graphgym_b200.config import cfg, reset_cfg
from graphgym_b200.contrib.layer.attconv import GeneralAddAttConvLayer, GeneralMulAttConvLayer
from oracle import attconv as A
from util import rel_err

TOL = 1e-5


def _case(d, tag):
    t = lambda k: torch.from_numpy(d[tag + '/' + k]).double()
    params = {k.split('/param/')[1]: torch.from_numpy(d[k]).double().clone().requires_grad_(True)
              for k in d.files if k.startswith(tag + '/param/')}
    grads = {k.split('/grad/')[1]: torch.from_numpy(d[k]).double() for k in d.files if k.startswith(tag + '/grad/')}
    return t('x').clone().requires_grad_(True), torch.from_numpy(d[tag + '/edge_index']), t('y'), t('gy'), t('gx'), params, \
        grads


@pytest.mark.parametrize('tag', ['gaddconv', 'gaddconv_wide', 'gmulconv', 'gmulconv_wide'])
def test_oracle_add_reproduces_reference_vectors(golden_dir, tag):
    d = np.load(os.path.join(golden_dir, 'contrib_layers.npz'), allow_pickle=False)
    x, ei, y, gy, gx, p, grads = _case(d, tag)
    w = p['model.linear_msg.weight']
    if tag.startswith('gadd'):
        att = p['model.att']
        out = A.gadd_conv(x, ei, w, att, p['model.bias'], heads=att.size(1), aggr='add')
    else:
        out = A.gmul_conv(x, ei, w, p['model.bias'], p['model.bias_att'], aggr='add')
    assert rel_err(out.detach(), y) < TOL
    out.backward(gy)
    assert rel_err(x.grad, gx) < TOL
    for k, want in grads.items():
        if k == 'model.bias_att':      # cancels in the softmax: rounding noise in the reference
            continue
        assert rel_err(p[k].grad, want) < TOL, k


def graphs():
    g = torch.Generator().manual_seed(5)
    n = 12
    src = torch.randint(0, n - 3, (40,), generator=g)              # nodes n-3 .. n-1 have no in-edges
    tgt = torch.randint(0, n - 3, (40,), generator=g)
    src = torch.cat([src, src[:6], torch.tensor([2, 4, 4])])       # duplicate edges and self loops
    tgt = torch.cat([tgt, tgt[:6], torch.tensor([2, 4, 4])])
    return n, torch.stack([src, tgt])


def loop_layer(h, ei, n, logit, heads, aggr):
    """Per-edge loop: softmax over each target's edges per head, then mean / max of alpha h_j per column."""
    e, f = ei.size(1), h.size(1)
    c = f // heads
    out = torch.zeros(n, f, dtype=torch.float64)
    for i in range(n):
        es = [k for k in range(e) if int(ei[1, k]) == i]
        if not es:
            continue
        for k in range(heads):
            zs = [logit(int(ei[1, s]), int(ei[0, s]), k) for s in es]
            m = max(zs)
            ex = [math.exp(z - m) for z in zs]
            den = sum(ex) + 1e-16
            for col in range(k * c, (k + 1) * c):
                vals = [ex[t] / den * float(h[int(ei[0, s]), col]) for t, s in enumerate(es)]
                out[i, col] = sum(vals) / len(vals) if aggr == 'mean' else max(vals)
    return out


@pytest.mark.parametrize('aggr', ['mean', 'max'])
@pytest.mark.parametrize('heads', [1, 2])
def test_gadd_conv_equals_edge_loop(aggr, heads):
    n, ei = graphs()
    g = torch.Generator().manual_seed(1)
    x = torch.randn(n, 5, generator=g, dtype=torch.float64)
    w = torch.randn(6, 5, generator=g, dtype=torch.float64)
    att = torch.randn(1, heads, 2 * (6 // heads), generator=g, dtype=torch.float64)
    h = x @ w.t()
    c = 6 // heads
    a = att.view(heads, 2 * c)

    def logit(i, j, k):
        return float(F.leaky_relu(h[i, k * c:(k + 1) * c] @ a[k, :c] + h[j, k * c:(k + 1) * c] @ a[k, c:], 0.2))

    want = loop_layer(h, ei, n, logit, heads, aggr)
    got = A.gadd_conv(x, ei, w, att, None, heads, aggr)
    assert (got - want).abs().max() <= 1e-12
    assert (got[n - 3:] == 0).all()


@pytest.mark.parametrize('aggr', ['mean', 'max'])
def test_gmul_conv_equals_edge_loop(aggr):
    n, ei = graphs()
    g = torch.Generator().manual_seed(2)
    x = torch.randn(n, 5, generator=g, dtype=torch.float64)
    w = torch.randn(6, 5, generator=g, dtype=torch.float64)
    h = x @ w.t()
    want = loop_layer(h, ei, n, lambda i, j, k: float(h[i] @ h[j]) / math.sqrt(6), 1, aggr)
    got = A.gmul_conv(x, ei, w, None, None, aggr)
    assert (got - want).abs().max() <= 1e-12


@pytest.mark.parametrize('aggr', ['add', 'mean', 'max'])
@pytest.mark.parametrize('heads', [1, 2])
def test_chunked_step_equals_oracle_autograd(aggr, heads):
    n, ei = graphs()
    g = torch.Generator().manual_seed(3)
    x = torch.randn(n, 4, generator=g, dtype=torch.float64, requires_grad=True)
    w = torch.randn(6, 4, generator=g, dtype=torch.float64, requires_grad=True)
    att = torch.randn(1, heads, 12 // heads, generator=g, dtype=torch.float64, requires_grad=True)
    b = torch.randn(6, generator=g, dtype=torch.float64, requires_grad=True)
    gy = torch.randn(n, 6, generator=g, dtype=torch.float64)
    out = A.gadd_conv(x, ei, w, att, b, heads, aggr)
    out.backward(gy)
    got = A.gadd_conv_step(x.detach(), ei, w.detach(), att.detach(), b.detach(), gy, aggr, heads, chunk=7)
    for k, want in ((0, out.detach()), (1, x.grad), (2, w.grad), (3, att.grad), (4, b.grad)):
        assert (got[k] - want).abs().max() <= 1e-12, k
    if aggr != 'max':
        return
    assert (got[6] == 0).all()
    # under another arg (the last edge into each row): the oracle's autograd under it, and the gap it leaves
    last = got[5].clone()
    for k in range(ei.size(1)):
        last[int(ei[1, k])] = k
    x2, w2, a2 = (t.detach().clone().requires_grad_(True) for t in (x, w, att))
    A.gadd_conv(x2, ei, w2, a2, b.detach(), heads, 'max', arg=last).backward(gy)
    got2 = A.gadd_conv_step(x.detach(), ei, w.detach(), att.detach(), b.detach(), gy, 'max', heads, arg=last, chunk=5)
    for k, want in ((1, x2.grad), (2, w2.grad), (3, a2.grad)):
        assert (got2[k] - want).abs().max() <= 1e-12, k
    assert (got2[6] >= 0).all() and (got2[6] > 0).any()


@pytest.mark.parametrize('agg', ['add', 'mean', 'max'])
def test_layers_construct_with_every_agg(agg):
    reset_cfg()
    try:
        cfg.gnn.agg = agg
        assert GeneralAddAttConvLayer(8, 8).agg == agg
        assert GeneralMulAttConvLayer(8, 8).agg == agg
        cfg.gnn.normalize_adj = True
        for cls in (GeneralAddAttConvLayer, GeneralMulAttConvLayer):
            with pytest.raises(NotImplementedError):
                cls(8, 8)
    finally:
        reset_cfg()
