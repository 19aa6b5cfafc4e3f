"""Max aggregation (cfg.gnn.agg = 'max') without a GPU: the oracle's propagate(aggr='max') against a per-edge Python loop
(strict `>` in edge order: the first edge reaching the maximum wins, its message alone gets the gradient), the chunked
fp64 step against that oracle + autograd, and the layer's construction-time checks."""
import pytest
import torch

from graphgym_b200 import functional as F_
from graphgym_b200.config import cfg, reset_cfg
from graphgym_b200.contrib.layer.generalconv import GeneralConvLayer
from oracle import layers as OL
from oracle import max_agg as M


def loop_max(ei, msg, n):
    """(out, arg) by a per-edge scan: strict `>` from -inf in edge order; empty rows 0 / -1."""
    f = msg.size(1)
    best = [[float('-inf')] * f for _ in range(n)]
    arg = [[-1] * f for _ in range(n)]
    for e in range(ei.size(1)):
        i = int(ei[1, e])
        for c in range(f):
            v = float(msg[e, c])
            if v > best[i][c]:
                best[i][c], arg[i][c] = v, e
    out = torch.tensor([[best[i][c] if arg[i][c] >= 0 else 0.0 for c in range(f)] for i in range(n)], dtype=torch.float64)
    return out, torch.tensor(arg, dtype=torch.long)


def graphs():
    g = torch.Generator().manual_seed(5)
    n = 12
    src = torch.randint(0, n - 3, (40,), generator=g)              # nodes n-3 .. n-1 have no in-edges
    tgt = torch.randint(0, n - 3, (40,), generator=g)
    src = torch.cat([src, src[:6], torch.tensor([2, 4, 4])])       # duplicate edges and self loops
    tgt = torch.cat([tgt, tgt[:6], torch.tensor([2, 4, 4])])
    return n, torch.stack([src, tgt])


@pytest.mark.parametrize('feat', ['randn', 'negative', 'equal', 'rounded'])
def test_propagate_max_equals_edge_loop(feat):
    n, ei = graphs()
    e, f = ei.size(1), 5
    g = torch.Generator().manual_seed(1)
    msg = {'randn': torch.randn(e, f, generator=g, dtype=torch.float64),
           'negative': -1.0 - torch.rand(e, f, generator=g, dtype=torch.float64),
           'equal': torch.full((e, f), 0.75, dtype=torch.float64),
           'rounded': torch.randint(-2, 3, (e, f), generator=g).double()}[feat]   # many ties inside a row
    msg.requires_grad_(True)
    out = M.propagate(ei, msg, n, 'max')
    want, arg = loop_max(ei, msg.detach(), n)
    assert (out.detach() - want).abs().max() <= 1e-12
    assert torch.equal(M.scatter_argmax(msg, ei[1], n), arg)
    assert (arg[n - 3:] == -1).all() and (out[n - 3:] == 0).all()
    gy = torch.randn(n, f, generator=g, dtype=torch.float64)
    out.backward(gy)
    gwant = torch.zeros(e, f, dtype=torch.float64)
    for i in range(n):
        for c in range(f):
            if arg[i, c] >= 0:
                gwant[arg[i, c], c] += gy[i, c]
    assert (msg.grad - gwant).abs().max() <= 1e-12
    if feat == 'equal':   # all messages of a row tie: the whole row's gradient lands on its first edge
        first = {}
        for k in range(e):
            first.setdefault(int(ei[1, k]), k)
        assert all((arg[i] == first[i]).all() for i in first)


def test_propagate_max_follows_a_given_arg():
    n, ei = graphs()
    g = torch.Generator().manual_seed(2)
    msg = torch.randn(ei.size(1), 3, generator=g, dtype=torch.float64, requires_grad=True)
    own = M.scatter_argmax(msg, ei[1], n)
    last = own.clone()
    for k in range(ei.size(1)):        # the LAST edge into each row instead of the winner
        last[int(ei[1, k])] = k
    out = M.propagate(ei, msg, n, 'max', arg=last)
    assert torch.equal(out.detach(), torch.where(last >= 0, msg.detach().gather(0, last.clamp(min=0)), torch.zeros(())))
    out.sum().backward()
    assert msg.grad.sum() == (last >= 0).sum()


@pytest.mark.parametrize('normalize', [False, True])
@pytest.mark.parametrize('self_msg', ['none', 'add', 'concat'])
def test_chunked_max_step_equals_oracle_autograd(normalize, self_msg):
    n, ei = graphs()
    g = torch.Generator().manual_seed(3)
    x = torch.randn(n, 4, generator=g, dtype=torch.float64, requires_grad=True)
    w = torch.randn(4, 6, generator=g, dtype=torch.float64, requires_grad=True)
    ws = torch.randn(4, 6, generator=g, dtype=torch.float64, requires_grad=True)
    b = torch.randn(6, generator=g, dtype=torch.float64, requires_grad=True)
    gy = torch.randn(n, 6, generator=g, dtype=torch.float64)
    out = M.general_conv(x, ei, w, ws, b, 'max', normalize, self_msg)
    out.backward(gy)
    got = M.general_conv_max_step(x.detach(), ei, w.detach(), ws.detach(), b.detach(), gy, normalize, self_msg,
                                  chunk=7)
    assert (got[0] - out.detach()).abs().max() <= 1e-12
    assert (got[1] - x.grad).abs().max() <= 1e-12 and (got[2] - w.grad).abs().max() <= 1e-12
    assert (got[4] - b.grad).abs().max() <= 1e-12 and (got[6] == 0).all()
    if self_msg == 'concat':
        assert (got[3] - ws.grad).abs().max() <= 1e-12
    # under another arg: the oracle's autograd under that arg, and the gap to the maximum it leaves
    h = x.detach() @ w.detach()
    eie, norm = OL.gcn_norm_src(ei, n, x.dtype) if normalize else (ei, None)
    msg = h[eie[0]] if norm is None else h[eie[0]] * norm.view(-1, 1)
    last = got[5].clone()
    for k in range(eie.size(1)):
        last[int(eie[1, k])] = k
    x2, w2 = x.detach().clone().requires_grad_(True), w.detach().clone().requires_grad_(True)
    M.general_conv(x2, ei, w2, ws.detach(), b.detach(), 'max', normalize, self_msg, arg=last).backward(gy)
    got2 = M.general_conv_max_step(x.detach(), ei, w.detach(), ws.detach(), b.detach(), gy, normalize, self_msg,
                                   arg=last, chunk=5)
    assert (got2[1] - x2.grad).abs().max() <= 1e-12 and (got2[2] - w2.grad).abs().max() <= 1e-12
    want_gap = M.gather_max(msg, got[5]) - M.gather_max(msg, last)
    assert (got2[6] - want_gap).abs().max() <= 1e-12 and (got2[6] >= 0).all()


@pytest.mark.parametrize('normalize', [False, True])
@pytest.mark.parametrize('self_msg', ['none', 'add', 'concat'])
def test_generalconv_constructs_with_max(normalize, self_msg):
    reset_cfg()
    cfg.gnn.agg, cfg.gnn.normalize_adj, cfg.gnn.self_msg = 'max', normalize, self_msg
    layer = GeneralConvLayer(5, 7)
    assert layer.aggr == 'max' and layer.normalize is normalize
    assert hasattr(layer, 'weight_self') == (self_msg == 'concat')
    reset_cfg()


def test_bf16_gather_with_max_raises():
    reset_cfg()
    cfg.b200.gather_dtype = 'bf16'
    try:
        for kind in ('max', 'gcn_src_max'):
            with pytest.raises(NotImplementedError):
                F_.aggregate(torch.zeros(4, 16), None, kind)
    finally:
        reset_cfg()
