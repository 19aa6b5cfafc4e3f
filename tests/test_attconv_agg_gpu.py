"""gaddconv / gmulconv with cfg.gnn.agg = 'mean' / 'max' on the GPU (csrc/attn_agg.cu, functional._GatAggregateMean /
_GatAggregateMax / _DotAttentionAgg).

Op level: the winner SDDMM against the fp64 masked sum under the kernel's arg, at widths 4 to 256 with one head and with
2 and 4 heads, on hub rows split into virtual rows, isolated nodes, duplicate edges, self loops, all-negative and all-equal
features; bitwise repeatable.  The multi-head max forward equals the fp32 oracle bit for bit, its backward is within 1e-5
of fp64.  Layer level: both layers, both aggregations, bias on and off, sliced-ELL and row paths, against
oracle.attconv in fp64 with the gradients taken under the kernel's arg; every place where the kernel's arg differs from
fp64's own is a near-tie.  Full size: the products-shaped graph, gaddconv 100 -> 128, one step against the chunked fp64
oracle on the device."""
import pytest
import torch

import bench
from graphgym_b200 import functional as F_
from graphgym_b200 import ops
from graphgym_b200.config import cfg, reset_cfg
from graphgym_b200.contrib.layer.attconv import GeneralAddAttConvLayer, GeneralMulAttConvLayer
from graphgym_b200.graph import clear_cache, get_layout
from oracle import attconv as A
from oracle import max_agg as M
from test_fullsize_step_parity_gpu import check_arrays, check_path, kernels_of
from test_max_agg_gpu import features, max_graph, to_edges
from util import FP32_TOL, powerlaw_graph

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def graph(cuda):
    return max_graph()


def small_graph():
    n0 = 600
    ei = powerlaw_graph(1, n0, 6)
    loops = torch.arange(0, n0, 37)
    ei = torch.cat([ei, ei[:, :100], torch.stack([loops, loops])], dim=1)
    return n0 + 20, ei


def winner_ref(csr, arg, g, h, heads):
    """fp64 dalpha [E', heads] and its magnitude bound: the masked sum of g[i, c] h[nbr[s], c] over the won columns."""
    n, f = g.shape
    a = arg.long()
    ok = a >= 0
    s = a.clamp(min=0)
    key = (s * heads + torch.arange(f, device=g.device) // (f // heads)).view(-1)
    prod = (g.double() * h.double().gather(0, csr.nbr.long()[s]) * ok).view(-1)
    want = torch.zeros(csr.num_slots * heads, dtype=torch.float64, device=g.device).index_add_(0, key, prod)
    mag = torch.zeros_like(want).index_add_(0, key, prod.abs())
    return want.view(-1, heads), mag.view(-1, heads)


@pytest.mark.parametrize('f,heads', [(4, 1), (16, 1), (36, 1), (128, 1), (200, 1), (256, 1), (64, 2), (128, 4)])
def test_winner_sddmm(cuda, graph, monkeypatch, f, heads):
    n, ei = graph
    monkeypatch.setattr(ops, 'SELL_SEG', 8)                 # hub rows split into many virtual rows
    lay = get_layout(ei.to(cuda), n, ops.LOOPS_KEEP)
    csr = lay.csr
    gen = torch.Generator().manual_seed(f + heads)
    w = (0.1 + torch.rand(csr.num_slots, heads, generator=gen)).to(cuda)
    g = torch.randn(n, f, generator=gen).to(cuda)
    w_rand = w
    for kind in ('randn', 'negative', 'equal'):
        h = features(kind, n, f, f).to(cuda)
        w = torch.ones_like(w_rand) if kind == 'equal' else w_rand     # equal messages: every row ties throughout
        if heads == 1:
            _, arg = ops.spmm_max(csr, h, w.view(-1))
        else:
            out, arg = ops.spmm_max_heads(csr, h, w, heads)
            # the fp32 oracle with the same weights, in edge order: bit for bit
            ids = csr.perm.long()
            w_edge = torch.empty_like(w)
            w_edge[ids] = w
            msg = (w_edge.repeat_interleave(f // heads, dim=1) * h[ei[0].to(cuda)])
            want_arg = M.scatter_argmax(msg, ei[1].to(cuda), n)
            assert torch.equal(to_edges(arg, ids), want_arg), kind
            assert torch.equal(out, M.gather_max(msg, want_arg)), kind
            dx = ops.spmm_max_heads_bwd(lay.csc, lay.csc2csr, g, arg, w, heads)
            a = arg.long()
            wv = w.double()[a.clamp(min=0), torch.arange(f, device=cuda) // (f // heads)] * (a >= 0)
            src = csr.nbr.long()[a.clamp(min=0)]
            dx_want = torch.zeros(n, f, dtype=torch.float64, device=cuda).scatter_add_(0, src, wv * g.double())
            dx_mag = torch.zeros(n, f, dtype=torch.float64, device=cuda).scatter_add_(0, src, (wv * g.double()).abs())
            check_arrays(f'max heads bwd f={f} H={heads} {kind}', {'dx': dx}, {'dx': dx_want}, {'dx': dx_mag})
        got = ops.max_winner_sddmm(csr, arg, g, h, heads)
        again = ops.max_winner_sddmm(csr, arg, g, h, heads)
        assert torch.equal(got, again), kind                   # bitwise repeatable
        want, mag = winner_ref(csr, arg, g, h, heads)
        check_arrays(f'winner f={f} H={heads} {kind}', {'dalpha': got}, {'dalpha': want}, {'dalpha': mag})
        if kind == 'equal' and heads == 1:                     # every row's arg is its first slot: the rest won nothing
            rp = csr.rowptr.long()
            first = torch.zeros(csr.num_slots, dtype=torch.bool, device=cuda)
            first[rp[:-1][rp[1:] > rp[:-1]]] = True
            assert (got.view(-1)[~first] == 0).all()


def make_layer(cuda, name, agg, fin, fout, bias, heads=1, seed=0):
    reset_cfg()
    cfg.gnn.agg, cfg.gnn.att_heads = agg, heads
    torch.manual_seed(seed)
    cls = GeneralAddAttConvLayer if name == 'gaddconv' else GeneralMulAttConvLayer
    layer = cls(fin, fout, bias=bias).to(cuda)
    reset_cfg()
    if bias:
        with torch.no_grad():
            layer.bias.uniform_(-0.3, 0.3)
    return layer


def run_layer(cuda, monkeypatch, layer, ei, x, gy):
    """forward + backward on the device -> (out, x.grad, the max's arg or None)."""
    seen = {}
    for fn in ('spmm_max', 'spmm_max_heads'):
        orig = getattr(ops, fn)

        def rec(*a, _orig=orig, **k):
            res = _orig(*a, **k)
            seen['arg'] = res[1]
            return res
        monkeypatch.setattr(ops, fn, rec)
    xg = x.detach().to(cuda).requires_grad_(True)
    out = layer(xg, ei.to(cuda))
    out.backward(gy.to(cuda))
    monkeypatch.undo()
    return out.detach(), xg.grad, seen.get('arg')


def oracle(name, layer, x, ei, agg, arg_e):
    """fp64 oracle on the device: (out, params with their grads after backward) — call ``backward`` on out."""
    p = {k: v.detach().double().clone().requires_grad_(True) for k, v in layer.named_parameters()}
    x64 = x.double().clone().requires_grad_(True)
    if name == 'gaddconv':
        out = A.gadd_conv(x64, ei, p['linear_msg.weight'], p['att'], p.get('bias'), layer.heads, agg, arg_e)
    else:
        out = A.gmul_conv(x64, ei, p['linear_msg.weight'], p.get('bias'), p['bias_att'], agg, arg_e)
    return out, x64, p


def check_layer(tag, name, layer, agg, out, gx, arg, lay, ei, x, gy, zero_grads=()):
    """``zero_grads``: parameters whose gradient is zero in exact arithmetic; both sides are rounding noise there, so the
    kernel's is held to 1e-5 of the largest weight gradient instead."""
    dev = out.device
    ei, x, gy = ei.to(dev), x.to(dev), gy.to(dev).double()
    arg_e = to_edges(arg, lay.csr.perm.long()) if arg is not None else None
    ref, x64, p = oracle(name, layer, x, ei, agg, arg_e)
    ref.backward(gy)
    if agg == 'max':     # a different winner is a near-tie: within 1e-5 of the row's scale of fp64's own maximum
        with torch.no_grad():
            own, _, _ = oracle(name, layer, x, ei, agg, None)
            b = p['bias'] if 'bias' in p else 0.0
            gap = (own - ref).abs()
            scale = (own - b).abs().amax(1, keepdim=True)
            assert (gap <= FP32_TOL * scale).all(), f'{tag}: the arg-max differs beyond a near-tie'
    got = {'out': out, 'dx': gx}
    want = {'out': ref.detach(), 'dx': x64.grad}
    for k, v in layer.named_parameters():
        if k == 'bias_att':         # cancels in the softmax: zero gradient, not computed
            continue
        if k in zero_grads:
            scale = float(layer.linear_msg.weight.grad.abs().max())
            assert float(v.grad.abs().max()) <= FP32_TOL * scale, f'{tag}: {k} should vanish'
            continue
        got[k], want[k] = v.grad, p[k].grad
    check_arrays(tag, got, want)


@pytest.mark.parametrize('name', ['gaddconv', 'gmulconv'])
@pytest.mark.parametrize('agg', ['mean', 'max'])
@pytest.mark.parametrize('path', ['sell', 'row'])
@pytest.mark.parametrize('bias', [False, True])
def test_layer(cuda, graph, monkeypatch, name, agg, path, bias):
    if path == 'sell':
        (n, ei), fin, fout = graph, 16, 36
    else:       # n + E' < 2**14: the merge-path / sliced-ELL kernels step aside (the scores need c % 4 == 0)
        (n, ei), fin, fout = small_graph(), 7, 12
    dims = (fin, fout)
    g = torch.Generator().manual_seed(fin * 10 + fout)
    x, gy = torch.randn(n, fin, generator=g), torch.randn(n, fout, generator=g)
    clear_cache()
    layer = make_layer(cuda, name, agg, fin, fout, bias)
    out, gx, arg = run_layer(cuda, monkeypatch, layer, ei, x, gy)
    lay = get_layout(ei.to(cuda), n, ops.LOOPS_KEEP)
    check_layer(f'{name} {agg} {dims} bias={bias}', name, layer, agg, out, gx, arg, lay, ei, x, gy)


@pytest.mark.parametrize('agg', ['mean', 'max'])
@pytest.mark.parametrize('heads', [2, 4])
def test_gaddconv_heads(cuda, graph, monkeypatch, agg, heads):
    n, ei = graph
    g = torch.Generator().manual_seed(heads)
    x, gy = torch.randn(n, 16, generator=g), torch.randn(n, 64, generator=g)
    clear_cache()
    layer = make_layer(cuda, 'gaddconv', agg, 16, 64, True, heads)
    out, gx, arg = run_layer(cuda, monkeypatch, layer, ei, x, gy)
    lay = get_layout(ei.to(cuda), n, ops.LOOPS_KEEP)
    check_layer(f'gaddconv {agg} H={heads}', 'gaddconv', layer, agg, out, gx, arg, lay, ei, x, gy)


@pytest.mark.parametrize('name', ['gaddconv', 'gmulconv'])
def test_max_all_ones_input(cuda, graph, monkeypatch, name):
    """node_feature = ones [N, 1]: every h_i is the same, so every alpha of a row and every message of a row is equal and
    every column's arg is the row's first slot."""
    n, ei = graph
    g = torch.Generator().manual_seed(7)
    x, gy = torch.ones(n, 1), torch.randn(n, 16, generator=g)
    clear_cache()
    layer = make_layer(cuda, name, 'max', 1, 16, True)
    out, gx, arg = run_layer(cuda, monkeypatch, layer, ei, x, gy)
    lay = get_layout(ei.to(cuda), n, ops.LOOPS_KEEP)
    rp = lay.csr.rowptr.long()
    nonempty = rp[1:] > rp[:-1]
    assert (arg.long()[nonempty] == rp[:-1][nonempty].view(-1, 1)).all()
    assert (arg[~nonempty] == -1).all()
    # equal logits in every row: the softmax's gradient sums to zero over each row, and datt = sum_i da_i h with one h
    check_layer(f'{name} all-ones', name, layer, 'max', out, gx, arg, lay, ei, x, gy, zero_grads=('att',))


@pytest.mark.parametrize('agg', ['max', 'mean'])
def test_gaddconv_full_size(cuda, monkeypatch, agg):
    """bench.WORKLOADS['products_gat']'s graph (seed 0), gaddconv 100 -> 128, one forward + backward against the chunked
    fp64 oracle on the device.  As test_fullsize_step_parity_gpu.py documents for products_gat, a few of the 64 M logits
    lie within float32 rounding of zero and take the other leaky-ReLU slope in float32 than in float64; here the oracle's
    backward takes the branches the kernels took (the sign of the float32 logit a_tgt[i] + a_src[j] that gat_alpha /
    gat_dz / the fused GAT kernels evaluate), as it takes the kernels' arg-max, and every array is held to 1e-5."""
    spec = bench.WORKLOADS['products_gat']
    n, ei_d = bench.gen_graph(spec, cuda, seed=0)
    g = torch.Generator(device=cuda).manual_seed(1)
    x = torch.randn(n, 100, generator=g, device=cuda)
    gy = torch.randn(n, 128, generator=g, device=cuda)
    clear_cache()
    layer = make_layer(cuda, 'gaddconv', agg, 100, 128, True)
    (out, gx, arg), kern = kernels_of(lambda: run_layer(cuda, monkeypatch, layer, ei_d, x, gy))
    if agg == 'max':
        check_path('full size max', kern, {'gat_alpha_kernel': 1, 'spmm_sell_max_kernel': 1, 'max_winner_sddmm_kernel': 1,
                                           'gat_dz_kernel': 1, 'gat_csc_gather_kernel': 1, 'spmm_sell_max_bwd_kernel': 1},
                   ('spmm_row_max_kernel', 'spmm_row_max_bwd_kernel', 'spmm_row_max_heads_kernel', 'gat_fwd_kernel'))
    else:
        check_path('full size mean', kern, {'gat_sell_fwd_train_kernel': 1, 'gat_sell_bwd_one_kernel': 1,
                                            'rows_epilogue_kernel': 2},
                   ('gat_fwd_kernel', 'gat_bwd_edge_kernel', 'gat_sell_bwd_edge_kernel'))
    lay = get_layout(ei_d, n, ops.LOOPS_KEEP)
    arg_e = to_edges(arg, lay.csr.perm.long()) if arg is not None else None
    with torch.no_grad():
        p = {k: v.detach() for k, v in layer.named_parameters()}
        args = (p['linear_msg.weight'], p['att'], p['bias'])
        a_tgt, a_src = ops.gat_scores(F_.linear(x, p['linear_msg.weight']), p['att'].view(1, -1))
        gate = (a_tgt[ei_d[1]] + a_src[ei_d[0]] > 0).view(-1, 1)
        ref = A.gadd_conv_step(x.double(), ei_d, *(t.double() for t in args), gy.double(), agg, arg=arg_e, gate=gate)
        s_t, s_s = (F_.linear(x, p['linear_msg.weight']).double() @ p['att'].double().view(2, -1).t()).unbind(1)
        flips = int(((s_t[ei_d[1]] + s_s[ei_d[0]] > 0).view(-1, 1) != gate).sum())
        print(f'full size {agg}: {flips} of {gate.numel()} logits take the other leaky-ReLU branch in float32')
        if agg == 'max':
            differ = ref[5] != arg_e
            scale = (ref[0] - p['bias'].double()).abs().amax(1, keepdim=True)
            assert ((ref[6].abs() <= FP32_TOL * scale) | ~differ).all(), 'the arg-max differs beyond a near-tie'
            print(f'full size max: {int(differ.sum())} of {differ.numel()} arg-max entries differ from fp64 (near-ties)')
        names = ('out', 'dx', 'dW', 'datt', 'db')
        got = dict(zip(names, (out, gx, layer.linear_msg.weight.grad, layer.att.grad, layer.bias.grad)))
        check_arrays(f'gaddconv full size {agg}', got, dict(zip(names, ref[:5])))
    clear_cache()
