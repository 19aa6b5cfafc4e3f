"""generaledgeconv / generalsampleedgeconv on the GPU (csrc/edge_agg.cu, functional.edge_aggregate).

Op level, on a power-law graph with hub rows split into virtual rows, isolated nodes, duplicate edges and self loops: the
edge-row reduce and its gather backward, the max with the edge term on both paths against fp64 (every arg-max disagreement
a near-tie), the winner and dW_a kernels against fp64 under the kernel's arg, and bitwise repeatability.  Layer level:
every agg x msg_direction x self_msg x bias against oracle.edgeconv in fp64.  Full size: the products-shaped graph,
100 -> 128, edge_dim 16, against the chunked fp64 oracle on the device, with the kernels that ran and the memory peak."""
import itertools

import pytest
import torch

import bench
from graphgym_b200 import functional as F_
from graphgym_b200 import ops
from graphgym_b200.config import cfg, reset_cfg
from graphgym_b200.contrib.layer.generalconv import GeneralEdgeConvLayer, GeneralSampleEdgeConv, sample_edges
from graphgym_b200.graph import clear_cache, get_layout
from graphgym_b200.models.layer import Batch
from oracle import edgeconv as E
from test_fullsize_step_parity_gpu import check_arrays, check_path, kernels_of
from test_max_agg_gpu import max_graph, to_edges
from util import FP32_TOL

pytestmark = pytest.mark.gpu

FS = [1, 3, 16, 64, 128, 200, 256]
KDS = [1, 7, 16, 64, 256]


@pytest.fixture(scope='module')
def graph(cuda):
    return max_graph()


@pytest.fixture(autouse=True)
def _fresh(monkeypatch):
    monkeypatch.setattr(ops, 'SELL_SEG', 8)       # hub rows split into many virtual rows: partials + fix-up
    reset_cfg()
    clear_cache()
    yield
    reset_cfg()
    clear_cache()


def layout(cuda, graph):
    n, ei = graph
    eid = ei.to(cuda)
    return n, eid, get_layout(eid, n, ops.LOOPS_KEEP)


@pytest.mark.parametrize('kd', [1, 3, 16, 128])
def test_edge_row_reduce(cuda, graph, kd):
    n, ei, lay = layout(cuda, graph)
    g = torch.Generator(device=cuda).manual_seed(kd)
    a = torch.randn(ei.size(1), kd, generator=g, device=cuda)
    deg = torch.zeros(n, dtype=torch.float64, device=cuda).index_add_(0, ei[1], torch.ones(ei.size(1), dtype=torch.float64,
                                                                                           device=cuda))
    for mean in (False, True):
        got = ops.edge_row_reduce(lay.csr, a, mean)
        assert torch.equal(got, ops.edge_row_reduce(lay.csr, a, mean))
        want = torch.zeros(n, kd, dtype=torch.float64, device=cuda).index_add_(0, ei[1], a.double())
        mag = torch.zeros(n, kd, dtype=torch.float64, device=cuda).index_add_(0, ei[1], a.double().abs())
        if mean:
            want, mag = want / deg.clamp(min=1).view(-1, 1), mag / deg.clamp(min=1).view(-1, 1)
        check_arrays(f'row reduce kd={kd} mean={mean}', {'sa': got}, {'sa': want}, {'sa': mag})
    # the backward: (g W_a)[target] (/ indeg), in edge order
    w = torch.randn(32, kd, generator=g, device=cuda)
    gy = torch.randn(n, 32, generator=g, device=cuda)
    for agg in ('add', 'mean'):
        a_ = a.clone().requires_grad_(True)
        w_ = w.clone().requires_grad_(True)
        hj = torch.zeros(n, 32, device=cuda, requires_grad=True)
        F_.edge_aggregate(hj, None, a_, w_, lay, agg).backward(gy)
        sc = (1.0 / deg.clamp(min=1)) if agg == 'mean' else torch.ones_like(deg)
        gs = gy.double() * sc.view(-1, 1)
        want = (gs @ w.double())[ei[1]]
        mag = ((gs.abs() @ w.double().abs()))[ei[1]]
        sa = torch.zeros(n, kd, dtype=torch.float64, device=cuda).index_add_(0, ei[1], a.double()) * sc.view(-1, 1)
        sam = torch.zeros(n, kd, dtype=torch.float64, device=cuda).index_add_(0, ei[1], a.double().abs()) * sc.view(-1, 1)
        check_arrays(f'row reduce bwd kd={kd} {agg}', {'da': a_.grad, 'dw': w_.grad},
                     {'da': want, 'dw': gy.double().t() @ sa}, {'da': mag, 'dw': gy.double().abs().t() @ sam})


def max_inputs(kind, n, e, f, kd, seed, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    if kind == 'randn':
        return (torch.randn(n, f, generator=g, device=dev), torch.randn(e, kd, generator=g, device=dev),
                torch.randn(f, kd, generator=g, device=dev) / kd ** 0.5)
    if kind == 'negative':           # every message negative: a padding entry (0) must never win
        return (-0.5 - torch.rand(n, f, generator=g, device=dev), torch.rand(e, kd, generator=g, device=dev),
                -torch.rand(f, kd, generator=g, device=dev))
    if kind == 'dominant':           # negative edge terms that dominate the node term
        return (0.01 * torch.randn(n, f, generator=g, device=dev), torch.rand(e, kd, generator=g, device=dev) + 1.0,
                -2.0 - torch.rand(f, kd, generator=g, device=dev))
    return torch.ones(n, f, device=dev), torch.zeros(e, kd, device=dev), torch.randn(f, kd, generator=g, device=dev)


def fp64_max(ei, n, hj, hi, a, w):
    """(out, own arg as edge ids, message function) of the max in fp64, 0 without in-edges."""
    msg = hj.double()[ei[0]] + a.double() @ w.double().t()
    if hi is not None:
        msg = msg + hi.double()[ei[1]]
    from oracle import max_agg as M
    own = M.scatter_argmax(msg, ei[1], n)
    mag = torch.zeros(n, hj.size(1), dtype=torch.float64, device=hj.device).index_reduce_(
        0, ei[1], hj.double().abs()[ei[0]] + a.double().abs() @ w.double().abs().t(), 'amax', include_self=True)
    if hi is not None:
        mag = mag + hi.double().abs()
    return M.gather_max(msg, own), own, msg, mag


@pytest.mark.parametrize('f,kd', list(itertools.product(FS, KDS)))
def test_edge_max_forward(cuda, graph, f, kd):
    n, ei, lay = layout(cuda, graph)
    csr = lay.csr
    perm = csr.perm.long()
    paths = ('row',) if f % 4 else ('sell', 'row')
    for kind in ('randn', 'negative', 'dominant', 'equal'):
        hj, a, w = max_inputs(kind, n, ei.size(1), f, kd, f * 1000 + kd, cuda)
        hi = None if kind == 'equal' else torch.randn(n, f, device=cuda)
        want, own, msg, mag = fp64_max(ei, n, hj, hi, a, w)
        res = {}
        for algo in paths:
            out, arg = ops.edge_max(csr, hj, hi, a, w, algo=algo)
            out2, arg2 = ops.edge_max(csr, hj, hi, a, w, algo=algo)
            assert torch.equal(out, out2) and torch.equal(arg, arg2), (kind, algo)       # bitwise repeatable
            res[algo] = (out, arg)
            arg_e = to_edges(arg, perm)
            assert torch.equal(arg_e < 0, own < 0), (kind, algo)
            chosen = torch.where(arg_e >= 0, msg.gather(0, arg_e.clamp(min=0)), torch.zeros_like(want))
            differ = arg_e != own
            assert ((want - chosen).abs() <= FP32_TOL * mag).all(), f'{kind} {algo}: arg-max differs beyond a near-tie'
            if int(differ.sum()):
                print(f'f={f} kd={kd} {kind} {algo}: {int(differ.sum())} near-tie arg differences')
            check_arrays(f'edge max f={f} kd={kd} {kind} {algo}', {'out': out}, {'out': want}, {'out': mag})
            if kind == 'equal':           # every row's arg is its first slot
                rp = csr.rowptr.long()
                nonempty = rp[1:] > rp[:-1]
                assert (arg.long()[nonempty] == rp[:-1][nonempty].view(-1, 1)).all()
                assert (arg[~nonempty] == -1).all() and (out[~nonempty] == 0).all()
        if len(paths) == 2:
            assert torch.equal(res['sell'][0], res['row'][0]) and torch.equal(res['sell'][1], res['row'][1])


@pytest.mark.parametrize('f,kd', [(16, 1), (64, 7), (128, 16), (200, 64), (256, 256), (3, 16)])
def test_edge_max_backward(cuda, graph, f, kd):
    n, ei, lay = layout(cuda, graph)
    csr = lay.csr
    hj, a, w = max_inputs('randn', n, ei.size(1), f, kd, f + kd, cuda)
    out, arg = ops.edge_max(csr, hj, None, a, w)
    gy = torch.randn(n, f, device=cuda)
    arg_e = to_edges(arg, csr.perm.long())
    e = ei.size(1)
    won = torch.zeros(e, f, dtype=torch.float64, device=cuda)        # dm[e, c] = g[i, c] where e won (i, c)
    wonm = torch.zeros(e, f, dtype=torch.float64, device=cuda)
    ok = arg_e >= 0
    cols = torch.arange(f, device=cuda).expand(n, f)
    won[arg_e[ok], cols[ok]] = gy.double()[ok]
    wonm[arg_e[ok], cols[ok]] = gy.double().abs()[ok]
    da = ops.edge_max_winner(csr, arg, gy, w)
    dw = ops.edge_max_wgrad(csr, arg, gy, a)
    assert torch.equal(da, ops.edge_max_winner(csr, arg, gy, w)) and torch.equal(dw, ops.edge_max_wgrad(csr, arg, gy, a))
    check_arrays(f'edge max bwd f={f} kd={kd}', {'da': da, 'dw': dw},
                 {'da': won @ w.double(), 'dw': won.t() @ a.double()},
                 {'da': wonm @ w.double().abs(), 'dw': wonm.t() @ a.double().abs()})
    assert (da[(won == 0).all(1)] == 0).all()          # edges that won nothing get zeros
    mask = ops.max_mask(gy, arg)
    assert torch.equal(mask, torch.where(arg >= 0, gy, torch.zeros_like(gy)))


def run_layer(cuda, ei, n, fin, fout, kd, agg, direction, self_msg, bias, x, a, gy, seed=0):
    cfg.gnn.agg, cfg.gnn.msg_direction, cfg.gnn.self_msg, cfg.dataset.edge_dim = agg, direction, self_msg, kd
    torch.manual_seed(seed)
    layer = GeneralEdgeConvLayer(fin, fout, bias=bias).to(cuda)
    if bias:
        with torch.no_grad():
            layer.bias.uniform_(-0.3, 0.3)
    xg = x.detach().clone().requires_grad_(True)
    ag = a.detach().clone().requires_grad_(True)
    out = layer(xg, ei, edge_feature=ag)
    out.backward(gy)
    arg = None
    if agg == 'max':      # the arg the layer used: same inputs, same deterministic kernels
        w = layer.linear_msg.weight.detach()
        hj = F_.linear(xg.detach(), w[:, fin:2 * fin] if direction == 'both' else w[:, :fin])
        hi = F_.linear(xg.detach(), w[:, :fin]) if direction == 'both' else None
        wa = w[:, (2 if direction == 'both' else 1) * fin:]
        _, arg = ops.edge_max(get_layout(ei, n, ops.LOOPS_KEEP).csr, hj, hi, a, wa)
    return layer, out.detach(), xg.grad, ag.grad, arg


def check_layer(tag, ei, n, layer, out, gx, ga, arg, x, a, gy, agg, direction, self_msg, chunk=1 << 22):
    with torch.no_grad():
        p = {k: v.detach().double() for k, v in layer.named_parameters()}
        ws, b = p.get('linear_self.weight'), p.get('bias')
        arg_e = to_edges(arg, get_layout(ei, n, ops.LOOPS_KEEP).csr.perm.long()) if arg is not None else None
        ref = E.general_edge_conv_step(x.double(), ei, a.double(), p['linear_msg.weight'], ws, b, gy.double(), agg,
                                       direction, self_msg, arg=arg_e, chunk=chunk)
        ab = lambda t: None if t is None else t.abs()
        mag = E.general_edge_conv_step(x.double().abs(), ei, a.double().abs(), p['linear_msg.weight'].abs(), ab(ws), ab(b),
                                       gy.double().abs(), 'add' if agg == 'max' else agg, direction, self_msg, chunk=chunk)
        if agg == 'max':
            # a different winner is a near-tie: its fp64 message lies within 1e-5 (of the row's scale) of the maximum
            assert (ref[7].abs() <= FP32_TOL * mag[0]).all(), f'{tag}: arg-max differs beyond a near-tie'
            print(f'{tag}: {int((ref[6] != arg_e).sum())} near-tie arg differences')
        got = {'out': out, 'dx': gx, 'da': ga, 'dWmsg': layer.linear_msg.weight.grad}
        want = {'out': ref[0], 'dx': ref[1], 'da': ref[2], 'dWmsg': ref[3]}
        bound = {'out': mag[0], 'dx': mag[1], 'da': mag[2], 'dWmsg': mag[3]}
        if ws is not None:
            got['dWself'], want['dWself'], bound['dWself'] = layer.linear_self.weight.grad, ref[4], mag[4]
        if b is not None:
            got['db'], want['db'], bound['db'] = layer.bias.grad, ref[5], mag[5]
        check_arrays(tag, got, want, bound)


@pytest.mark.parametrize('width', [16, 63, 128])
@pytest.mark.parametrize('agg,direction,self_msg,bias',
                         list(itertools.product(['add', 'mean', 'max'], ['single', 'both'], ['none', 'add', 'concat'],
                                                [False, True])))
def test_layer(cuda, graph, width, agg, direction, self_msg, bias):
    n, ei, _ = layout(cuda, graph)
    kd = 7
    g = torch.Generator(device=cuda).manual_seed(width)
    x = torch.randn(n, width, generator=g, device=cuda)
    a = torch.rand(ei.size(1), kd, generator=g, device=cuda) * 2 - 1
    gy = torch.randn(n, width, generator=g, device=cuda)
    layer, out, gx, ga, arg = run_layer(cuda, ei, n, width, width, kd, agg, direction, self_msg, bias, x, a, gy)
    check_layer(f'layer w={width} {agg} {direction} {self_msg} bias={bias}', ei, n, layer, out, gx, ga, arg, x, a, gy,
                agg, direction, self_msg)
    # bitwise repeatable, forward and backward
    layer2, out2, gx2, ga2, _ = run_layer(cuda, ei, n, width, width, kd, agg, direction, self_msg, bias, x, a, gy)
    assert torch.equal(out, out2) and torch.equal(gx, gx2) and torch.equal(ga, ga2)
    assert torch.equal(layer.linear_msg.weight.grad, layer2.linear_msg.weight.grad)


def test_sample_edge_conv(cuda, graph):
    n, ei, _ = layout(cuda, graph)
    cfg.dataset.edge_dim, cfg.gnn.agg, cfg.gnn.msg_direction = 5, 'max', 'both'
    x = torch.randn(n, 16, device=cuda)
    a = torch.randn(ei.size(1), 5, device=cuda)
    torch.manual_seed(0)
    conv = GeneralSampleEdgeConv(16, 16, bias=True).to(cuda)
    with torch.no_grad():
        conv.model.bias.uniform_(-1, 1)
    for keep in (0.5, 0.2):
        cfg.gnn.keep_edge = keep
        torch.cuda.manual_seed(123)
        got = conv(Batch(x, ei, edge_feature=a)).node_feature
        torch.cuda.manual_seed(123)
        mask = torch.rand(ei.size(1), device=cuda) < keep
        want = conv.model(x, ei[:, mask], edge_feature=a[mask])
        assert torch.equal(got, want)
    cfg.gnn.keep_edge = 1.0
    got = conv(Batch(x, ei, edge_feature=a)).node_feature
    assert torch.equal(got, conv.model(x, ei, edge_feature=a))
    cfg.gnn.keep_edge = 0.0
    got = conv(Batch(x, ei, edge_feature=a)).node_feature
    want = F_.linear(x, conv.model.linear_self.weight, conv.model.bias)
    assert torch.allclose(got, want, rtol=1e-6, atol=1e-6)
    # the kept fraction of a 1 M-edge list is within 5 sigma of keep_edge
    big = torch.zeros(2, 1 << 20, dtype=torch.long, device=cuda)
    feat = torch.zeros(1 << 20, 1, device=cuda)
    for keep in (0.1, 0.5, 0.9):
        kept, kf = sample_edges(big, feat, keep)
        m = big.size(1)
        assert kept.size(1) == kf.size(0)
        assert abs(kept.size(1) - keep * m) <= 5 * (m * keep * (1 - keep)) ** 0.5


def test_collate_and_model(cuda):
    """Small graphs with edge features through loader.collate (edge_feature rows stay aligned with edge_index) and a
    GNN of two generaledgeconv layers under stack and skipsum: forward + backward, bitwise repeatable, the first layer
    against the fp64 oracle."""
    from graphgym_b200.loader import GraphData, collate
    from graphgym_b200.models.gnn import GNN
    g = torch.Generator().manual_seed(5)
    graphs = []
    for k in range(6):
        nk = 20 + 7 * k
        ek = torch.randint(0, nk, (2, 3 * nk), generator=g)
        graphs.append(GraphData(node_feature=torch.randn(nk, 8, generator=g).to(cuda), edge_index=ek.to(cuda),
                                edge_feature=torch.randn(ek.size(1), 4, generator=g).to(cuda)))
    b = collate(graphs)
    off = 0
    pos = 0
    for gr in graphs:
        e = gr.edge_index.size(1)
        assert torch.equal(b.edge_index[:, pos:pos + e], gr.edge_index + off)
        assert torch.equal(b.edge_feature[pos:pos + e], gr.edge_feature)
        off, pos = off + gr.num_nodes, pos + e
    for stage in ('stack', 'skipsum'):
        reset_cfg()
        cfg.gnn.layer_type, cfg.gnn.stage_type, cfg.gnn.agg, cfg.dataset.edge_dim = 'generaledgeconv', stage, 'max', 4
        cfg.gnn.layers_mp, cfg.gnn.dim_inner, cfg.gnn.layers_pre_mp = 2, 8, 0
        outs = []
        for _ in range(2):
            torch.manual_seed(0)
            model = GNN(8, 3).to(cuda)
            taps = []
            conv0 = [m for m in model.modules() if isinstance(m, GeneralEdgeConvLayer)][0]
            conv0.register_forward_hook(lambda m, i, o: taps.append(o.detach()))
            batch = Batch(b.node_feature.clone(), b.edge_index, edge_feature=b.edge_feature)
            y, _ = model(batch)
            y.square().sum().backward()
            outs.append((y.detach(), conv0.linear_msg.weight.grad.clone()))
        assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
        p = {k: v.detach().double() for k, v in conv0.named_parameters()}
        want = E.general_edge_conv(b.node_feature.double(), b.edge_index, b.edge_feature.double(),
                                   p['linear_msg.weight'], p.get('linear_self.weight'), p.get('bias'), 'max', 'single',
                                   'concat')
        mag = E.general_edge_conv(b.node_feature.double().abs(), b.edge_index, b.edge_feature.double().abs(),
                                  p['linear_msg.weight'].abs(), p['linear_self.weight'].abs(), None, 'add', 'single',
                                  'concat')
        check_arrays(f'model {stage} first layer', {'out': taps[0]}, {'out': want}, {'out': mag})
        assert torch.isfinite(y).all()


@pytest.mark.parametrize('agg', ['add', 'max'])
def test_full_size(cuda, agg):
    """The products-shaped graph of bench.py (seed 0), generaledgeconv 100 -> 128, edge_dim 16, U(-1, 1) edge features,
    msg_direction 'both', self_msg 'concat': one step against the chunked fp64 oracle on the device, the kernels that ran,
    and the step's memory peak (no [E, 128] float32 tensor)."""
    spec = bench.WORKLOADS['products_gcn']
    n, ei = bench.gen_graph(spec, cuda, seed=0)
    g = torch.Generator(device=cuda).manual_seed(1)
    x = torch.randn(n, 100, generator=g, device=cuda)
    gy = torch.randn(n, 128, generator=g, device=cuda)
    a = torch.rand(ei.size(1), 16, generator=g, device=cuda) * 2 - 1
    monkey_seg = ops.SELL_SEG
    ops.SELL_SEG = 256
    try:
        run = lambda: run_layer(cuda, ei, n, 100, 128, 16, agg, 'both', 'concat', True, x, a, gy)
        run()                                   # builds and caches the layout
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        (layer, out, gx, ga, arg), kern = kernels_of(run)
        peak = torch.cuda.max_memory_allocated() - base
        one = ei.size(1) * 128 * 4
        print(f'full size {agg}: step peak {peak / 2**30:.2f} GiB above inputs + layout (one [E, 128] fp32 = '
              f'{one / 2**30:.2f} GiB)')
        assert peak < one
        if agg == 'max':
            check_path('full size max', kern, {'edge_sell_max_kernel': 2, 'edge_max_winner_kernel': 1,
                                               'edge_max_wgrad_partial_kernel': 1, 'spmm_sell_max_bwd_kernel': 1,
                                               'max_mask_kernel': 1},
                       ('edge_row_max_kernel', 'spmm_sell_max_kernel'))
        else:
            check_path('full size add', kern, {'edge_row_reduce_kernel': 1, 'edge_rows_self_kernel': 2,
                                               'gather_rows_kernel': 1, 'spmm_sell_kernel': 2},
                       ('edge_sell_max_kernel', 'edge_row_max_kernel'))
        check_layer(f'full size {agg}', ei, n, layer, out, gx, ga, arg, x, a, gy, agg, 'both', 'concat')
    finally:
        ops.SELL_SEG = monkey_seg
        clear_cache()
