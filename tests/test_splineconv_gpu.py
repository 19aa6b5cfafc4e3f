"""splineconv on the GPU (csrc/spline_agg.cu, functional.spline_aggregate).

Kernel level, on a power-law graph with hub rows split into virtual rows, isolated nodes, duplicate edges and self loops:
spread and blend on the CSR and the CSC against fp64 at widths that cover the sliced-ELL path, its column tiles and the
warp-per-row path, bitwise repeatable.  Layer level: both factorisations, bias on and off, out and every gradient (the
pseudo-coordinate's too) against oracle.splineconv in fp64, with u at 0 and 1, in (-1, 0) and in (1, 3).  Batches: a
collated batch with 1-D edge features and a two-layer GNN.  Full size: the products-shaped graph, 100 -> 128, against the
chunked fp64 oracle on the device, with the kernels that ran and the memory peak."""
import pytest
import torch

import bench
from graphgym_b200 import ops
from graphgym_b200.config import cfg, reset_cfg
from graphgym_b200.graph import clear_cache, get_layout
from graphgym_b200.models.layer import Batch, _SplineConvLayer
from oracle import splineconv as S
from test_fullsize_step_parity_gpu import check_arrays, check_path, kernels_of
from test_max_agg_gpu import max_graph

pytestmark = pytest.mark.gpu

FS = [1, 3, 16, 64, 100, 128, 200, 256]


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


def pseudo(e, seed, dev):
    """0 and 1 exactly, values in (-1, 0) and (1, 3), the rest U(0, 1)."""
    g = torch.Generator(device=dev).manual_seed(seed)
    u = torch.rand(e, generator=g, device=dev)
    k = torch.arange(e, device=dev) % 8
    u = torch.where(k == 1, torch.zeros_like(u), u)
    u = torch.where(k == 2, torch.ones_like(u), u)
    u = torch.where(k == 3, -u, u)
    u = torch.where(k == 4, 1 + 2 * u, u)
    return u


def fp64_walk(rows, nbr, n, u, w, xs, scale):
    """sum over the edges of row r of w_e (c0_e xs[0][nbr] + c1_e xs[1][nbr]) * scale[r], and the same on magnitudes."""
    c = S.coefficients(u.double()) * w.view(-1, 1)
    out = torch.zeros(n, xs[0].size(1), dtype=torch.float64, device=u.device)
    mag = torch.zeros_like(out)
    for k in range(2):
        out.index_add_(0, rows, c[:, k:k + 1] * xs[k].double()[nbr])
        mag.index_add_(0, rows, c[:, k:k + 1].abs() * xs[k].double().abs()[nbr])
    return out * scale.view(-1, 1), mag * scale.view(-1, 1)


def sides(ei, n, lay):
    """(layout, its rows, its gathered ends, slot weights of the layout or None, mean flag, fp64 per-edge weight, row
    scale) of the CSR forward (mean) and the CSC backward (1/indeg(target) per slot)."""
    dev = ei.device
    deg = torch.zeros(n, dtype=torch.float64, device=dev).index_add_(0, ei[1], torch.ones(ei.size(1), dtype=torch.float64,
                                                                                         device=dev))
    inv = 1.0 / deg.clamp(min=1)
    ones_e = torch.ones(ei.size(1), dtype=torch.float64, device=dev)
    return {'csr': (lay.csr, ei[1], ei[0], None, True, ones_e, inv),
            'csc': (lay.csc, ei[0], ei[1], lay.weights('mean')[1], False, inv[ei[1]], torch.ones_like(inv))}


@pytest.mark.parametrize('f', FS)
def test_spread_and_blend(cuda, graph, f):
    n, ei = graph
    ei = ei.to(cuda)
    lay = get_layout(ei, n, ops.LOOPS_KEEP)
    g = torch.Generator(device=cuda).manual_seed(f)
    u = pseudo(ei.size(1), f, cuda)
    x = torch.randn(n, f, generator=g, device=cuda)
    y = torch.randn(n, 2 * f, generator=g, device=cuda)
    res = torch.randn(n, f, generator=g, device=cuda)
    bias = torch.randn(f, generator=g, device=cuda)
    paths = ('row',) if f % 4 else ('sell', 'row')
    for side, (csr, rows, nbr, w_slot, mean, w_e, scale) in sides(ei, n, lay).items():
        s0, m0 = fp64_walk(rows, nbr, n, u, w_e, (x, torch.zeros_like(x)), scale)
        s1, m1 = fp64_walk(rows, nbr, n, u, w_e, (torch.zeros_like(x), x), scale)
        want, mag = torch.cat([s0, s1], 1), torch.cat([m0, m1], 1)
        bw, bmag = fp64_walk(rows, nbr, n, u, w_e, (y[:, :f], y[:, f:]), scale)
        r_b = (res, bias) if side == 'csr' else (None, None)
        if side == 'csr':
            bw, bmag = bw + res.double() + bias.double(), bmag + res.double().abs() + bias.double().abs()
        for algo in paths:
            got = ops.spline_spread(csr, x, u, w_slot, mean, algo=algo)
            assert torch.equal(got, ops.spline_spread(csr, x, u, w_slot, mean, algo=algo)), (side, algo)
            gb = ops.spline_blend(csr, y, u, w_slot, mean, r_b[0], r_b[1], algo=algo)
            assert torch.equal(gb, ops.spline_blend(csr, y, u, w_slot, mean, r_b[0], r_b[1], algo=algo)), (side, algo)
            check_arrays(f'spline f={f} {side} {algo}', {'spread': got, 'blend': gb}, {'spread': want, 'blend': bw},
                         {'spread': mag, 'blend': bmag})


def du_magnitude(x, ei, n, w, gy):
    """sum_k <|g_i| |W_k|^T / indeg(i), |x_j|> per edge: a bound on the terms behind du_e."""
    src, tgt = ei
    deg = torch.zeros(n, dtype=torch.float64, device=x.device).index_add_(0, tgt, torch.ones_like(tgt, dtype=torch.float64))
    inv = (1.0 / deg.clamp(min=1)).view(-1, 1)
    return sum(((gy.abs() @ w[k].abs().t()) * inv)[tgt].mul(x.abs()[src]).sum(1) for k in range(2))


def run_layer(cuda, ei, n, fin, fout, bias, x, u, gy, seed=0):
    torch.manual_seed(seed)
    layer = _SplineConvLayer(fin, fout, bias=bias).to(cuda)
    xg = x.detach().clone().requires_grad_(True)
    ug = u.detach().clone().requires_grad_(u.requires_grad)
    out = layer(xg, ei, ug)
    out.backward(gy)
    return layer, out.detach(), xg.grad, ug.grad


def check_layer(tag, ei, n, layer, out, gx, gu, x, u, gy, chunk=1 << 22):
    with torch.no_grad():
        p = {k: v.detach().double() for k, v in layer.named_parameters()}
        b = p.get('bias')
        ref = S.spline_conv_step(x.double(), ei, u.double(), p['weight'], p['root'], b, gy.double(), chunk=chunk)
        ab = lambda t: None if t is None else t.abs()
        mag = S.spline_conv_step(x.double().abs(), ei, u.double(), p['weight'].abs(), p['root'].abs(), ab(b),
                                 gy.double().abs(), chunk=chunk)       # the coefficients are never negative
        got = {'out': out, 'dx': gx, 'dweight': layer.weight.grad, 'droot': layer.root.grad}
        want = {'out': ref[0], 'dx': ref[1], 'dweight': ref[3], 'droot': ref[4]}
        bound = {'out': mag[0], 'dx': mag[1], 'dweight': mag[3], 'droot': mag[4]}
        if b is not None:
            got['db'], want['db'], bound['db'] = layer.bias.grad, ref[5], mag[5]
        if gu is not None:
            assert gu.shape == u.shape
            got['du'], want['du'] = gu, ref[2]
            bound['du'] = du_magnitude(x.double(), ei, n, p['weight'], gy.double()).view(u.shape)
        check_arrays(tag, got, want, bound)


@pytest.mark.parametrize('fin,fout', [(16, 64), (64, 16), (32, 32), (3, 5), (7, 2), (100, 128), (200, 64)])
@pytest.mark.parametrize('bias', [False, True])
def test_layer(cuda, graph, fin, fout, bias):
    n, ei = graph
    ei = ei.to(cuda)
    g = torch.Generator(device=cuda).manual_seed(fin * 1000 + fout)
    x = torch.randn(n, fin, generator=g, device=cuda)
    gy = torch.randn(n, fout, generator=g, device=cuda)
    for shape in ('flat', 'column'):
        u = pseudo(ei.size(1), fin + fout, cuda)
        u = (u if shape == 'flat' else u.view(-1, 1)).requires_grad_(True)
        tag = f'layer {fin}->{fout} bias={bias} u {shape}'
        layer, out, gx, gu = run_layer(cuda, ei, n, fin, fout, bias, x, u, gy)
        check_layer(tag, ei, n, layer, out, gx, gu, x, u.detach(), gy)
        layer2, out2, gx2, gu2 = run_layer(cuda, ei, n, fin, fout, bias, x, u, gy)
        assert torch.equal(out, out2) and torch.equal(gx, gx2) and torch.equal(gu, gu2), tag
        assert torch.equal(layer.weight.grad, layer2.weight.grad) and torch.equal(layer.root.grad, layer2.root.grad), tag
    # raw dataset features do not require a gradient: none is computed
    _, _, _, gu = run_layer(cuda, ei, n, fin, fout, bias, x, pseudo(ei.size(1), 1, cuda), gy)
    assert gu is None


def test_collate_and_model(cuda):
    """Small graphs with 1-D edge features through loader.collate (they become an [E, 1] column) and a GNN of two
    splineconv layers under stack and skipsum: forward + backward, bitwise repeatable, the first layer against fp64."""
    from graphgym_b200.loader import GraphData, collate
    from graphgym_b200.models.gnn import GNN
    g = torch.Generator().manual_seed(5)
    graphs = []
    for k in range(6):
        nk = 20 + 7 * k
        ek = torch.randint(0, nk, (2, 3 * nk), generator=g)
        graphs.append(GraphData(node_feature=torch.randn(nk, 8, generator=g).to(cuda), edge_index=ek.to(cuda),
                                edge_feature=torch.rand(ek.size(1), generator=g).to(cuda)))
    b = collate(graphs)
    assert b.edge_feature.shape == (b.edge_index.size(1), 1)
    assert torch.equal(b.edge_feature.view(-1), torch.cat([gr.edge_feature for gr in graphs]))
    for stage in ('stack', 'skipsum'):
        reset_cfg()
        cfg.gnn.layer_type, cfg.gnn.stage_type = 'splineconv', stage
        cfg.gnn.layers_mp, cfg.gnn.dim_inner, cfg.gnn.layers_pre_mp = 2, 8, 0
        outs = []
        for _ in range(2):
            torch.manual_seed(0)
            model = GNN(8, 3).to(cuda)
            taps = []
            conv0 = [m for m in model.modules() if isinstance(m, _SplineConvLayer)][0]
            conv0.register_forward_hook(lambda m, i, o: taps.append(o.detach()))
            batch = Batch(b.node_feature.clone(), b.edge_index, edge_feature=b.edge_feature)
            y, _ = model(batch)
            y.square().sum().backward()
            outs.append((y.detach(), conv0.weight.grad.clone(), conv0.root.grad.clone()))
        assert all(torch.equal(p, q) for p, q in zip(outs[0], outs[1]))
        p = {k: v.detach().double() for k, v in conv0.named_parameters()}
        want = S.spline_conv(b.node_feature.double(), b.edge_index, b.edge_feature.double(), p['weight'], p['root'],
                             p.get('bias'))
        mag = S.spline_conv(b.node_feature.double().abs(), b.edge_index, b.edge_feature.double(), p['weight'].abs(),
                            p['root'].abs(), None if 'bias' not in p else p['bias'].abs())
        check_arrays(f'model {stage} first layer', {'out': taps[0]}, {'out': want}, {'out': mag})
        assert torch.isfinite(y).all()


def test_full_size(cuda):
    """The products-shaped graph of bench.py (seed 0), splineconv 100 -> 128 (aggregate first), U(0, 1) pseudo-coordinates:
    one step against the chunked fp64 oracle on the device, the kernels that ran, and the step's memory peak (no
    [E, 128] float32 tensor)."""
    spec = bench.WORKLOADS['products_gcn']
    n, ei = bench.gen_graph(spec, cuda, seed=0)
    g = torch.Generator(device=cuda).manual_seed(1)
    x = torch.randn(n, 100, generator=g, device=cuda)
    gy = torch.randn(n, 128, generator=g, device=cuda)
    u = torch.rand(ei.size(1), generator=g, device=cuda)
    ops.SELL_SEG = 256
    run = lambda: run_layer(cuda, ei, n, 100, 128, True, x, u, gy)
    run()                                   # builds and caches the layout
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    (layer, out, gx, gu), kern = kernels_of(run)
    peak = torch.cuda.max_memory_allocated() - base
    one = ei.size(1) * 128 * 4
    print(f'full size: step peak {peak / 2**30:.2f} GiB above inputs + layout (one [E, 128] fp32 = {one / 2**30:.2f} GiB)')
    assert peak < one
    # [P0 | P1 | x] [W0; W1; root] and g [W0 | W1]^T on the multi-segment tensor-core GEMM, g root^T and x^T g on the
    # persistent ones, P^T g (K = 200) on the split-K tensor-core kernel
    check_path('full size', kern, {'spline_sell_kernel': 2, 'tc_gemm_kernel': 2, 'tc_gemm_persist_kernel': 1,
                                   'tc_gemm_tn_kernel': 1, 'tc_gemm_tn_persist_kernel': 1},
               ('spline_row_kernel', 'spline_du_kernel', 'id_gemm_kernel', 'gemm_tn_kernel'))
    assert gu is None
    check_layer('full size 100->128', ei, n, layer, out, gx, None, x, u, gy)
