"""Max aggregation on the GPU (csrc/spmm_max.cu, functional._AggregateMax, generalconv with cfg.gnn.agg = 'max').

Op level: out and arg equal the oracle evaluated in fp32 on the same inputs bit for bit (a message fl(w * h) is one
rounding on both sides), on hub rows split into virtual rows, isolated nodes, duplicate edges, self loops, all-negative
features (a padding entry must never win) and all-equal features (the first slot of every row wins); the backward within
1e-5 of the fp64 masked sum under the same arg, bitwise repeatable.  Layer level: generalconv against oracle.max_agg.general_conv
in fp64, gradients under the kernel's arg with every disagreement of the arg-max shown to be a near-tie.  Full size: the
products-shaped graph, 100 -> 128, against the chunked fp64 oracle on the device."""
import pytest
import torch

import bench
from graphgym_b200 import functional as F_
from graphgym_b200 import ops
from graphgym_b200.config import cfg, reset_cfg
from graphgym_b200.contrib.layer.generalconv import GeneralConvLayer
from graphgym_b200.graph import clear_cache, get_layout
from oracle import max_agg as M
from oracle import pyg_utils as U
from test_fullsize_step_parity_gpu import check_arrays, check_path, kernels_of
from util import FP32_TOL, powerlaw_graph

pytestmark = pytest.mark.gpu

WIDTHS = [1, 3, 16, 36, 128, 200, 256]


def max_graph(seed=0):
    """Power-law graph with hub rows, 150 isolated nodes, duplicate edges and self loops."""
    n0 = 3000
    ei = powerlaw_graph(seed, n0, 12)
    loops = torch.arange(0, n0, 37)
    ei = torch.cat([ei, ei[:, :700], torch.stack([loops, loops])], dim=1)
    return n0 + 150, ei


def edited_ids(csr, ei, policy):
    """CSR slot -> edge id in the edited edge list the oracle aggregates (LOOPS_KEEP: the edge list itself;
    LOOPS_ADD_REMAINING: the non-loop edges in order, then one loop per node)."""
    perm = csr.perm.long()
    if policy == ops.LOOPS_KEEP:
        return perm
    ei = ei.to(perm.device)
    keep = ei[0] != ei[1]
    rank = torch.cumsum(keep.long(), 0) - 1
    e = ei.size(1)
    return torch.where(perm < e, rank[perm.clamp(max=e - 1)], int(keep.sum()) + (perm - e))


def edited_edges(ei, n, policy):
    if policy == ops.LOOPS_KEEP:
        return ei
    return U.add_remaining_self_loops(ei, None, 1, n)[0]


def to_edges(arg, ids):
    """kernel arg (CSR slots, -1) -> edge ids of the edited list (-1), on the arg's device."""
    a = arg.long()
    return torch.where(a >= 0, ids[a.clamp(min=0)], a)


def features(kind, n, f, seed):
    g = torch.Generator().manual_seed(seed)
    if kind == 'randn':
        return torch.randn(n, f, generator=g)
    if kind == 'negative':
        return -0.5 - torch.rand(n, f, generator=g)
    return torch.ones(n, f)


@pytest.fixture(scope='module')
def graph(cuda):
    return max_graph()


@pytest.mark.parametrize('f', WIDTHS)
@pytest.mark.parametrize('weighted', [False, True])
def test_forward_bit_exact(cuda, graph, monkeypatch, f, weighted):
    n, ei = graph
    monkeypatch.setattr(ops, 'SELL_SEG', 8)                 # hub rows split into many virtual rows: partials + fix-up
    policy = ops.LOOPS_ADD_REMAINING if weighted else ops.LOOPS_KEEP
    lay = get_layout(ei.to(cuda), n, policy)
    csr = lay.csr
    w_slot = lay.weights('gcn_src')[0] if weighted else None
    ids = edited_ids(csr, ei, policy)
    eie = edited_edges(ei, n, policy)
    w_edge = None
    if weighted:       # the kernel's own fp32 weights, in edge order
        w_edge = torch.empty(csr.num_slots)
        w_edge[ids.cpu()] = w_slot.cpu()
    paths = ('row',) if f % 4 else ('sell', 'row')
    for kind in ('randn', 'negative', 'equal'):
        x = features(kind, n, f, f)
        msg = x.index_select(0, eie[0])
        if weighted:
            msg = msg * w_edge.view(-1, 1)
        want_arg = M.scatter_argmax(msg, eie[1], n)
        want = M.gather_max(msg, want_arg)
        for algo in paths:
            out, arg = ops.spmm_max(csr, x.to(cuda), w_slot, algo=algo)
            assert torch.equal(to_edges(arg, ids).cpu(), want_arg), (kind, algo)
            assert torch.equal(out.cpu(), want), (kind, algo)
        if kind == 'equal' and not weighted:      # every row's arg is its first slot
            rp = csr.rowptr.long().cpu()
            nonempty = rp[1:] > rp[:-1]
            assert (arg.long().cpu()[nonempty] == rp[:-1][nonempty].view(-1, 1)).all()
            assert (arg.cpu()[~nonempty] == -1).all()
    # epilogue: + self_scale * x_self + bias, fused (same bits as the separate fp32 additions: fl(1 * x) = x)
    g = torch.Generator().manual_seed(99)
    x, xs, b = (torch.randn(n, f, generator=g), torch.randn(n, f, generator=g), torch.randn(f, generator=g))
    for algo in paths:
        base, _ = ops.spmm_max(csr, x.to(cuda), w_slot, algo=algo)
        out, _ = ops.spmm_max(csr, x.to(cuda), w_slot, xs.to(cuda), 1.0, b.to(cuda), algo=algo)
        assert torch.equal(out.cpu(), (base.cpu() + xs) + b), algo


@pytest.mark.parametrize('f', WIDTHS)
@pytest.mark.parametrize('weighted', [False, True])
def test_backward_masked_sum(cuda, graph, monkeypatch, f, weighted):
    n, ei = graph
    monkeypatch.setattr(ops, 'SELL_SEG', 8)
    policy = ops.LOOPS_ADD_REMAINING if weighted else ops.LOOPS_KEEP
    lay = get_layout(ei.to(cuda), n, policy)
    kind = 'gcn_src_max' if weighted else 'max'
    w_csr, w_csc = lay.weights(kind)
    gen = torch.Generator().manual_seed(f)
    x = torch.randn(n, f, generator=gen).to(cuda)
    g = torch.randn(n, f, generator=gen).to(cuda)
    paths = ('row',) if f % 4 else ('sell', 'row')
    outs = {a: ops.spmm_max(lay.csr, x, w_csr, algo=a) for a in paths}
    if len(paths) == 2:       # both forwards give the same bits
        assert torch.equal(outs['sell'][0], outs['row'][0]) and torch.equal(outs['sell'][1], outs['row'][1])
    arg = outs[paths[0]][1]
    # fp64 masked sum under that arg: dx[nbr[s]] += w[s] g[i] for s = arg[i, c]
    a = arg.long()
    ok = a >= 0
    s = a.clamp(min=0)
    src = lay.csr.nbr.long()[s]
    w = (w_csr.double()[s] if weighted else torch.ones_like(s, dtype=torch.float64)) * ok
    for scale in (0.0, 1.0):
        want = torch.zeros(n, f, dtype=torch.float64, device=cuda).scatter_add_(0, src, w * g.double())
        mag = torch.zeros(n, f, dtype=torch.float64, device=cuda).scatter_add_(0, src, w.abs() * g.double().abs())
        want, mag = want + scale * g.double(), mag + scale * g.double().abs()
        for algo in paths:
            got = ops.spmm_max_bwd(lay.csc, lay.csc2csr, g, arg, w_csc, scale, algo=algo)
            again = ops.spmm_max_bwd(lay.csc, lay.csc2csr, g, arg, w_csc, scale, algo=algo)
            assert torch.equal(got, again), algo                      # bitwise repeatable
            check_arrays(f'bwd f={f} w={weighted} scale={scale} {algo}', {'dx': got}, {'dx': want}, {'dx': mag})


def run_layer(cuda, ei, n, fin, fout, normalize, self_msg, bias, x, gy, seed=0):
    """generalconv with agg='max' on the device -> (layer, out, x.grad, kernel arg as edited edge ids)."""
    reset_cfg()
    cfg.gnn.agg, cfg.gnn.normalize_adj, cfg.gnn.self_msg = 'max', normalize, self_msg
    torch.manual_seed(seed)
    layer = GeneralConvLayer(fin, fout, bias=bias).to(cuda)
    if bias:
        with torch.no_grad():
            layer.bias.uniform_(-0.3, 0.3)
    reset_cfg()
    eid = ei.to(cuda)
    xg = x.detach().to(cuda).requires_grad_(True)
    out = layer(xg, eid)
    out.backward(gy.to(cuda))
    # the arg the layer used: same inputs, same deterministic kernels
    policy = ops.LOOPS_ADD_REMAINING if normalize else ops.LOOPS_KEEP
    lay = get_layout(eid, n, policy)
    h = F_.seg_linear([xg.detach()], [layer.weight.detach()], [(0, 0, False)])
    _, arg = ops.spmm_max(lay.csr, h, lay.weights('gcn_src_max' if normalize else 'max')[0])
    return layer, out.detach(), xg.grad, arg, lay, policy


def check_step(tag, cuda, ei, n, layer, out, gx, arg, lay, policy, x, gy, normalize, self_msg, chunk=1 << 22):
    """fp64 oracle: forward with its own arg-max, gradients under the kernel's, every arg disagreement a near-tie."""
    with torch.no_grad():
        _check_step(tag, ei, layer, out, gx, arg, lay, policy, x, gy, normalize, self_msg, chunk)


def _check_step(tag, ei, layer, out, gx, arg, lay, policy, x, gy, normalize, self_msg, chunk):
    dev = out.device
    p = {k: v.detach().double() for k, v in layer.named_parameters()}
    ws = p.get('weight_self')
    ei_d = ei.to(dev)
    x64, gy64 = x.to(dev).double(), gy.to(dev).double()
    arg_e = to_edges(arg, edited_ids(lay.csr, ei, policy))
    ref = M.general_conv_max_step(x64, ei_d, p['weight'], ws, p.get('bias'), gy64, normalize, self_msg, arg=arg_e,
                                        chunk=chunk)
    mag = M.general_conv_max_step(x64.abs(), ei_d, p['weight'].abs(), None if ws is None else ws.abs(),
                                        None if 'bias' not in p else p['bias'].abs(), gy64.abs(), normalize, self_msg,
                                        arg=arg_e, chunk=chunk)
    differ = ref[5] != arg_e
    # a different winner is a near-tie: its fp64 message lies within 1e-5 (of the row's scale) of the maximum
    assert ((ref[6].abs() <= FP32_TOL * mag[0].abs()) | ~differ).all(), f'{tag}: arg-max differs beyond a near-tie'
    print(f'{tag}: {int(differ.sum())} of {differ.numel()} arg-max entries differ from the fp64 oracle (near-ties)')
    got = {'out': out, 'dx': gx, 'dW': layer.weight.grad}
    want = {'out': ref[0], 'dx': ref[1], 'dW': ref[2]}
    bound = {'out': mag[0], 'dx': mag[1], 'dW': mag[2]}
    if ws is not None:
        got['dWself'], want['dWself'], bound['dWself'] = layer.weight_self.grad, ref[3], mag[3]
    if 'bias' in p:
        got['db'], want['db'], bound['db'] = layer.bias.grad, ref[4], mag[4]
    check_arrays(tag, got, want, bound)


@pytest.mark.parametrize('dims', [(16, 36), (7, 5)])      # sliced-ELL path / row path
@pytest.mark.parametrize('normalize', [False, True])
@pytest.mark.parametrize('self_msg', ['none', 'add', 'concat'])
@pytest.mark.parametrize('bias', [False, True])
def test_generalconv_max_layer(cuda, graph, dims, normalize, self_msg, bias):
    n, ei = graph
    fin, fout = dims
    g = torch.Generator().manual_seed(fin * 10 + fout)
    x, gy = torch.randn(n, fin, generator=g), torch.randn(n, fout, generator=g)
    clear_cache()
    layer, out, gx, arg, lay, policy = run_layer(cuda, ei, n, fin, fout, normalize, self_msg, bias, x, gy)
    check_step(f'generalconv {dims} norm={normalize} {self_msg} bias={bias}', cuda, ei, n, layer, out, gx, arg, lay,
               policy, x, gy, normalize, self_msg, chunk=5000)


def test_generalconv_max_all_ones_input(cuda, graph):
    """Cfg-A feeds node_feature = ones [N, 1]: on the first layer every message of a row is equal, so every column's
    gradient sits on the row's first edge."""
    n, ei = graph
    g = torch.Generator().manual_seed(7)
    x, gy = torch.ones(n, 1), torch.randn(n, 16, generator=g)
    clear_cache()
    layer, out, gx, arg, lay, policy = run_layer(cuda, ei, n, 1, 16, False, 'concat', True, x, gy)
    rp = lay.csr.rowptr.long()
    nonempty = rp[1:] > rp[:-1]
    assert (arg.long()[nonempty] == rp[:-1][nonempty].view(-1, 1)).all()
    assert (arg[~nonempty] == -1).all()
    check_step('generalconv all-ones', cuda, ei, n, layer, out, gx, arg, lay, policy, x, gy, False, 'concat')


@pytest.mark.parametrize('normalize', [False, True])
def test_generalconv_max_full_size(cuda, normalize):
    """The products-shaped graph of bench.py (seed 0), generalconv 100 -> 128 with agg='max', one forward + backward
    against the chunked fp64 oracle on the device; a profile of the step shows the sliced-ELL max kernels ran."""
    spec = bench.WORKLOADS['products_gcn']
    n, ei_d = bench.gen_graph(spec, cuda, seed=0)
    ei = ei_d.cpu()
    g = torch.Generator(device=cuda).manual_seed(1)
    x = torch.randn(n, 100, generator=g, device=cuda)
    gy = torch.randn(n, 128, generator=g, device=cuda)
    clear_cache()
    (layer, out, gx, arg, lay, policy), kern = kernels_of(
        lambda: run_layer(cuda, ei_d, n, 100, 128, normalize, 'concat', True, x, gy))
    check_path(f'full size norm={normalize}', kern, {'spmm_sell_max_kernel': 2, 'spmm_sell_max_bwd_kernel': 1},
               ('spmm_row_max_kernel', 'spmm_row_max_bwd_kernel', 'spmm_sell_kernel'))
    check_step(f'full size norm={normalize}', cuda, ei, n, layer, out, gx, arg, lay, policy, x, gy, normalize, 'concat')
    clear_cache()
