"""GraphGym's skip stages (cfg.gnn.stage_type = 'skipsum' / 'skipconcat', ref: graphgym/models/gnn.py GNNSkipBlock /
GNNSkipStage) on the device: the fused skip epilogue (gg_postops_skip_*_f32) against fp64 autograd, the fused block
against its own modules, whole stages against the fp64 oracle (oracle/stages.py) under the kernels' activation gates,
the profile of a fused block, 'stack' unchanged, the main_zd front door, and the PReLU fallback."""
import os

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from graphgym_b200 import functional as F_
from graphgym_b200 import ops
from graphgym_b200.config import cfg, reset_cfg
from oracle import layers as olayers
from oracle import max_agg
from oracle import stages
from util import FP32_TOL, powerlaw_graph, random_graph, rel_err

pytestmark = pytest.mark.gpu
ACTS = {ops.ACT_RELU: F.relu, ops.ACT_LRELU: lambda t: F.leaky_relu(t, 0.25)}


@pytest.fixture(autouse=True)
def _fresh_cfg():
    reset_cfg()
    yield
    reset_cfg()


# ---- the epilogue op ---------------------------------------------------------------------------------------------
def _bn_pair(f, g, mode):
    """(float32 module, float64 twin) in 'train' / 'eval' mode, or (None, None)."""
    if mode == 'none':
        return None, None
    bn64 = nn.BatchNorm1d(f, eps=1e-5, momentum=0.1).double()
    with torch.no_grad():
        bn64.weight.uniform_(0.5, 1.5, generator=g)
        bn64.bias.uniform_(-1, 1, generator=g)
        if mode == 'eval':
            bn64.running_mean.uniform_(-1, 1, generator=g)
            bn64.running_var.uniform_(0.5, 2, generator=g)
    bn = nn.BatchNorm1d(f, eps=1e-5, momentum=0.1)
    bn.load_state_dict({k: v.float() if v.is_floating_point() else v for k, v in bn64.state_dict().items()})
    if mode == 'eval':
        bn.eval(), bn64.eval()
    return bn, bn64


def _epilogue_ref(y, res, gy, bn64, skip, act, l2):
    y = y.double().requires_grad_(True)
    res = res.double().requires_grad_(True)
    a = bn64(y) if bn64 is not None else y
    r = ACTS[act](a + res if skip == ops.SKIP_SUM else torch.cat([res, a], 1))
    o = F.normalize(r, p=2, dim=1) if l2 else r
    o.backward(gy.double())
    return o.detach(), y.grad, res.grad


@pytest.mark.parametrize('n,f', [(1000, 128), (777, 100), (5000, 33), (64, 256), (3, 8), (300, 1024)])
@pytest.mark.parametrize('skip,p', [(ops.SKIP_SUM, 0), (ops.SKIP_PREFIX, 1), (ops.SKIP_PREFIX, 16),
                                    (ops.SKIP_PREFIX, 100), (ops.SKIP_PREFIX, 384)])
@pytest.mark.parametrize('act', [ops.ACT_RELU, ops.ACT_LRELU])
def test_epilogue_against_fp64_autograd(cuda, n, f, skip, p, act):
    for bn_mode in ('train', 'eval', 'none'):
        for l2 in (False, True):
            g = torch.Generator().manual_seed(n + f + p)
            y = torch.randn(n, f, generator=g) * 3 + 50 * torch.randn(f, generator=g)   # |mean| >> std columns
            w = f if skip == ops.SKIP_SUM else p
            res = torch.randn(n, w, generator=g)
            gy = torch.randn(n, w + (f if skip == ops.SKIP_PREFIX else 0), generator=g)
            bn, bn64 = _bn_pair(f, g, bn_mode)
            want, want_dy, want_dres = _epilogue_ref(y, res, gy, bn64, skip, act, l2)
            if bn is not None:
                bn = bn.to(cuda)
            yc = y.to(cuda).requires_grad_(True)
            rc = res.to(cuda).requires_grad_(True)
            out = F_.skip_post_ops(yc, rc, skip, bn, bn_mode != 'eval', act, 0.25, l2)
            out.backward(gy.to(cuda))
            case = (bn_mode, l2)
            assert out.shape == want.shape, case
            assert rel_err(out, want) < FP32_TOL, case
            # gradients: gates of pre-activations within rounding of zero may differ (test_postops_gpu's band)
            assert rel_err(yc.grad, want_dy) < 2e-5, case
            assert rel_err(rc.grad, want_dres) < 2e-5, case
            if bn is not None:
                assert rel_err(bn.weight.grad, bn64.weight.grad) < FP32_TOL, case
                assert rel_err(bn.bias.grad, bn64.bias.grad) < FP32_TOL, case
                assert rel_err(bn.running_mean, bn64.running_mean) < FP32_TOL, case
                assert rel_err(bn.running_var, bn64.running_var) < FP32_TOL, case
                assert int(bn.num_batches_tracked) == int(bn64.num_batches_tracked), case


@pytest.mark.parametrize('skip', [ops.SKIP_SUM, ops.SKIP_PREFIX])
def test_all_zero_rows_l2(cuda, skip):
    """ReLU kills a whole row: F.normalize returns 0 / eps = 0, gradient 0 (both the y and the res side)."""
    y = torch.full((10, 16), -1.0)
    y[3] = 1.0
    res = torch.full((10, 16 if skip == ops.SKIP_SUM else 8), -0.5)
    res[3] = 0.5
    yc = y.to(cuda).requires_grad_(True)
    rc = res.to(cuda).requires_grad_(True)
    out = F_.skip_post_ops(yc, rc, skip, None, True, ops.ACT_RELU, 0.0, True)
    out.backward(torch.ones_like(out))
    assert torch.isfinite(out).all() and torch.isfinite(yc.grad).all() and torch.isfinite(rc.grad).all()
    assert float(out[0].abs().max()) == 0.0 and abs(float(out[3].norm()) - 1.0) < 1e-6
    assert float(yc.grad[0].abs().max()) == 0.0 and float(rc.grad[0].abs().max()) == 0.0
    want, want_dy, want_dres = _epilogue_ref(y, res, torch.ones(out.shape), None, skip, ops.ACT_RELU, True)
    assert rel_err(out, want) < FP32_TOL and rel_err(yc.grad, want_dy) < FP32_TOL
    assert rel_err(rc.grad, want_dres) < FP32_TOL


# ---- blocks and stages -------------------------------------------------------------------------------------------
def _set_cfg(stage_type, skip_every=1, act='relu'):
    reset_cfg()
    cfg.gnn.stage_type, cfg.gnn.skip_every, cfg.gnn.act = stage_type, skip_every, act


@pytest.mark.parametrize('layer_type', ['generalconv', 'gcnidconv'])
@pytest.mark.parametrize('skip_every', [1, 2])
@pytest.mark.parametrize('stage_type', ['skipsum', 'skipconcat'])
def test_block_fused_equals_unfused_modules(cuda, stage_type, skip_every, layer_type):
    """GNNSkipBlock with the fused epilogue == the same block running its nn modules one by one (train mode, with the
    stage's L2), the pattern of test_postops_gpu.test_general_layer_fused_equals_unfused_modules."""
    from graphgym_b200.models.gnn import GNNSkipBlock
    from graphgym_b200.models.layer import Batch
    n, d = 2000, 48
    ei = random_graph(1, n, 12000).to(cuda)
    ids = torch.arange(0, n, 10, device=cuda)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(n, d, generator=g).to(cuda)
    w_out = d if stage_type == 'skipsum' else 2 * d
    gy = torch.randn(n, w_out, generator=g).to(cuda)
    res, keys = {}, {}
    for fused in (True, False):
        _set_cfg(stage_type, skip_every)
        cfg.b200.fused_postops = fused
        torch.manual_seed(0)
        block = GNNSkipBlock(d, d, skip_every, layer_type, has_l2norm=True).to(cuda)
        xg = x.clone().requires_grad_(True)
        out = block(Batch(xg, ei, ids)).node_feature
        out.backward(gy)
        bns = [m for m in block.modules() if isinstance(m, nn.BatchNorm1d)]
        res[fused] = ([out.detach(), xg.grad] + [p.grad for _, p in sorted(block.named_parameters())] +
                      [b.running_mean.clone() for b in bns] + [b.running_var.clone() for b in bns])
        keys[fused] = sorted(block.state_dict())
        assert int(bns[-1].num_batches_tracked) == 1
    assert keys[True] == keys[False]
    assert len(res[True]) == len(res[False])
    for i, (a, b) in enumerate(zip(res[True], res[False])):
        assert rel_err(a, b) < 2e-5, i


def _stage_against_oracle(cuda, stage, x, ei, ids, conv64, mode, act=('relu',)):
    """Run ``stage`` block by block (its own forward), read every activation gate it took, and compare out, dx and every
    parameter gradient with oracle.stages under those gates."""
    from graphgym_b200.models.layer import Batch
    gy = torch.randn(x.size(0), stage.dim_out, generator=torch.Generator().manual_seed(1)).to(cuda)
    xg = x.clone().requires_grad_(True)
    b = Batch(xg, ei, ids)
    gates, hooks = [], []
    for blk in stage.children():
        for lay in list(blk.f)[:-1]:
            hooks.append(lay.register_forward_hook(lambda m, i, o: gates.append((o.node_feature.detach() > 0).cpu())))
    for blk in stage.children():
        b = blk(b)
        gates.append((b.node_feature.detach() > 0).cpu())
    for h in hooks:
        h.remove()
    out = b.node_feature
    out.backward(gy)
    P = {k: v.detach().cpu().double().requires_grad_(True) for k, v in stage.named_parameters()}
    blocks = []
    for i, blk in enumerate(stage.children()):
        convs, bns = [], []
        for j in range(len(blk.f)):
            pre = 'block{}.f.{}.'.format(i, j)
            convs.append(lambda h, pre=pre: conv64(h, P, pre + 'layer.model.'))
            bns.append((P[pre + 'post_layer.0.weight'], P[pre + 'post_layer.0.bias']))
        blocks.append((convs, bns))
    k = len(blocks[0][0])
    per_block = [gates[i * k:(i + 1) * k] for i in range(len(blocks))]
    if act[0] == 'prelu':   # every PReLU module has its own weight: the inner layers' post_layer.1, the block's act
        act = [[('prelu', P['block{}.f.{}.post_layer.1.weight'.format(i, j)]) for j in range(k - 1)] +
               [('prelu', P['block{}.act.weight'.format(i)])] for i in range(len(blocks))]
    x64 = x.detach().cpu().double().requires_grad_(True)
    tap = []
    h = stages.skip_stage(x64, blocks, mode, act, True, per_block, tap)
    for pre, gate in zip(tap, gates):
        # a pre-activation within rounding of zero may gate differently in fp32 and fp64; such disagreements must be tiny
        flipped = (pre > 0) != gate
        if flipped.any():
            assert float(pre[flipped].abs().max() / pre.abs().max()) < 1e-4
    h.backward(gy.cpu().double())
    assert rel_err(out.detach(), h.detach()) < 5e-5          # several BN + activation layers deep: 1e-5 per layer
    assert rel_err(xg.grad, x64.grad) < 2e-4
    for name, v in stage.named_parameters():
        assert rel_err(v.grad, P[name].grad) < 2e-4, name


def _general64(h, P, pre, ei):
    return max_agg.general_conv(h, ei, P[pre + 'weight'], P[pre + 'weight_self'])


@pytest.mark.parametrize('stage_type', ['skipsum', 'skipconcat'])
def test_powerlaw_generalconv_stage_matches_the_fp64_oracle(cuda, stage_type):
    from graphgym_b200.models.gnn import GNNSkipStage
    n, d = 30000, 32
    ei = powerlaw_graph(7, n, 8, max_deg=2000)
    _set_cfg(stage_type, skip_every=2)
    torch.manual_seed(0)
    stage = GNNSkipStage(d, d, 4, 'generalconv').to(cuda)
    x = torch.randn(n, d, generator=torch.Generator().manual_seed(2)).to(cuda)
    _stage_against_oracle(cuda, stage, x, ei.to(cuda), None, lambda h, P, pre: _general64(h, P, pre, ei), stage_type)


@pytest.mark.parametrize('stage_type', ['skipsum', 'skipconcat'])
def test_cfg_a_gcnidconv_stage_matches_the_fp64_oracle(cuda, golden_dir, stage_type):
    """The Cfg-A ego batch of test_main_zd_gpu.test_cfg_a_stack_matches_the_fp64_oracle, two skip blocks of gcnidconv on
    random inputs."""
    import numpy as np
    from graphgym_b200.models import transform as gtr
    from graphgym_b200.models.gnn import GNNSkipStage
    d_ = np.load(os.path.join(golden_dir, 'scalefree16.npz'))
    ei = torch.from_numpy(d_['edge_index']).to(cuda)
    gp = torch.from_numpy(d_['graph_ptr']).to(cuda).int()
    res = gtr.ego_nets_batch(ei, int(d_['graph_ptr'][-1]), 3, gp)
    eo, ids, n_out = res['edge_index'], res['node_id_index'], res['num_nodes']
    eo_c, ids_c = eo.cpu(), ids.cpu()
    _set_cfg(stage_type, skip_every=1)
    torch.manual_seed(0)
    stage = GNNSkipStage(32, 32, 2, 'gcnidconv').to(cuda)
    x = torch.randn(n_out, 32, generator=torch.Generator().manual_seed(3)).to(cuda)

    def conv64(h, P, pre):
        return olayers.gcn_idconv(h, eo_c, ids_c, P[pre + 'weight'], P[pre + 'weight_id'], None)
    _stage_against_oracle(cuda, stage, x, eo, ids, conv64, stage_type)


@pytest.mark.parametrize('stage_type', ['skipsum', 'skipconcat'])
def test_fused_block_profile_has_no_torch_epilogue(cuda, monkeypatch, stage_type):
    """One fused skip block forward + backward in train mode: the BN, the skip (+ / cat), the activation and the L2 run as
    the gg post-op kernels (the skip entry points and the launches they make), with no aten add / cat / relu /
    leaky_relu / norm / div over [N, *] tensors.  The input needs no gradient here: a block input that does gets its two
    gradients (the conv's and the skip's) summed by autograd at the fan-out, in any implementation, which is not part of
    the epilogue."""
    from torch.profiler import ProfilerActivity, profile
    from graphgym_b200.models.gnn import GNNSkipBlock
    from graphgym_b200.models.layer import Batch
    n, d = 4096, 64
    ei = random_graph(2, n, 30000).to(cuda)
    x = torch.randn(n, d, device=cuda)
    _set_cfg(stage_type, skip_every=1)
    block = GNNSkipBlock(d, d, 1, 'generalconv', has_l2norm=True).to(cuda)

    def step():
        out = block(Batch(x, ei)).node_feature
        out.backward(torch.ones_like(out))

    for _ in range(2):   # layouts, module loads
        step()
    torch.cuda.synchronize()
    # the torch ops, with their input shapes (host-side profile) ...
    with profile(activities=[ProfilerActivity.CPU], record_shapes=True) as prof:
        step()
        torch.cuda.synchronize()
    banned = {'aten::add', 'aten::add_', 'aten::cat', 'aten::relu', 'aten::relu_', 'aten::leaky_relu',
              'aten::threshold_backward', 'aten::leaky_relu_backward', 'aten::norm', 'aten::linalg_vector_norm',
              'aten::div', 'aten::div_'}
    evts = prof.key_averages(group_by_input_shape=True)
    bad = [(e.key, e.input_shapes) for e in evts
           if e.key in banned and any(s and s[0] == n for s in e.input_shapes)]
    assert not bad, bad
    keys = [e.key for e in prof.key_averages()]
    assert '_SkipPostOps' in keys and any('_SkipPostOpsBackward' in k for k in keys), keys
    # ... and the gg entry points the step called (the skip epilogue, not the plain post-ops), with the kernels each one
    # launched (the library's own launch counter: statistics 2, epilogue forward 1, backward 3 — column sums, their
    # fixed-order merge, apply)
    calls = {}

    def counted(fn, key):
        def run(*a, **k):
            before = ops.launch_count()
            r = fn(*a, **k)
            calls[key] = calls.get(key, 0) + ops.launch_count() - before
            return r
        return run
    for key in ('bn_stats', 'postops_skip_fwd', 'postops_skip_bwd', 'postops_fwd', 'postops_bwd'):
        monkeypatch.setattr(ops, key, counted(getattr(ops, key), key))
    step()
    torch.cuda.synchronize()
    assert calls == {'bn_stats': 2, 'postops_skip_fwd': 1, 'postops_skip_bwd': 3}, calls


def test_stack_stage_type_is_the_stack_stage(cuda):
    """stage_type = 'stack' builds exactly the GNNStackStage of before: bitwise the same output and gradients."""
    from graphgym_b200.models.gnn import GNN, GNNStackStage
    from graphgym_b200.models.layer import Batch
    reset_cfg()
    cfg.gnn.layers_pre_mp, cfg.gnn.layers_mp, cfg.gnn.dim_inner = 0, 2, 32
    n, d = 3000, 32
    ei = random_graph(4, n, 20000).to(cuda)
    x = torch.randn(n, d, generator=torch.Generator().manual_seed(4)).to(cuda)
    torch.manual_seed(0)
    m = GNN(d, 6).to(cuda)
    assert type(m.mp) is GNNStackStage
    torch.manual_seed(0)
    stage = GNNStackStage(d, 32, 2).to(cuda)
    stage.load_state_dict(m.mp.state_dict())
    assert sorted(stage.state_dict()) == sorted(k[3:] for k in m.state_dict() if k.startswith('mp.'))
    x1, x2 = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    pred, _ = m(Batch(x1, ei))
    h = stage(Batch(x2, ei)).node_feature
    pred2, _ = m.post_mp(Batch(h, ei))
    assert torch.equal(pred, pred2)
    gy = torch.randn(pred.shape, generator=torch.Generator().manual_seed(5)).to(cuda)
    head_w = m.post_mp.layer_post_mp.weight
    pred.backward(gy)
    grads = {k: v.grad.clone() for k, v in m.mp.named_parameters()}
    dx1 = x1.grad.clone()
    head_w.grad = None
    pred2.backward(gy)
    assert torch.equal(dx1, x2.grad)
    for k, v in stage.named_parameters():
        assert torch.equal(grads[k], v.grad), k


@pytest.mark.parametrize('stage_type', ['skipsum', 'skipconcat'])
def test_driver_trains_a_skip_stage_on_the_scalefree_fixture(cuda, golden_dir, tmp_path, stage_type):
    from graphgym_b200 import main_zd
    src = open(os.path.join(golden_dir, 'idgcn_node_scalefree.yaml')).read()
    assert '  stage_type: stack\n' in src
    path = tmp_path / 'skip.yaml'
    path.write_text(src.replace('  stage_type: stack\n', '  stage_type: {}\n'.format(stage_type)))
    graphs = os.path.join(golden_dir, 'scalefree16.npz')
    r = main_zd.main(['--cfg', str(path), '--graphs', graphs, '--epochs', '8'])[0]
    assert r['layer_type'] == 'Tfg-idgcn' and r['graphs'] == 16 and r['labels'] == 10
    assert r['train_loss'] == r['train_loss'] and r['train_loss'] < 2.3     # finite, below ln(10): it learns
    first = main_zd.main(['--cfg', str(path), '--graphs', graphs, '--epochs', '1'])[0]
    assert r['train_loss'] < first['train_loss']


def test_prelu_skipsum_runs_the_modules_and_matches_the_oracle(cuda, monkeypatch):
    from graphgym_b200.models.gnn import GNNSkipStage

    def no_fused(*a, **k):
        raise AssertionError('PReLU must not take the fused skip epilogue')
    monkeypatch.setattr(F_, 'skip_post_ops', no_fused)
    n, d = 5000, 32
    ei = random_graph(6, n, 40000)
    _set_cfg('skipsum', skip_every=2, act='prelu')
    torch.manual_seed(0)
    stage = GNNSkipStage(d, d, 2, 'generalconv').to(cuda)
    assert isinstance(stage.block0.act, nn.PReLU)
    x = torch.randn(n, d, generator=torch.Generator().manual_seed(8)).to(cuda)
    _stage_against_oracle(cuda, stage, x, ei.to(cuda), None, lambda h, P, pre: _general64(h, P, pre, ei), 'skipsum',
                          act=('prelu',))
