"""GraphGym's stage dimension (cfg.gnn.stage_type, ref: graphgym/models/gnn.py GNNSkipBlock / GNNSkipStage / stage_dict)
on the host: stage selection, the construction errors, block widths, state_dict keys, and the fp64 oracle
(oracle/stages.py) against a hand composition of the oracle layers."""
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from graphgym_b200.config import cfg, reset_cfg
from graphgym_b200.models import gnn
from oracle import layers as olayers
from oracle import max_agg
from oracle import stages
from util import random_graph


@pytest.fixture(autouse=True)
def _fresh_cfg():
    reset_cfg()
    yield
    reset_cfg()


def _gnn(stage_type, layers_mp=2, skip_every=1, dim_in=7, pre_mp=1, dim_inner=16, layer_type='generalconv'):
    cfg.gnn.stage_type, cfg.gnn.layers_mp, cfg.gnn.skip_every = stage_type, layers_mp, skip_every
    cfg.gnn.layers_pre_mp, cfg.gnn.dim_inner, cfg.gnn.layer_type = pre_mp, dim_inner, layer_type
    return gnn.GNN(dim_in, 5)


def test_config_default_and_stage_dict():
    assert cfg.gnn.skip_every == 1 and cfg.gnn.stage_type == 'stack'
    assert gnn.stage_dict == {'stack': gnn.GNNStackStage, 'skipsum': gnn.GNNSkipStage,
                              'skipconcat': gnn.GNNSkipStage}
    assert isinstance(_gnn('stack').mp, gnn.GNNStackStage)
    assert isinstance(_gnn('skipsum').mp, gnn.GNNSkipStage)
    assert isinstance(_gnn('skipconcat').mp, gnn.GNNSkipStage)


def test_construction_errors():
    with pytest.raises(ValueError):
        _gnn('skipmean')
    with pytest.raises(ValueError):
        _gnn('skipsum', layers_mp=3, skip_every=2)
    with pytest.raises(ValueError):
        _gnn('skipconcat', layers_mp=4, skip_every=3)
    with pytest.raises(ValueError):                        # no pre-MP layer: the first block sees dim_in != dim_inner
        _gnn('skipsum', pre_mp=0, dim_in=7, dim_inner=16)
    _gnn('skipconcat', pre_mp=0, dim_in=7, dim_inner=16)   # concat takes any input width
    _gnn('skipsum', pre_mp=0, dim_in=16, dim_inner=16)


@pytest.mark.parametrize('skip_every', [1, 2])
@pytest.mark.parametrize('stage_type', ['skipsum', 'skipconcat'])
def test_block_widths_and_head(stage_type, skip_every):
    layers_mp, d = 4, 16
    m = _gnn(stage_type, layers_mp=layers_mp, skip_every=skip_every, dim_inner=d)
    blocks = list(m.mp.children())
    nb = layers_mp // skip_every
    assert [n for n, _ in m.mp.named_children()] == ['block{}'.format(i) for i in range(nb)]
    for i, b in enumerate(blocks):
        want_in = d if (i == 0 or stage_type == 'skipsum') else d + i * d
        assert len(b.f) == skip_every
        assert b.f[0].layer.model.weight.shape == (want_in, d)
        for j, layer in enumerate(b.f):
            if j > 0:
                assert layer.layer.model.weight.shape == (d, d)
            acts = [mod for mod in layer.post_layer if isinstance(mod, (nn.ReLU, nn.LeakyReLU, nn.PReLU))]
            assert len(acts) == (0 if j == skip_every - 1 else 1)
        assert isinstance(b.act, nn.ReLU)
        assert b.has_l2norm == (i == nb - 1)
    want_out = d if stage_type == 'skipsum' else d + nb * d
    assert m.mp.dim_out == want_out
    assert m.post_mp.layer_post_mp.weight.shape == (5, want_out)


def test_state_dict_keys():
    m = _gnn('skipconcat', layers_mp=4, skip_every=2)
    keys = [k for k in m.state_dict() if k.startswith('mp.')]
    want = []
    for i in range(2):
        for j in range(2):
            want += ['mp.block{}.f.{}.layer.model.{}'.format(i, j, w) for w in ('weight', 'weight_self')]
            want += ['mp.block{}.f.{}.post_layer.0.{}'.format(i, j, b) for b in
                     ('weight', 'bias', 'running_mean', 'running_var', 'num_batches_tracked')]
    assert sorted(keys) == sorted(want)
    cfg.gnn.act = 'prelu'
    m = _gnn('skipsum', layers_mp=2, skip_every=1)
    keys = set(m.state_dict())
    assert {'mp.block0.act.weight', 'mp.block1.act.weight'} <= keys
    assert not any('post_layer.1' in k for k in keys if k.startswith('mp.'))   # the last layer has BN only


def test_stack_keeps_its_keys():
    m = _gnn('stack', layers_mp=2)
    keys = sorted(k for k in m.state_dict() if k.startswith('mp.'))
    want = []
    for i in range(2):
        want += ['mp.layer{}.layer.model.{}'.format(i, w) for w in ('weight', 'weight_self')]
        want += ['mp.layer{}.post_layer.0.{}'.format(i, b) for b in
                 ('weight', 'bias', 'running_mean', 'running_var', 'num_batches_tracked')]
    assert keys == sorted(want)
    assert m.mp.dim_out == 16


@pytest.mark.parametrize('act', [('relu',), ('lrelu', 0.25), ('prelu', torch.tensor([0.3], dtype=torch.float64))])
@pytest.mark.parametrize('mode', ['skipsum', 'skipconcat'])
def test_oracle_equals_a_hand_composition(mode, act):
    n, d, k = 60, 8, 2
    g = torch.Generator().manual_seed(5)
    ei = random_graph(3, n, 300)
    x = torch.randn(n, d, generator=g, dtype=torch.float64)
    blocks, params = [], []
    w_in = d
    for i in range(2):
        convs, bns = [], []
        for j in range(k):
            fin = w_in if j == 0 else d
            w = torch.randn(fin, d, generator=g, dtype=torch.float64) / fin ** 0.5
            ws = torch.randn(fin, d, generator=g, dtype=torch.float64) / fin ** 0.5
            convs.append(lambda h, w=w, ws=ws: max_agg.general_conv(h, ei, w, ws))
            params.append((w, ws))
            bns.append((torch.rand(d, generator=g, dtype=torch.float64) + 0.5,
                        torch.randn(d, generator=g, dtype=torch.float64) * 0.1))
        blocks.append((convs, bns))
        w_in = d if mode == 'skipsum' else w_in + d
    got = stages.skip_stage(x, blocks, mode, act, l2norm=True)

    def a(t):
        if act[0] == 'relu':
            return F.relu(t)
        if act[0] == 'lrelu':
            return F.leaky_relu(t, act[1])
        return F.prelu(t, act[1])

    h, ps = x, iter(params)
    for convs, bns in blocks:
        y = h
        for j, bn in enumerate(bns):
            # generalconv (add, self_msg concat) restated from oracle.layers' primitives: gather, scatter-add, + x W_self
            w, ws = next(ps)
            y2 = olayers._prop(ei, y @ w, n, 'add') + y @ ws
            y2 = F.batch_norm(y2, None, None, bn[0], bn[1], True, 0.0, 1e-5)
            y = a(y2) if j < len(convs) - 1 else y2
        h = a(h + y) if mode == 'skipsum' else a(torch.cat([h, y], 1))
    want = F.normalize(h, p=2, dim=1)
    assert got.shape == want.shape == (n, d if mode == 'skipsum' else 3 * d)
    assert float((got - want).abs().max()) < 1e-12


def test_oracle_gates_replace_the_activation():
    h = torch.tensor([[-1.0, 2.0, -3.0]], dtype=torch.float64, requires_grad=True)
    gate = torch.tensor([[True, True, False]])
    out = stages.activation(h, ('lrelu', 0.5), gate)
    assert out.tolist() == [[-1.0, 2.0, -1.5]]
    out.sum().backward()
    assert h.grad.tolist() == [[1.0, 1.0, 0.5]]
