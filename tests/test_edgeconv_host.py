"""generaledgeconv / generalsampleedgeconv on the host: the oracle against its definition edge by edge, the chunked step
against autograd over the oracle, the module's parameters, config defaults, refusals and registration (no GPU)."""
import itertools

import pytest
import torch

from graphgym_b200 import ops
from graphgym_b200.config import cfg, reset_cfg
from graphgym_b200.contrib.layer.generalconv import GeneralEdgeConvLayer
from graphgym_b200.models.layer import Batch, GeneralLayer, layer_dict
from oracle import edgeconv as E

CASES = list(itertools.product(['add', 'mean', 'max'], ['single', 'both'], ['none', 'add', 'concat'], [False, True]))


@pytest.fixture(autouse=True)
def _cfg():
    reset_cfg()
    yield
    reset_cfg()


def tiny_graph():
    """7 nodes: duplicate edges (0 -> 1 twice), self loops (2 -> 2, 4 -> 4), isolated nodes 5 and 6."""
    ei = torch.tensor([[0, 0, 1, 2, 3, 1, 4, 0, 3, 2],
                       [1, 1, 2, 2, 0, 3, 4, 3, 1, 0]])
    return 7, ei


def params(fin, fout, kd, direction, self_msg, bias, seed):
    g = torch.Generator().manual_seed(seed)
    k = (2 if direction == 'both' else 1) * fin + kd
    w = torch.randn(fout, k, generator=g, dtype=torch.float64)
    ws = torch.randn(fout, fin, generator=g, dtype=torch.float64) if self_msg == 'concat' else None
    b = torch.randn(fout, generator=g, dtype=torch.float64) if bias else None
    return w, ws, b


@pytest.mark.parametrize('aggr,direction,self_msg,bias', CASES)
def test_oracle_matches_edge_loop(aggr, direction, self_msg, bias):
    n, ei = tiny_graph()
    fin, kd = 4, 3
    fout = fin if self_msg == 'add' else 5
    g = torch.Generator().manual_seed(1)
    x = torch.randn(n, fin, generator=g, dtype=torch.float64)
    a = torch.randn(ei.size(1), kd, generator=g, dtype=torch.float64)
    w, ws, b = params(fin, fout, kd, direction, self_msg, bias, 2)
    want = E.general_edge_conv_loop(x, ei, a, w, ws, b, aggr, direction, self_msg)
    got = E.general_edge_conv(x, ei, a, w, ws, b, aggr, direction, self_msg)
    assert torch.allclose(got, want, rtol=1e-12, atol=1e-12)
    rest = ((b if b is not None else 0) + (x[5:] @ ws.t() if ws is not None else 0) + (x[5:] if self_msg == 'add' else 0))
    assert torch.allclose(got[5:], rest + torch.zeros_like(got[5:]), atol=1e-12)   # no in-edges: 0 from the aggregation


@pytest.mark.parametrize('aggr,direction,self_msg,bias', CASES)
def test_chunked_step_matches_autograd(aggr, direction, self_msg, bias):
    n, ei = tiny_graph()
    fin, kd = 4, 3
    fout = fin if self_msg == 'add' else 5
    g = torch.Generator().manual_seed(3)
    x = torch.randn(n, fin, generator=g, dtype=torch.float64, requires_grad=True)
    a = torch.randn(ei.size(1), kd, generator=g, dtype=torch.float64, requires_grad=True)
    w, ws, b = params(fin, fout, kd, direction, self_msg, bias, 4)
    leaves = [t.requires_grad_(True) for t in (w, ws, b) if t is not None]
    gy = torch.randn(n, fout, generator=g, dtype=torch.float64)
    out = E.general_edge_conv(x, ei, a, w, ws, b, aggr, direction, self_msg)
    out.backward(gy)
    with torch.no_grad():
        ref = E.general_edge_conv_step(x, ei, a, w, ws, b, gy, aggr, direction, self_msg, chunk=3)
    assert torch.allclose(ref[0], out, atol=1e-12)
    assert torch.allclose(ref[1], x.grad, atol=1e-12)
    assert torch.allclose(ref[2], a.grad, atol=1e-12)
    assert torch.allclose(ref[3], w.grad, atol=1e-12)
    if ws is not None:
        assert torch.allclose(ref[4], ws.grad, atol=1e-12)
    if b is not None:
        assert torch.allclose(ref[5], b.grad, atol=1e-12)
    if aggr == 'max':
        assert (ref[6][5:] == -1).all() and (ref[7] == 0).all()
    assert leaves


def test_max_ties_go_to_the_first_edge():
    """All-equal messages: every column's gradient sits on the first in-edge of the row (edge order)."""
    n, ei = tiny_graph()
    x = torch.ones(n, 2, dtype=torch.float64)
    a = torch.zeros(ei.size(1), 3, dtype=torch.float64, requires_grad=True)
    w = torch.ones(4, 5, dtype=torch.float64)
    gy = torch.ones(n, 4, dtype=torch.float64)
    ref = E.general_edge_conv_step(x, ei, a.detach(), w, None, None, gy, 'max', 'single', 'none', chunk=4)
    first = {}
    for e, i in enumerate(ei[1].tolist()):
        first.setdefault(i, e)
    for i in range(n):
        assert (ref[6][i] == first.get(i, -1)).all()


def test_parameters_and_state_dict():
    cfg.dataset.edge_dim, cfg.gnn.msg_direction = 6, 'both'
    layer = GeneralEdgeConvLayer(4, 5)
    shapes = {k: tuple(v.shape) for k, v in layer.named_parameters()}
    assert shapes == {'linear_msg.weight': (5, 14), 'linear_self.weight': (5, 4), 'bias': (5,)}
    assert (layer.bias == 0).all()
    cfg.gnn.msg_direction, cfg.gnn.self_msg = 'single', 'none'
    layer = GeneralEdgeConvLayer(4, 5, bias=False)
    assert {k: tuple(v.shape) for k, v in layer.named_parameters()} == {'linear_msg.weight': (5, 10)}
    cfg.gnn.self_msg = 'concat'
    gl = GeneralLayer('generaledgeconv', 4, 5)
    assert set(gl.state_dict()) >= {'layer.model.linear_msg.weight', 'layer.model.linear_self.weight'}
    assert 'layer.model.bias' not in gl.state_dict()          # bias=False under BatchNorm, as GraphGym
    gl = GeneralLayer('generalsampleedgeconv', 4, 5, has_bn=False)
    assert 'layer.model.bias' in gl.state_dict()


def test_config_defaults_and_registration():
    assert cfg.dataset.edge_dim == 128 and cfg.gnn.msg_direction == 'single' and cfg.gnn.keep_edge == 0.5
    assert 'generaledgeconv' in layer_dict and 'generalsampleedgeconv' in layer_dict
    assert Batch(torch.zeros(1, 1), torch.zeros(2, 0, dtype=torch.long)).edge_feature is None


def test_refusals():
    cfg.gnn.normalize_adj = True
    with pytest.raises(NotImplementedError):
        GeneralEdgeConvLayer(4, 4)
    reset_cfg()
    cfg.gnn.self_msg = 'add'
    with pytest.raises(ValueError):
        GeneralEdgeConvLayer(4, 5)
    GeneralEdgeConvLayer(4, 4)
    reset_cfg()
    cfg.gnn.agg, cfg.dataset.edge_dim = 'max', ops.EDGE_MAX_KD + 1
    with pytest.raises(NotImplementedError):
        GeneralEdgeConvLayer(4, 4)
    cfg.gnn.agg = 'add'
    GeneralEdgeConvLayer(4, 4)
    reset_cfg()
    cfg.dataset.edge_dim = 3
    layer = GeneralEdgeConvLayer(4, 4)
    ei = torch.tensor([[0, 1], [1, 0]])
    x = torch.randn(2, 4)
    for bad in (None, torch.randn(2, 2), torch.randn(3, 3), torch.randn(2, 3, dtype=torch.float64), torch.randn(6)):
        with pytest.raises(ValueError, match='edge_feature'):
            layer(x, ei, edge_feature=bad)
    cfg.b200.gather_dtype = 'bf16'
    with pytest.raises(NotImplementedError):
        layer(x, ei, edge_feature=torch.randn(2, 3))


@pytest.mark.parametrize('stage', ['stack', 'skipsum'])
def test_gnn_builds(stage):
    from graphgym_b200.models.gnn import GNN
    cfg.gnn.layer_type, cfg.gnn.stage_type, cfg.dataset.edge_dim = 'generaledgeconv', stage, 4
    cfg.gnn.layers_mp, cfg.gnn.dim_inner = 2, 8
    model = GNN(8, 3)
    names = [k for k in model.state_dict() if 'linear_msg' in k]
    assert len(names) == 2, names
