"""splineconv on the host: the oracle against torch_spline_conv's formula edge by edge, known answers of the degree-1 basis,
the chunked step against autograd, the module's parameters and buffers, registration and refusals (no GPU)."""
import math

import pytest
import torch

from graphgym_b200.config import cfg, reset_cfg
from graphgym_b200.models.layer import Batch, GeneralLayer, SplineConv, _SplineConvLayer, layer_dict
from oracle import splineconv as S


@pytest.fixture(autouse=True)
def _cfg():
    reset_cfg()
    yield
    reset_cfg()


def tiny_graph():
    """7 nodes: duplicate edges (0 -> 1 twice), self loops (2 -> 2, 4 -> 4), isolated nodes 5 and 6."""
    ei = torch.tensor([[0, 0, 1, 2, 3, 1, 4, 0, 3, 2, 1, 4],
                       [1, 1, 2, 2, 0, 3, 4, 3, 1, 0, 0, 2]])
    return 7, ei


def pseudo(e, seed):
    """{0, 0.5, 1, 1.3, -0.4} first, then U(0, 1)."""
    g = torch.Generator().manual_seed(seed)
    fixed = torch.tensor([0.0, 0.5, 1.0, 1.3, -0.4], dtype=torch.float64)
    return torch.cat([fixed, torch.rand(e - fixed.numel(), generator=g, dtype=torch.float64)])


def params(fin, fout, seed, bias=True):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(2, fin, fout, generator=g, dtype=torch.float64),
            torch.randn(fin, fout, generator=g, dtype=torch.float64),
            torch.randn(fout, generator=g, dtype=torch.float64) if bias else None)


@pytest.mark.parametrize('bias', [False, True])
def test_oracle_matches_edge_loop(bias):
    n, ei = tiny_graph()
    g = torch.Generator().manual_seed(1)
    x = torch.randn(n, 4, generator=g, dtype=torch.float64)
    u = pseudo(ei.size(1), 2)
    w, root, b = params(4, 5, 3, bias)
    want = S.spline_conv_loop(x, ei, u, w, root, b)
    assert torch.allclose(S.spline_conv(x, ei, u, w, root, b), want, rtol=1e-12, atol=1e-12)
    assert torch.allclose(S.spline_conv(x, ei, u.view(-1, 1), w, root, b), want, rtol=1e-12, atol=1e-12)
    rest = x[5:] @ root + (b if b is not None else 0)
    assert torch.allclose(want[5:], rest, atol=1e-12)          # no in-edges: x root + bias


def test_known_answers():
    """One edge 0 -> 1 into an otherwise empty row: u in [0, 1) gives (1 - u) W0 + u W1, u = 1 gives W1 exactly, u in
    (1, 2) gives fr W0 + (1 - fr) W1, u in (-1, 0) gives -u W0 + (1 + u) W1; du has the literal sign at u = 1."""
    ei = torch.tensor([[0], [1]])
    x = torch.tensor([[1.0, 0.0], [0.0, 0.0]], dtype=torch.float64)
    w, root, _ = params(2, 3, 4)
    for u, c in [(0.0, (1, 0)), (0.25, (0.75, 0.25)), (1.0, (0, 1)), (1.5, (0.5, 0.5)), (1.25, (0.25, 0.75)),
                 (-0.4, (0.4, 0.6))]:
        out = S.spline_conv(x, ei, torch.tensor([u], dtype=torch.float64), w, root)
        assert torch.allclose(out[1], c[0] * w[0, 0] + c[1] * w[1, 0], atol=1e-15), u
        assert torch.allclose(S.coefficients(torch.tensor([u], dtype=torch.float64))[0],
                              torch.tensor(c, dtype=torch.float64), atol=1e-15)
    out = S.spline_conv(x, ei, torch.tensor([1.0], dtype=torch.float64), w, root)
    assert torch.equal(out[1], w[1, 0])
    # du_e = dc[(t+1) mod 2] - dc[t mod 2]: at u = 1 (t = 1) that is dc0 - dc1, the opposite of u = 1 - eps
    gy = torch.randn(2, 3, dtype=torch.float64, generator=torch.Generator().manual_seed(5))
    dc = [float(gy[1] @ w[k, 0]) for k in range(2)]
    for u, want in [(1.0, dc[0] - dc[1]), (0.999, dc[1] - dc[0]), (0.0, dc[1] - dc[0]), (1.5, dc[0] - dc[1]),
                    (-0.4, dc[1] - dc[0])]:
        uu = torch.tensor([u], dtype=torch.float64, requires_grad=True)
        S.spline_conv(x, ei, uu, w, root).backward(gy)
        assert math.isclose(float(uu.grad), want, rel_tol=1e-12, abs_tol=1e-12), u
        ref = S.spline_conv_step(x, ei, uu.detach(), w, root, None, gy)
        assert math.isclose(float(ref[2]), want, rel_tol=1e-12, abs_tol=1e-12), u


def test_negative_pseudo_uses_the_non_negative_mod():
    """u <= -1 (undefined in the reference): t mod 2 taken in {0, 1}; u = -1.5 -> t = -1, fr = 0.5, matrices 1 and 0."""
    i0, i1, b0, b1 = S.basis(torch.tensor([-1.5, -2.25], dtype=torch.float64))
    assert i0.tolist() == [1, 0] and i1.tolist() == [0, 1]
    assert torch.allclose(b0, torch.tensor([0.5, 0.25], dtype=torch.float64))


@pytest.mark.parametrize('bias', [False, True])
@pytest.mark.parametrize('shape', ['flat', 'column'])
def test_chunked_step_matches_autograd(bias, shape):
    n, ei = tiny_graph()
    g = torch.Generator().manual_seed(6)
    x = torch.randn(n, 4, generator=g, dtype=torch.float64, requires_grad=True)
    u0 = torch.cat([pseudo(ei.size(1) - 3, 7), torch.tensor([2.5, -0.9, 0.0], dtype=torch.float64)])
    u = (u0 if shape == 'flat' else u0.view(-1, 1)).clone().requires_grad_(True)
    w, root, b = params(4, 5, 8, bias)
    leaves = [t.requires_grad_(True) for t in (w, root, b) if t is not None]
    gy = torch.randn(n, 5, generator=g, dtype=torch.float64)
    S.spline_conv(x, ei, u, w, root, b).backward(gy)
    with torch.no_grad():
        ref = S.spline_conv_step(x, ei, u, w, root, b, gy, chunk=5)
        out = S.spline_conv(x, ei, u, w, root, b)
    assert torch.allclose(ref[0], out, atol=1e-12)
    assert torch.allclose(ref[1], x.grad, atol=1e-12)
    assert ref[2].shape == u.shape and torch.allclose(ref[2], u.grad, atol=1e-12)
    assert torch.allclose(ref[3], w.grad, atol=1e-12)
    assert torch.allclose(ref[4], root.grad, atol=1e-12)
    if b is not None:
        assert torch.allclose(ref[5], b.grad, atol=1e-12)
    assert leaves


def test_parameters_buffers_and_init():
    torch.manual_seed(0)
    layer = _SplineConvLayer(6, 5)
    assert {k: tuple(v.shape) for k, v in layer.named_parameters()} == {'weight': (2, 6, 5), 'root': (6, 5), 'bias': (5,)}
    sd = layer.state_dict()
    assert set(sd) == {'weight', 'root', 'bias', 'kernel_size', 'is_open_spline'}
    assert sd['kernel_size'].dtype == torch.int64 and sd['kernel_size'].tolist() == [2]
    assert sd['is_open_spline'].dtype == torch.uint8 and sd['is_open_spline'].tolist() == [1]
    bound = 1 / math.sqrt(2 * 6)
    for k in ('weight', 'root', 'bias'):
        assert sd[k].abs().max() <= bound and sd[k].abs().max() > 0.5 * bound, k
    # a reference-keyed state_dict loads strictly
    ref = {'weight': torch.randn(2, 6, 5), 'root': torch.randn(6, 5), 'bias': torch.randn(5),
           'kernel_size': torch.tensor([2]), 'is_open_spline': torch.tensor([1], dtype=torch.uint8)}
    layer.load_state_dict(ref, strict=True)
    assert torch.equal(layer.weight, ref['weight']) and torch.equal(layer.root, ref['root'])
    assert 'bias' not in dict(_SplineConvLayer(6, 5, bias=False).named_parameters())


def test_registration_and_general_layer():
    assert layer_dict['splineconv'] is SplineConv
    gl = GeneralLayer('splineconv', 4, 5)
    assert set(gl.state_dict()) >= {'layer.model.weight', 'layer.model.root', 'layer.model.kernel_size',
                                    'layer.model.is_open_spline'}
    assert 'layer.model.bias' not in gl.state_dict()          # bias=False under BatchNorm, as GraphGym
    assert 'layer.model.bias' in GeneralLayer('splineconv', 4, 5, has_bn=False).state_dict()
    cfg.gnn.agg, cfg.gnn.normalize_adj = 'max', True          # not read: the wrapper passes neither
    GeneralLayer('splineconv', 4, 5)


@pytest.mark.parametrize('stage', ['stack', 'skipsum'])
def test_gnn_builds(stage):
    from graphgym_b200.models.gnn import GNN
    cfg.gnn.layer_type, cfg.gnn.stage_type = 'splineconv', stage
    cfg.gnn.layers_mp, cfg.gnn.dim_inner = 2, 8
    model = GNN(8, 3)
    assert len([k for k in model.state_dict() if k.endswith('model.root')]) == 2


def test_refusals():
    for kw in ({'dim': 2}, {'kernel_size': 3}, {'degree': 2}, {'is_open_spline': False}):
        with pytest.raises(NotImplementedError):
            _SplineConvLayer(4, 4, **kw)
    layer = _SplineConvLayer(4, 4)
    ei = torch.tensor([[0, 1, 1], [1, 0, 1]])
    x = torch.randn(2, 4)
    for bad, match in ((None, 'edge_feature'), (torch.rand(3, dtype=torch.float64), 'float32'),
                       (torch.rand(3, 2), 'out of bounds'), (torch.rand(4), 'edge_feature'),
                       (torch.rand(2, 1), 'edge_feature'), (torch.rand(3, 1, 1), 'edge_feature')):
        with pytest.raises(ValueError, match=match):
            layer(x, ei, bad)
    with pytest.raises(ValueError, match='edge_feature'):
        SplineConv(4, 4)(Batch(x, ei))
    cfg.b200.gather_dtype = 'bf16'
    with pytest.raises(NotImplementedError):
        layer(x, ei, torch.rand(3))
