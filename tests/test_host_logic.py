"""Host-side logic that needs no GPU: registry contract, config loading, parameter naming, the
no-CPU-fallback rule."""
import os

import pytest
import torch

from graphgym_b200 import register
from graphgym_b200.config import cfg, load_cfg, reset_cfg
from graphgym_b200.models.layer import Batch, GeneralLayer, TFG_ALIASES, layer_dict, resolve_layer


def test_registry_names_and_duplicate_key_error():
    for name in ('gcnconv', 'sageconv', 'ginconv', 'gatconv', 'idconv', 'gcnidconv', 'sageidconv', 'ginidconv', 'gatidconv'):
        assert name in layer_dict
    with pytest.raises(KeyError, match='Key gcnidconv is already pre-defined.'):
        register.register_layer('gcnidconv', object)
    register.register_layer('my_test_layer', object)
    assert register.layer_dict['my_test_layer'] is object
    del register.layer_dict['my_test_layer']


def test_tfg_aliases_cover_main_zd_names():
    # plain Tfg-* names (tf_geometric's own layers, not in the reference tree) select the PyG-semantics operators; the four
    # ID layers of TfgIDLayer.py are registered under their main_zd.py names with their own semantics
    assert set(TFG_ALIASES) == {'Tfg-gcnconv', 'Tfg-sageconv', 'Tfg-gatconv', 'Tfg-ginconv'}
    assert {'Tfg-idgcn', 'Tfg-idsage', 'Tfg-idgat', 'Tfg-idgin'} <= set(layer_dict)
    assert resolve_layer('Tfg-idsage') is layer_dict['Tfg-idsage'] and resolve_layer('Tfg-sageconv') is layer_dict['sageconv']


def test_parameter_names_match_reference_state_dict():
    """checkpoint round-trip contract (SURVEY §5): weight / weight_id / bias / nn.* names."""
    reset_cfg()
    l = layer_dict['gcnidconv'](5, 7, bias=True)
    assert sorted(dict(l.named_parameters())) == ['model.bias', 'model.weight', 'model.weight_id']
    assert l.model.weight.shape == (5, 7) and l.model.bias.abs().sum() == 0
    a = (6.0 / 12) ** 0.5
    assert l.model.weight.abs().max() <= a
    l = layer_dict['sageidconv'](5, 7, bias=False)
    assert l.model.weight.shape == (10, 7) and l.model.bias is None
    l = layer_dict['ginidconv'](5, 7)
    assert 'model.nn_id.2.weight' in dict(l.named_parameters()) and 'model.eps' in l.state_dict()
    l = layer_dict['sageconv'](5, 7, bias=True)
    assert sorted(dict(l.named_parameters())) == ['model.lin_l.bias', 'model.lin_l.weight', 'model.lin_r.weight']


def test_general_idconv_reads_cfg_at_construction():
    reset_cfg()
    cfg.gnn.agg, cfg.gnn.normalize_adj = 'mean', True
    l = layer_dict['idconv'](3, 3)
    assert l.model.aggr == 'mean' and l.model.normalize is True
    cfg.gnn.agg = 'max'
    with pytest.raises(NotImplementedError):
        layer_dict['idconv'](3, 3)
    reset_cfg()


def test_general_layer_bias_follows_batchnorm():
    reset_cfg()
    assert GeneralLayer('gcnconv', 4, 4).layer.model.bias is None
    cfg.gnn.batchnorm = False
    assert GeneralLayer('gcnconv', 4, 4).layer.model.bias is not None
    reset_cfg()


def test_load_reference_yaml(tmp_path):
    p = tmp_path / 'c.yaml'
    p.write_text('gnn:\n  layers_mp: 3\n  dim_inner: 128\n  layer_type: Tfg-idgcn\n  agg: add\n'
                 'dataset:\n  transform: ego\n  augment_feature: [node_identity]\n  augment_feature_dims: [10]\n')
    reset_cfg()
    load_cfg(str(p))
    assert cfg.gnn.dim_inner == 128 and cfg.gnn.layer_type == 'Tfg-idgcn' and cfg.gnn.batchnorm is True
    assert cfg.dataset.transform == 'ego' and cfg.dataset.augment_feature_dims == [10]
    reset_cfg()


def test_no_cpu_fallback():
    """CPU tensors must fail loudly — the oracle is never reachable from the product path."""
    reset_cfg()
    l = layer_dict['gcnconv'](4, 4)
    b = Batch(torch.randn(5, 4), torch.tensor([[0, 1], [1, 0]]))
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        l(b)


def test_product_never_imports_oracle():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for dirpath, _, files in os.walk(os.path.join(root, 'graphgym_b200')):
        for f in files:
            if f.endswith('.py'):
                src = open(os.path.join(dirpath, f)).read()
                assert 'import oracle' not in src and 'from oracle' not in src, f


def test_new_entry_points_have_no_cpu_path():
    """pooling, the clustering label, the bf16 cast and the peer-memory exchange reject CPU tensors like every op"""
    from graphgym_b200 import ops, parallel
    from graphgym_b200.contrib.transform.clustering import clustering_coefficient
    from graphgym_b200.models import pooling
    x = torch.randn(6, 4)
    batch = torch.tensor([0, 0, 1, 1, 2, 2])
    with pytest.raises(RuntimeError, match='CUDA tensors only'):
        pooling.global_mean_pool(x, batch, size=3)
    with pytest.raises(RuntimeError, match='CUDA tensors only'):
        clustering_coefficient(torch.tensor([[0, 1], [1, 0]]), 2)
    with pytest.raises(RuntimeError, match='CUDA tensors only'):
        ops.cast_bf16(x)
    # round 2: fused post-ops, collation, binning, the Tfg scorer passes
    from graphgym_b200 import functional as F_
    from graphgym_b200 import loader
    from graphgym_b200.contrib.transform import binning
    with pytest.raises(RuntimeError, match='CUDA tensors only'):
        F_.post_ops(x, None, True, ops.ACT_RELU, 0.0, True)
    with pytest.raises(RuntimeError, match='CUDA tensors only'):
        loader.collate([loader.GraphData(node_feature=x, edge_index=torch.zeros((2, 0), dtype=torch.int64))])
    with pytest.raises(RuntimeError, match='CUDA tensors only'):
        binning.argsort_f64(torch.zeros(4, dtype=torch.float64))
    assert sorted(parallel.ROW_PARTITIONED) == ['gatconv', 'gatidconv', 'gcnconv', 'gcnidconv', 'ginconv', 'ginidconv',
                                                'idconv', 'sageconv', 'sageidconv']
    assert ops.bf16_gather_ok(128) and not ops.bf16_gather_ok(100) and not ops.bf16_gather_ok(512)


def test_bench_generators_are_seeded_and_well_formed():
    import bench
    cpu = torch.device('cpu')
    n, ei, ptr = bench.gen_ba_batch(bench.WORKLOADS['ego_idgin'], cpu)
    n2, ei2, _ = bench.gen_ba_batch(bench.WORKLOADS['ego_idgin'], cpu)
    assert n == n2 == 256 * 64 and torch.equal(ei, ei2)                       # seeded
    assert ptr.tolist() == list(range(0, n + 1, 64))
    assert ((ei[0] // 64) == (ei[1] // 64)).all() and (ei[0] != ei[1]).all()      # block-diagonal, no self loops
    code = ei[0] * n + ei[1]
    assert code.unique().numel() == code.numel()                                # simple graphs
    assert torch.equal(torch.sort(code).values, torch.sort(ei[1] * n + ei[0]).values)   # symmetric
    spec = dict(bench.WORKLOADS['products_gcn'], n=5000, e_und=40000, max_deg=500)
    m, e = bench.gen_graph(spec, cpu)
    assert m == 5000 and e.shape == (2, 80000) and int(e.max()) < m
    assert bench.spmm_bytes(10, 100, 8, True) == 100 * 8 * 4 + 10 * 8 * 4 + 100 * 4 + 11 * 4 + 100 * 4
    assert bench.spmm_bytes(10, 100, 8, False, gather_bytes=2) == 100 * 8 * 2 + 10 * 8 * 4 + 100 * 4 + 11 * 4


def test_bench_dump_outputs_keeps_one_seeded_row_sample_within_budget(tmp_path, monkeypatch):
    """bench.py --dump-outputs: every per-node array keeps the same rows, the same ones on every call; whole arrays are
    written whole; float32 on disk unless float64; the array data fits DUMP_BYTES."""
    import numpy as np

    import bench
    monkeypatch.setattr(bench, 'DUMP_BYTES', 40_000)
    g = torch.Generator().manual_seed(0)
    out = torch.randn(1000, 8, generator=g)
    rows = {'out': out, 'grad_x': out[:, :4].double() * 2}      # 64 bytes a row: (40000 - 128) // 64 = 623 rows
    whole = {'grad_w': torch.randn(4, 8, generator=g)}
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), rows=rows, whole=whole)
    a = {f[:-4]: np.load(tmp_path / 'a' / f) for f in os.listdir(tmp_path / 'a')}
    b = {f[:-4]: np.load(tmp_path / 'b' / f) for f in os.listdir(tmp_path / 'b')}
    assert sorted(a) == ['grad_w', 'grad_x', 'out'] and all(np.array_equal(a[k], b[k]) for k in a)
    assert a['out'].shape == (623, 8) and a['out'].dtype == np.float32 and a['grad_x'].dtype == np.float64
    assert np.array_equal(a['grad_x'], a['out'][:, :4].astype(np.float64) * 2)        # the same rows in every array
    assert np.array_equal(a['grad_w'], whole['grad_w'].numpy())
    assert sum(v.nbytes for v in a.values()) <= 40_000
    picked = {tuple(r) for r in a['out'].tolist()}
    assert len(picked) == 623 and picked <= {tuple(r) for r in out.tolist()}
    bench.dump_outputs(str(tmp_path / 'c'), rows={'out': out[:10]})                  # small arrays are written whole
    assert np.array_equal(np.load(tmp_path / 'c' / 'out.npy'), out[:10].numpy())


def test_every_environment_switch_is_documented():
    """INTEGRATION.md §7 lists every GG_* variable the package, the C-ABI library sources and bench.py read."""
    import os
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    used = set()
    pat = re.compile(r'''(?:getenv\(\s*"|environ\.get\(\s*['"])(GG_[A-Z0-9_]+)''')
    for base, _, files in os.walk(os.path.join(root, 'graphgym_b200')):
        if 'build' in base:
            continue
        for name in files:
            if name.endswith(('.py', '.cu', '.cuh')):
                used |= set(pat.findall(open(os.path.join(base, name), errors='ignore').read()))
    used |= set(pat.findall(open(os.path.join(root, 'bench.py')).read()))
    doc = open(os.path.join(root, 'INTEGRATION.md')).read()
    missing = sorted(v for v in used if v not in doc)
    assert used and not missing, missing
