"""Times generaledgeconv (csrc/edge_agg.cu) on the products-shaped graph of bench.py and prints one JSON line.

At F = 128 and edge_dim 16 / 64 (U(-1, 1) edge features): the layer step (100 -> 128, forward + backward, self_msg
'concat') for agg add / mean / max x msg_direction single / both, beside generalconv with the same agg; the edge-row
reduce, the max forward with the edge term against spmm_sell_max in the same run, the winner and dW_a kernels; the torch
composition of the reference's message (concatenation, linear, scatter) in fp32 on a 4 M-edge chunk; the per-step layout
build of generalsampleedgeconv (keep_edge 0.5: the compaction and the CSR / CSC / sliced-ELL builds the step needs).
CUDA events after warm-up.  Algorithmic bytes (E = edges, N = rows, kd = edge_dim):
  edge-row reduce   E*kd*4 (edge rows) + E*4 (perm) + N*kd*4 (out)
  max forward       spmm_sell_max's bytes + E*kd*4 (edge rows) + E*4 (perm)
The JSON line and a torch.profiler trace of one max step at edge_dim 16 are written to OUT_DIR (argument 1; default: a new
temporary directory, printed)."""
import json
import os
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import bench  # noqa: E402
from max_agg_probe import card, timeit  # noqa: E402
from graphgym_b200 import ops  # noqa: E402
from graphgym_b200.config import cfg, reset_cfg  # noqa: E402
from graphgym_b200.contrib.layer.generalconv import GeneralConvLayer, GeneralEdgeConvLayer, sample_edges  # noqa: E402
from graphgym_b200.graph import GraphLayout, clear_cache, get_layout  # noqa: E402


def make_step(layer, x, ei, gy, a=None):
    xg = x.clone().requires_grad_(True)

    def step():
        layer.zero_grad(set_to_none=True)
        xg.grad = None
        out = layer(xg, ei) if a is None else layer(xg, ei, edge_feature=a)
        out.backward(gy)
    return step


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else tempfile.mkdtemp(prefix='edgeconv_probe_')
    os.makedirs(out_dir, exist_ok=True)
    print('writing to', out_dir, file=sys.stderr)
    dev = torch.device('cuda')
    n, ei = bench.gen_graph(bench.WORKLOADS['products_gcn'], dev, seed=0)
    e = ei.size(1)
    lay = get_layout(ei, n, ops.LOOPS_KEEP)
    csr, csc, c2c = lay.csr, lay.csc, lay.csc2csr
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.randn(n, 100, generator=g, device=dev)
    gy = torch.randn(n, 128, generator=g, device=dev)
    res = dict(probe='edgeconv', nodes=n, edges=e, fin=100, fout=128, edge_dims={})

    def gbs(b, ms):
        return b / ms / 1e6

    for agg in ('add', 'mean', 'max'):
        reset_cfg()
        cfg.gnn.agg = agg
        torch.manual_seed(0)
        layer = GeneralConvLayer(100, 128).to(dev)
        res[f'generalconv_{agg}_step_ms'] = timeit(make_step(layer, x, ei, gy), it=5, warm=2)
        del layer
    for kd in (16, 64):
        a = torch.rand(e, kd, generator=g, device=dev) * 2 - 1
        r = {}
        for agg in ('add', 'mean', 'max'):
            for direction in ('single', 'both'):
                reset_cfg()
                cfg.gnn.agg, cfg.gnn.msg_direction, cfg.dataset.edge_dim = agg, direction, kd
                torch.manual_seed(0)
                layer = GeneralEdgeConvLayer(100, 128).to(dev)
                ms = timeit(make_step(layer, x, ei, gy, a), it=5, warm=2)
                r[f'{agg}_{direction}_step_ms'] = ms
                r[f'{agg}_{direction}_over_generalconv'] = ms / res[f'generalconv_{agg}_step_ms']
                print(kd, agg, direction, ms, file=sys.stderr, flush=True)
                del layer
        # per kernel, F = 128
        h = torch.randn(n, 128, generator=g, device=dev)
        w_a = torch.randn(128, kd, generator=g, device=dev) / kd ** 0.5
        r['row_reduce_ms'] = timeit(lambda: ops.edge_row_reduce(csr, a))
        r['row_reduce_gbs'] = gbs(e * kd * 4 + e * 4 + n * kd * 4, r['row_reduce_ms'])
        r['spmm_sell_max_ms'] = timeit(lambda: ops.spmm_max(csr, h))
        r['edge_max_fwd_ms'] = timeit(lambda: ops.edge_max(csr, h, None, a, w_a))
        r['edge_max_fwd_over_spmm_sell_max'] = r['edge_max_fwd_ms'] / r['spmm_sell_max_ms']
        _, arg = ops.edge_max(csr, h, None, a, w_a)
        r['spmm_sell_max_bwd_ms'] = timeit(lambda: ops.spmm_max_bwd(csc, c2c, gy, arg))
        r['edge_max_winner_ms'] = timeit(lambda: ops.edge_max_winner(csr, arg, gy, w_a))
        r['edge_max_wgrad_ms'] = timeit(lambda: ops.edge_max_wgrad(csr, arg, gy, a))
        # the reference's composition in fp32 on one 4 M-edge chunk (the whole graph does not fit as a concatenation)
        w = torch.randn(128, 200 + kd, generator=g, device=dev) / 15
        c = 1 << 22
        src, tgt = ei[0, :c], ei[1, :c]

        def torch_chunk():
            m = torch.cat([x.index_select(0, tgt), x.index_select(0, src), a[:c]], 1) @ w.t()
            return torch.zeros(n, 128, device=dev).index_add_(0, tgt, m)
        r['torch_chunk_4M_ms'] = timeit(torch_chunk, it=3, warm=1)
        r['torch_chunk_scaled_to_E_ms'] = r['torch_chunk_4M_ms'] * e / c
        res['edge_dims'][str(kd)] = r
        del a, h, arg
    # generalsampleedgeconv: the per-step compaction and layout build
    a = torch.rand(e, 16, generator=g, device=dev)

    def sample_layout():
        ei_s, _ = sample_edges(ei, a, 0.5)
        l = GraphLayout(ei_s, n, ops.LOOPS_KEEP)
        ops.sell_layout(l.csr), ops.sell_layout(l.csc), l.csc2csr
    res['sample_layout_build_ms'] = timeit(sample_layout, it=3, warm=1)
    clear_cache()

    from torch.profiler import ProfilerActivity, profile
    reset_cfg()
    cfg.gnn.agg, cfg.gnn.msg_direction, cfg.dataset.edge_dim = 'max', 'both', 16
    layer = GeneralEdgeConvLayer(100, 128).to(dev)
    step = make_step(layer, x, ei, gy, a * 2 - 1)
    step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    prof.export_chrome_trace(os.path.join(out_dir, 'edgeconv_probe.pt.trace.json'))
    res['profile_max_both_kd16_us'] = {k.key: round(k.device_time_total, 1) for k in prof.key_averages()
                                       if k.device_time_total > 0}
    res['card'], res['power_limit'] = card()
    line = json.dumps(res)
    with open(os.path.join(out_dir, 'edgeconv_probe.json'), 'w') as fh:
        fh.write(line + '\n')
    print(line)


if __name__ == '__main__':
    main()
