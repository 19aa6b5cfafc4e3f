"""Times gaddconv / gmulconv with cfg.gnn.agg = 'add' / 'mean' / 'max' on the products-shaped graph of bench.py (gatconv's
graph, F = 128, one head) and prints one JSON line.

  steps    the layer step 100 -> 128 (forward + backward through ``layer(x, edge_index)``) per layer and aggregation, and
           generalconv's max step (normalize_adj, concat) from the same run as the yardstick of the max path
  passes   gaddconv max's passes one by one at F = 128: scores + alpha, the sliced-ELL max forward, the winner SDDMM,
           gat_dz, gat_csc_gather, the max backward, and the rows epilogue (one n x F pass)
  torch    the oracle's composition in fp32 on the device as the library comparator: alpha h_j over 4 M-edge chunks reduced
           with scatter_reduce('amax') (forward only)
CUDA events after warm-up; the feature matrices (1.25 GB at F = 128) are larger than the L2.  The JSON line and a
torch.profiler trace of one gaddconv max step are written to OUT_DIR (argument 1; default: a new temporary directory)."""
import json
import os
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import bench  # noqa: E402
from graphgym_b200 import functional as F_  # noqa: E402
from graphgym_b200 import ops  # noqa: E402
from graphgym_b200.config import cfg, reset_cfg  # noqa: E402
from graphgym_b200.contrib.layer.attconv import GeneralAddAttConvLayer, GeneralMulAttConvLayer  # noqa: E402
from graphgym_b200.contrib.layer.generalconv import GeneralConvLayer  # noqa: E402
from graphgym_b200.graph import get_layout  # noqa: E402
from max_agg_probe import card, timeit  # noqa: E402


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else tempfile.mkdtemp(prefix='attconv_agg_probe_')
    os.makedirs(out_dir, exist_ok=True)
    print('writing to', out_dir, file=sys.stderr)
    dev = torch.device('cuda')
    n, ei = bench.gen_graph(bench.WORKLOADS['products_gat'], dev, seed=0)
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.randn(n, 100, generator=g, device=dev)
    gy = torch.randn(n, 128, generator=g, device=dev)
    res = dict(probe='attconv_agg', nodes=n, f=128, heads=1, steps_ms={}, passes_ms={})

    def layer_step(cls, agg, **kw):
        reset_cfg()
        cfg.gnn.agg = agg
        for k, v in kw.items():
            setattr(cfg.gnn, k, v)
        torch.manual_seed(0)
        layer = cls(100, 128, bias=True).to(dev)
        reset_cfg()
        xg = x.clone().requires_grad_(True)

        def step():
            layer.zero_grad(set_to_none=True)
            xg.grad = None
            layer(xg, ei).backward(gy)
        return layer, step

    for name, cls in (('gaddconv', GeneralAddAttConvLayer), ('gmulconv', GeneralMulAttConvLayer)):
        for agg in ('add', 'mean', 'max'):
            _, step = layer_step(cls, agg)
            res['steps_ms'][f'{name}_{agg}'] = timeit(step, it=5, warm=2)
            print(name, agg, res['steps_ms'][f'{name}_{agg}'], file=sys.stderr, flush=True)
    _, step = layer_step(GeneralConvLayer, 'max', normalize_adj=True, self_msg='concat')
    res['steps_ms']['generalconv_max'] = timeit(step, it=5, warm=2)

    # gaddconv max, pass by pass (the composition of functional._GatAggregateMax, heads = 1)
    lay = get_layout(ei, n, ops.LOOPS_KEEP)
    csr, csc, m = lay.csr, lay.csc, lay.csc2csr
    layer, step = layer_step(GeneralAddAttConvLayer, 'max')
    h = F_.linear(x, layer.linear_msg.weight.detach())
    att = layer.att.detach().view(1, -1)
    a_tgt, a_src = ops.gat_scores(h, att)
    alpha = ops.gat_alpha(csr, a_tgt, a_src, 0.2)
    _, arg = ops.spmm_max(csr, h, alpha)
    dalpha = ops.max_winner_sddmm(csr, arg, gy, h)
    dz, da_tgt = ops.gat_dz(csr, a_tgt, a_src, alpha, dalpha.view(-1), 0.2)
    alpha_t, da_src = ops.gat_csc_gather(csc, m, alpha, dz)
    P = res['passes_ms']
    P['scores'] = timeit(lambda: ops.gat_scores(h, att))
    P['alpha'] = timeit(lambda: ops.gat_alpha(csr, a_tgt, a_src, 0.2))
    P['max_fwd'] = timeit(lambda: ops.spmm_max(csr, h, alpha))
    P['winner'] = timeit(lambda: ops.max_winner_sddmm(csr, arg, gy, h))
    P['dz'] = timeit(lambda: ops.gat_dz(csr, a_tgt, a_src, alpha, dalpha.view(-1), 0.2))
    P['csc_gather'] = timeit(lambda: ops.gat_csc_gather(csc, m, alpha, dz))
    P['max_bwd'] = timeit(lambda: ops.spmm_max_bwd(csc, m, gy, arg, alpha_t))
    P['rows_epilogue'] = timeit(lambda: ops.rows_epilogue(gy, csr))
    P['sum_sell_f128'] = timeit(lambda: ops.spmm(csr, h, alpha))
    res['winner_over_max_bwd'] = P['winner'] / P['max_bwd']

    src, tgt = csr.nbr.long(), csr.rowid.long()

    def torch_amax():
        o = torch.full((n, 128), float('-inf'), device=dev)
        for a in range(0, csr.num_slots, 1 << 22):
            b = min(csr.num_slots, a + (1 << 22))
            msg = h.index_select(0, src[a:b]) * alpha[a:b].view(-1, 1)
            o.scatter_reduce_(0, tgt[a:b].view(-1, 1).expand(-1, 128), msg, 'amax')
        return o
    res['torch_amax_fwd_ms'] = timeit(torch_amax, it=3, warm=1)

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    prof.export_chrome_trace(os.path.join(out_dir, 'attconv_agg_probe.pt.trace.json'))
    res['profile_gaddconv_max_step_us'] = {e.key: round(e.device_time_total, 1) for e in prof.key_averages()
                                           if e.device_time_total > 0}
    res['card'], res['power_limit'] = card()
    line = json.dumps(res)
    with open(os.path.join(out_dir, 'attconv_agg_probe.json'), 'w') as fh:
        fh.write(line + '\n')
    print(line)


if __name__ == '__main__':
    main()
