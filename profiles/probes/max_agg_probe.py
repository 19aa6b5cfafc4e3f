"""Times the max aggregation (csrc/spmm_max.cu) on the products-shaped graph of bench.py and prints one JSON line.

Per width F in 16 / 64 / 128 / 256 and one odd width (row kernels): the sum aggregation (sliced ELL up to 128 columns,
the merge-path kernel beyond), the max forward and the max backward, each with the GCN normalisation weights of
generalconv(normalize_adj=True); torch's scatter_reduce('amax') over 4 M-edge chunks of the same messages as the library
comparator; the whole generalconv step (100 -> 128, forward + backward) with agg = 'add' against 'max'.  CUDA events
after warm-up; the feature matrices are larger than the L2 from F = 16 up.  Algorithmic bytes (E' = slots, N = rows):
  forward  E'*F*4 (gathered rows) + E'*8 (index + slot units) [+ E'*4 weights] + N*F*8 (out + arg)
  backward E'*F*8 (g and arg rows) + E'*8 (index + edge-map units) [+ E'*4 weights] + N*F*4 (dx)
The JSON line and a torch.profiler trace of one max forward + backward at F = 128 are also written to OUT_DIR
(argument 1; default: a new temporary directory, printed)."""
import json
import os
import subprocess
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from graphgym_b200 import ops  # noqa: E402
from graphgym_b200.config import cfg, reset_cfg  # noqa: E402
from graphgym_b200.contrib.layer.generalconv import GeneralConvLayer  # noqa: E402
from graphgym_b200.graph import GraphLayout  # noqa: E402


def timeit(fn, it=10, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(it):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / it


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = 'unknown'
    return name, q


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else tempfile.mkdtemp(prefix='max_agg_probe_')
    os.makedirs(out_dir, exist_ok=True)
    print('writing to', out_dir, file=sys.stderr)
    dev = torch.device('cuda')
    n, ei = bench.gen_graph(bench.WORKLOADS['products_gcn'], dev, seed=0)
    lay = GraphLayout(ei, n, ops.LOOPS_ADD_REMAINING)
    csr, csc, c2c = lay.csr, lay.csc, lay.csc2csr
    w_csr, w_csc = lay.weights('gcn_src_max')
    slots = csr.num_slots
    src, tgt = csr.nbr.long(), csr.rowid.long()
    peak, peak_src = bench.load_peaks()
    res = dict(probe='max_agg', nodes=n, slots=slots, copy_peak_gbs=peak, copy_peak_source=peak_src, widths={})
    g = torch.Generator(device=dev).manual_seed(0)

    def gbs(b, ms):
        return b / ms / 1e6

    for f in (16, 64, 128, 256, 63):
        x = torch.randn(n, f, generator=g, device=dev)
        gy = torch.randn(n, f, generator=g, device=dev)
        r = {}
        if f % 4 == 0:
            r['sum_ms'] = timeit(lambda: ops.spmm(csr, x, w_csr))
            r['sum_kernel'] = 'sell' if f <= 128 else 'mp'
        r['path'] = 'sell' if f % 4 == 0 else 'row'
        _, arg = ops.spmm_max(csr, x, w_csr)
        r['max_fwd_ms'] = timeit(lambda: ops.spmm_max(csr, x, w_csr))
        r['max_bwd_ms'] = timeit(lambda: ops.spmm_max_bwd(csc, c2c, gy, arg, w_csc))
        fwd_b = slots * f * 4 + slots * 8 + slots * 4 + n * f * 8
        bwd_b = slots * f * 8 + slots * 8 + slots * 4 + n * f * 4
        r['max_fwd_gbs'], r['max_bwd_gbs'] = gbs(fwd_b, r['max_fwd_ms']), gbs(bwd_b, r['max_bwd_ms'])
        r['max_fwd_copy_frac'], r['max_bwd_copy_frac'] = r['max_fwd_gbs'] / peak, r['max_bwd_gbs'] / peak
        if 'sum_ms' in r:
            r['fwd_over_sum'], r['bwd_over_sum'] = r['max_fwd_ms'] / r['sum_ms'], r['max_bwd_ms'] / r['sum_ms']

        def torch_amax():
            o = torch.full((n, f), float('-inf'), device=dev)
            for a in range(0, slots, 1 << 22):
                b = min(slots, a + (1 << 22))
                m = x.index_select(0, src[a:b]) * w_csr[a:b].view(-1, 1)
                o.scatter_reduce_(0, tgt[a:b].view(-1, 1).expand(-1, f), m, 'amax')
            return o
        r['torch_amax_ms'] = timeit(torch_amax, it=3, warm=1)
        res['widths'][str(f)] = r
        print(f, json.dumps(r), file=sys.stderr, flush=True)
        del x, gy, arg

    # the generalconv step, 100 -> 128, forward + backward
    x = torch.randn(n, 100, generator=g, device=dev)
    gy = torch.randn(n, 128, generator=g, device=dev)
    for agg in ('add', 'max'):
        reset_cfg()
        cfg.gnn.agg, cfg.gnn.normalize_adj = agg, True
        layer = GeneralConvLayer(100, 128).to(dev)
        reset_cfg()
        xg = x.clone().requires_grad_(True)

        def step():
            layer.zero_grad(set_to_none=True)
            xg.grad = None
            layer(xg, ei).backward(gy)
        res[f'generalconv_{agg}_step_ms'] = timeit(step, it=5, warm=2)
    res['generalconv_max_over_add'] = res['generalconv_max_step_ms'] / res['generalconv_add_step_ms']

    from torch.profiler import ProfilerActivity, profile
    x = torch.randn(n, 128, generator=g, device=dev)
    gy = torch.randn(n, 128, generator=g, device=dev)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _, arg = ops.spmm_max(csr, x, w_csr)
        ops.spmm_max_bwd(csc, c2c, gy, arg, w_csc)
        ops.spmm(csr, x, w_csr)
        torch.cuda.synchronize()
    prof.export_chrome_trace(os.path.join(out_dir, 'max_agg_probe.pt.trace.json'))
    res['profile_f128_us'] = {e.key: round(e.device_time_total, 1) for e in prof.key_averages() if e.device_time_total > 0}
    res['card'], res['power_limit'] = card()
    line = json.dumps(res)
    with open(os.path.join(out_dir, 'max_agg_probe.json'), 'w') as fh:
        fh.write(line + '\n')
    print(line)


if __name__ == '__main__':
    main()
