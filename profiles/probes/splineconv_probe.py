"""Times splineconv (csrc/spline_agg.cu) on the products-shaped graph of bench.py and prints one JSON line.

U(0, 1) pseudo-coordinates.  Per kernel, on the same CSR: spread at gathered width k against spmm_sell_kernel (the sum
aggregation) at k, blend at gathered width 2k against the sum aggregation at 2k; the pseudo-coordinate gradient pass.
Steps (forward + backward): splineconv 100 -> 128 (aggregate first) and 128 -> 64 (transform first), generalconv add at
the same widths in the same run.  Baseline: the torch composition of the reference's message (gather, basis, two matmuls,
index_add_) in fp32 on one 4 M-edge chunk, scaled to the graph.  CUDA events after warm-up.  Bytes per slot gathered
(forward + backward): 3 in (aggregate first), 3 out (transform first).
The JSON line is written to OUT_DIR (argument 1; default: a new temporary directory, printed)."""
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
from graphgym_b200.config import reset_cfg  # noqa: E402
from graphgym_b200.contrib.layer.generalconv import GeneralConvLayer  # noqa: E402
from graphgym_b200.graph import get_layout  # noqa: E402
from graphgym_b200.models.layer import _SplineConvLayer  # noqa: E402


def make_step(layer, x, ei, gy, u=None):
    xg = x.clone().requires_grad_(True)

    def step():
        layer.zero_grad(set_to_none=True)
        xg.grad = None
        out = layer(xg, ei) if u is None else layer(xg, ei, u)
        out.backward(gy)
    return step


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else tempfile.mkdtemp(prefix='splineconv_probe_')
    os.makedirs(out_dir, exist_ok=True)
    print('writing to', out_dir, file=sys.stderr)
    dev = torch.device('cuda')
    n, ei = bench.gen_graph(bench.WORKLOADS['products_gcn'], dev, seed=0)
    e = ei.size(1)
    lay = get_layout(ei, n, ops.LOOPS_KEEP)
    csr, csc = lay.csr, lay.csc
    g = torch.Generator(device=dev).manual_seed(0)
    u = torch.rand(e, generator=g, device=dev)
    res = dict(probe='splineconv', nodes=n, edges=e, kernels={}, steps={})
    for k in (32, 64, 100):
        x = torch.randn(n, k, generator=g, device=dev)
        y = torch.randn(n, 2 * k, generator=g, device=dev)
        r = {}
        r['spmm_k_ms'] = timeit(lambda: ops.spmm(csr, x, reduce=ops.MEAN))
        r['spread_ms'] = timeit(lambda: ops.spline_spread(csr, x, u, mean=True))
        r['spread_over_spmm'] = r['spread_ms'] / r['spmm_k_ms']
        r['spmm_2k_ms'] = timeit(lambda: ops.spmm(csr, y, reduce=ops.MEAN))
        r['blend_ms'] = timeit(lambda: ops.spline_blend(csr, y, u, mean=True))
        r['blend_over_spmm_2k'] = r['blend_ms'] / r['spmm_2k_ms']
        r['spread_csc_ms'] = timeit(lambda: ops.spline_spread(csc, x, u, lay.weights('mean')[1]))
        r['blend_csc_ms'] = timeit(lambda: ops.spline_blend(csc, y, u, lay.weights('mean')[1]))
        r['du_ms'] = timeit(lambda: ops.spline_du(csr, u, y, k, x, 0, k), it=3, warm=1)
        res['kernels'][str(k)] = r
        print(k, r, file=sys.stderr, flush=True)
        del x, y
    for fin, fout in ((100, 128), (128, 64)):
        x = torch.randn(n, fin, generator=g, device=dev)
        gy = torch.randn(n, fout, generator=g, device=dev)
        reset_cfg()
        torch.manual_seed(0)
        gc = GeneralConvLayer(fin, fout).to(dev)
        s = {'generalconv_add_step_ms': timeit(make_step(gc, x, ei, gy), it=5, warm=2)}
        del gc
        torch.manual_seed(0)
        sp = _SplineConvLayer(fin, fout).to(dev)
        s['splineconv_step_ms'] = timeit(make_step(sp, x, ei, gy, u), it=5, warm=2)
        s['order'] = 'aggregate_first' if fin <= fout else 'transform_first'
        s['over_generalconv_add'] = s['splineconv_step_ms'] / s['generalconv_add_step_ms']
        res['steps'][f'{fin}_{fout}'] = s
        print(fin, fout, s, file=sys.stderr, flush=True)
        del sp
        # the reference's composition in fp32 on one 4 M-edge chunk (the whole [E, out] message does not fit)
        w = torch.randn(2, fin, fout, generator=g, device=dev) / fin ** 0.5
        c = 1 << 22
        src, tgt, uc = ei[0, :c], ei[1, :c], u[:c]

        def torch_chunk():
            t = torch.trunc(uc).long() % 2
            fr = (uc - torch.floor(uc)).view(-1, 1)
            c0 = torch.where(t.view(-1, 1) == 0, 1 - fr, fr)
            xj = x.index_select(0, src)
            m = c0 * (xj @ w[0]) + (1 - c0) * (xj @ w[1])
            return torch.zeros(n, fout, device=dev).index_add_(0, tgt, m)
        s['torch_chunk_4M_fwd_ms'] = timeit(torch_chunk, it=3, warm=1)
        s['torch_fwd_scaled_to_E_ms'] = s['torch_chunk_4M_fwd_ms'] * e / c
        del x, gy, w
    res['card'], res['power_limit'] = card()
    line = json.dumps(res)
    with open(os.path.join(out_dir, 'splineconv_probe.json'), 'w') as fh:
        fh.write(line + '\n')
    print(line)


if __name__ == '__main__':
    main()
