"""Times the skip stages (cfg.gnn.stage_type = 'skipsum' / 'skipconcat') on the products-shaped graph of bench.py
(2.45 M nodes, F = 128) and prints one JSON line.

  epilogue  the fused skip epilogue (functional.skip_post_ops: BN statistics, BN + skip + ReLU + row L2 forward, column
            sums and dy / dres backward) against the module chain it replaces (nn.BatchNorm1d, + or torch.cat, nn.ReLU,
            F.normalize), forward + backward, train mode, for both modes (skipconcat with a carried width p = F)
  bytes     the epilogue's byte model (each operand read or written once per kernel, below) over its time, as a fraction
            of a device-to-device copy measured in the same run
  steps     one GNN training step (forward, cross-entropy, backward) with layers_pre_mp = 1, layers_mp = 2, generalconv,
            100 -> 128, for stage_type 'stack', 'skipsum' and 'skipconcat'
CUDA events after warm-up; every [N, F] operand (1.25 GB) is larger than the L2.  The card's name and power limit are read
in the same run.  The JSON line is written to OUT_DIR (argument 1; default: a new temporary directory)."""
import json
import os
import sys
import tempfile

import torch
import torch.nn as nn
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import bench  # noqa: E402
from graphgym_b200 import functional as F_  # noqa: E402
from graphgym_b200 import ops  # noqa: E402
from graphgym_b200.config import cfg, reset_cfg  # noqa: E402
from graphgym_b200.models.gnn import GNN  # noqa: E402
from graphgym_b200.models.layer import Batch  # noqa: E402
from max_agg_probe import card, timeit  # noqa: E402


def epilogue_bytes(n, f, p, mode):
    """Least DRAM traffic of the fused epilogue (train-mode BN, L2): every operand once per kernel that needs it.
    W = output width (f, or p + f), R = residual width (f, or p).
      forward   statistics: y;  apply: y, res, out, rownorm
      backward  column sums: go, out (whole rows: the L2 dot), y, rownorm;  apply: go, out, y, rownorm, dy, dres"""
    w = f if mode == ops.SKIP_SUM else p + f
    r = f if mode == ops.SKIP_SUM else p
    fwd = 4 * n * f + 4 * n * (f + r + w) + 4 * n
    bwd = 4 * n * (2 * w + f) + 4 * n + 4 * n * (2 * w + f) + 4 * n * (f + r) + 4 * n
    return fwd + bwd


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else tempfile.mkdtemp(prefix='skip_stage_probe_')
    os.makedirs(out_dir, exist_ok=True)
    print('writing to', out_dir, file=sys.stderr)
    dev = torch.device('cuda')
    n, ei = bench.gen_graph(bench.WORKLOADS['products_gcn'], dev, seed=0)
    f = 128
    g = torch.Generator(device=dev).manual_seed(0)
    res = dict(probe='skip_stage', nodes=n, f=f, epilogue_ms={}, chain_ms={}, speedup={}, epilogue_bytes={},
               epilogue_tbps={}, epilogue_of_copy={}, steps_ms={})

    big = torch.empty(n * f * 2, device=dev)
    dst = torch.empty_like(big)
    copy_ms = timeit(lambda: dst.copy_(big), it=10, warm=3)
    res['copy_tbps'] = 2 * big.numel() * 4 / copy_ms / 1e9
    del big, dst

    y = torch.randn(n, f, generator=g, device=dev)
    for name, mode in (('skipsum', ops.SKIP_SUM), ('skipconcat', ops.SKIP_PREFIX)):
        x = torch.randn(n, f, generator=g, device=dev)
        w = f if mode == ops.SKIP_SUM else 2 * f
        gy = torch.randn(n, w, generator=g, device=dev)
        bn = nn.BatchNorm1d(f).to(dev)
        yg, xg = y.clone().requires_grad_(True), x.clone().requires_grad_(True)

        def fused():
            yg.grad = xg.grad = bn.weight.grad = bn.bias.grad = None
            F_.skip_post_ops(yg, xg, mode, bn, True, ops.ACT_RELU, 0.0, True).backward(gy)

        def chain():
            yg.grad = xg.grad = bn.weight.grad = bn.bias.grad = None
            a = bn(yg)
            h = a + xg if mode == ops.SKIP_SUM else torch.cat([xg, a], 1)
            F.normalize(torch.relu(h), p=2, dim=-1).backward(gy)

        for label, fn, d in (('fused', fused, res['epilogue_ms']), ('chain', chain, res['chain_ms'])):
            d[name] = timeit(fn, it=10, warm=3)
            print(name, label, d[name], file=sys.stderr, flush=True)
        res['speedup'][name] = res['chain_ms'][name] / res['epilogue_ms'][name]
        b = epilogue_bytes(n, f, f if mode == ops.SKIP_PREFIX else 0, mode)
        res['epilogue_bytes'][name] = b
        res['epilogue_tbps'][name] = b / res['epilogue_ms'][name] / 1e9
        res['epilogue_of_copy'][name] = res['epilogue_tbps'][name] / res['copy_tbps']
        del x, gy, yg, xg
    del y

    x = torch.randn(n, 100, generator=g, device=dev)
    labels = torch.randint(0, 47, (n,), generator=g, device=dev)
    for stage_type in ('stack', 'skipsum', 'skipconcat'):
        reset_cfg()
        cfg.gnn.stage_type, cfg.gnn.layer_type = stage_type, 'generalconv'
        cfg.gnn.layers_pre_mp, cfg.gnn.layers_mp, cfg.gnn.dim_inner = 1, 2, f
        torch.manual_seed(0)
        model = GNN(100, 47).to(dev).train()

        def step():
            model.zero_grad(set_to_none=True)
            pred, _ = model(Batch(x, ei))
            F.cross_entropy(pred, labels).backward()
        res['steps_ms'][stage_type] = timeit(step, it=5, warm=2)
        print(stage_type, res['steps_ms'][stage_type], file=sys.stderr, flush=True)
        del model
    reset_cfg()
    res['card'], res['power_limit'] = card()
    line = json.dumps(res)
    with open(os.path.join(out_dir, 'skip_stage_probe.json'), 'w') as fh:
        fh.write(line + '\n')
    print(line)


if __name__ == '__main__':
    main()
