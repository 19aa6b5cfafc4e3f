#!/usr/bin/env python
"""Headline benchmark: message-passing layer forward+backward throughput in GEdge-feat/s
(SURVEY §8d) on synthetic graphs of the shapes BASELINE.json names, through the reference's own
layer API (layer_dict[name](dim_in, dim_out, bias) + forward(batch) + backward).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl ours|reference] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  See DESIGN.md "Measurement" for every field.
  value     device-resident: inputs and the graph layout already in HBM, K timed steps (CUDA events)
  e2e       host buffers in, result out: pinned-host -> device copies of node_feature and edge_index,
            layout build, layer fwd+bwd, device -> host read of the bias gradient, every step
  roofline  the aggregation (SpMM) kernel: algorithmic bytes / CUDA-event time inside the timed steps
  cpu_baseline / --impl reference: the oracle restatement of the reference's CPU op sequence
            (gather -> scale -> index_add_ -> matmul) on a bounded sample, all host threads
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[3] graph (ogbn-products shape) under the GCN layer: the 62M-edge graph the
    # north star's scaling target is stated on.  L2 (126 MB) << feature matrix (1.25 GB).
    'products_gcn': dict(layer='gcnconv', graph='powerlaw', n=2_449_029, e_und=30_929_570, fin=100,
                         fout=128, max_deg=17_481, desc='gcnconv 100->128 on products-shaped power-law '
                         'graph (2.45M nodes, 61.9M directed edges)'),
    'products_gat': dict(layer='gatconv', graph='powerlaw', n=2_449_029, e_und=30_929_570, fin=100,
                         fout=128, max_deg=17_481, desc='gatconv 100->128 (H=1) on products-shaped '
                         'power-law graph (2.45M nodes, 61.9M directed edges)'),
    # configs[2]: BA 1M nodes / 10M directed edges, 256 hidden
    'ba1m_sage': dict(layer='sageconv', graph='ba', n=1_000_000, m=5, fin=256, fout=256,
                      desc='sageconv 256->256 on BA graph (1M nodes, 10M directed edges)'),
    'ba1m_gcn': dict(layer='gcnconv', graph='ba', n=1_000_000, m=5, fin=256, fout=256,
                     desc='gcnconv 256->256 on BA graph (1M nodes, 10M directed edges)'),
    # configs[1]: Cora-shaped, fits L2 entirely -> launch-bound, reported for completeness
    'cora_gcn': dict(layer='gcnconv', graph='uniform', n=2708, e_und=5278, fin=1433, fout=128,
                     desc='gcnconv 1433->128 on Cora-shaped graph (2708 nodes, 10556 directed edges)'),
    # configs[2] first half: ID-GNN Fast cycle-count augmentation diag(A_hat^p), p = 1..10, on the BA graph
    'ba1m_cycles': dict(aux='cycles', graph='ba', n=1_000_000, m=5, k=10,
                        desc='ID-GNN Fast cycle features diag(A_hat^1..10) on BA graph (1M nodes, 10M directed '
                             'edges): blocks of 128 source nodes, 5 hops each (half-power trick)'),
    # configs[4] / configs[0] shape: ID-GNN Full — batched 3-hop ego-net extraction, then 3 GIN-ID layers, 256 hidden
    'ego_idgin': dict(aux='ego', graph='ba_batch', graphs=256, nodes_per_graph=64, m=4, radius=3, hidden=256,
                      layers=3, desc='ID-GNN Full: 3-hop ego-nets of every node of 256 BA graphs x 64 nodes '
                                     '(reference dataset shape), then 3 ginidconv layers 256->256 fwd+bwd'),
    # configs[0] (Cfg-A, SURVEY §8d): idgcn_tf on the bundled ScaleFree graphs [0:16] (committed fixture
    # tests/golden/scalefree16.npz, made from /root/reference/datasets/scalefree.pkl), 3-hop ego-nets, X = ones [N,1],
    # pre_mp-free stack of 3 gcnidconv GeneralLayers 1 -> 128 -> 128 -> 128 (BN + ReLU, stage L2 norm), fwd + bwd
    'scalefree_idgcn': dict(aux='cfg_a', fixture='tests/golden/scalefree16.npz', radius=3, hidden=128, layers=3,
                            desc='idgcn_tf (ID-GNN Full GCN): 16 bundled ScaleFree graphs x 64 nodes, 3-hop ego-nets, '
                                 '3 gcnidconv GeneralLayers 1->128->128->128 (BN, ReLU, L2), fwd+bwd'),
}
DEFAULT_WORKLOAD = 'products_gcn'
DEFAULT_HALO = 'sliced'
# dram__bytes_read.sum + dram__bytes_write.sum of ONE aggregation launch from an `ncu --set full` capture of this bench
# (profiles/r02_spmm_sell128_bench_ncu_raw.csv: spmm_sell_kernel<32,1,0> 18.58 + 1.27 GB in 3.26 ms = 6.1 TB/s = 0.93 of
# the measured copy peak; the algorithmic figure is 34.7 GB — the L2 serves the rest).  Keyed by (workload, kernel): a
# line produced with another aggregation kernel reports null.
NCU_TRAFFIC = {('products_gcn', 'sell'): 19_850_000_000, ('products_gcn', 'mpg'): 18_829_800_000,
               # profiles/r02_gat_onepass_launches.csv: per-node pass + walk + fix-up; training forward + fix-up
               ('products_gat', 'bwd_one'): 29_894_374_912, ('products_gat', 'fwd_train'): 24_095_261_440}
HALO_DESC = {
    'allgather': 'halo all-gather of the feature rows over NCCL, rank-local SpMM',
    'pipelined': 'P-1 NCCL send/recv rounds overlapped with the per-peer SpMMs',
    'sliced': 'feature-sliced transposition over NVLink peer memory (column-scatter kernel out, SpMM epilogue '
              'stores finished rows to their owners, flag barrier; no NCCL on the data path)',
    'sliced_nccl': 'feature-sliced transposition over two NCCL all-to-alls around a full-graph SpMM of F/P columns',
}


# ------------------------------------------------------------------------------------------------
# synthetic graphs (seeded; torch ops so the big ones can be drawn on the GPU in < 1 s)
# ------------------------------------------------------------------------------------------------
def gen_graph(spec, device, seed=0, scale=1.0):
    """-> edge_index [2,E] int64 on `device` (symmetric: both directions of every undirected edge).
    `scale` < 1 shrinks nodes and edges together (the CPU-baseline sample of the same family)."""
    g = torch.Generator(device=device).manual_seed(seed)
    n = max(8, int(spec['n'] * scale))
    if spec['graph'] == 'powerlaw':
        m = max(8, int(spec['e_und'] * scale))
        w = torch.arange(1, n + 1, device=device, dtype=torch.float64).pow(-1.0 / 1.1)  # exponent 2.1
        cap = min(float(spec['max_deg']), n / 8.0)
        for _ in range(4):  # expected degree sequence: mean 2m/n, clipped at max_deg
            w = (w * (2.0 * m / w.sum())).clamp(max=cap)
        cdf = torch.cumsum(w / w.sum(), 0)
        a = torch.searchsorted(cdf, torch.rand(m, device=device, dtype=torch.float64, generator=g)).clamp(max=n - 1)
        b = torch.searchsorted(cdf, torch.rand(m, device=device, dtype=torch.float64, generator=g)).clamp(max=n - 1)
        perm = torch.randperm(n, device=device, generator=g)  # hubs are not the low ids
        a, b = perm[a], perm[b]
    elif spec['graph'] == 'ba':
        m0 = spec['m']
        k = torch.arange(m0 * (n - m0), device=device)
        t = m0 + k // m0
        limit = 2 * m0 * (t - m0)  # endpoint-list entries that exist before node t arrives
        r = (torch.rand(k.numel(), device=device, dtype=torch.float64, generator=g) * limit.clamp(min=1)).long()
        ptr, even = r // 2, (r % 2 == 0)
        tgt = torch.full_like(k, -1)
        first = limit == 0
        tgt[first] = torch.randint(0, m0, (int(first.sum()),), device=device, generator=g)
        sel = even & ~first
        tgt[sel] = m0 + ptr[sel] // m0
        while True:  # odd entries point at an earlier edge's target: pointer-jump until resolved
            idx = torch.nonzero(tgt < 0).flatten()
            if idx.numel() == 0:
                break
            tgt[idx] = tgt[ptr[idx]]
        a, b = t, tgt
    else:  # 'uniform': distinct undirected pairs, uniformly at random
        m = max(4, int(spec['e_und'] * scale))
        a = torch.randint(0, n, (4 * m,), device=device, generator=g)
        b = torch.randint(0, n, (4 * m,), device=device, generator=g)
        keep = a < b
        code = torch.unique(a[keep] * n + b[keep])
        code = code[torch.randperm(code.numel(), device=device, generator=g)[:m]]
        a, b = code // n, code % n
    return n, torch.stack([torch.cat([a, b]), torch.cat([b, a])]).contiguous()


def gen_features(n, f, device, seed=0):
    g = torch.Generator(device=device).manual_seed(seed + 1)
    return torch.randn(n, f, device=device, generator=g)


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')

    def __init__(self, index=0, enabled=True):
        # only the rank that prints the line samples: eight nvidia-smi pollers at 20 ms contend for the driver and the
        # host cores the ranks need to enqueue their own work
        self.samples, self.proc, self.index, self.enabled = [], None, index, enabled

    def __enter__(self):
        if not self.enabled:
            return self
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.QUERY}',
                                          '--format=csv,noheader,nounits', '-lms', '20'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append([c.strip() for c in line.split(',')])

    def __exit__(self, *exc):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            self.thread.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for s in self.samples:
            try:
                sm.append(float(s[0])); mx.append(float(s[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(names, s[2:6]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': max(mx), 'reasons': sorted(reasons),
                'samples': len(sm)}


# ------------------------------------------------------------------------------------------------
# the measured step
# ------------------------------------------------------------------------------------------------
def edge_feat_per_step(layer_name, n, num_slots, fin, fout):
    """E' x F_agg x 2 passes (SURVEY §8d): GCN/GAT aggregate F_out-wide, SAGE/GIN F_in-wide."""
    f_agg = fout if layer_name in ('gcnconv', 'gatconv', 'gcnidconv', 'gatidconv', 'idconv') else fin
    return num_slots * f_agg * 2, f_agg


def spmm_bytes(n, slots, f, weighted, gather_bytes=4):
    """Algorithmic bytes of one aggregation launch (SURVEY §8d): gathered rows + output rows + nbr
    indices + rowptr (+ per-slot weights); ``gather_bytes`` = 2 in the bf16-gather mode."""
    return slots * f * gather_bytes + n * f * 4 + slots * 4 + (n + 1) * 4 + (slots * 4 if weighted else 0)


def gat_pass_bytes(kind, n, slots, f):
    """Algorithmic bytes of the fused GAT passes (counted like spmm_bytes: every gathered row counts).
    fwd (training): per slot the index, the source logit half and the gathered h row; per row a_tgt, out, out_pos,
    (max, sum), a_pos.  bwd: the per-node pass reads g, out, out_pos rows and writes the 16-byte record and da_tgt; the
    walk reads per slot the index, the target's record and the gathered g row, per row h_j, a_src, da_tgt and writes dh,
    da_src."""
    if kind == 'fwd':
        return slots * (4 + 4 + f * 4) + n * (4 + 2 * f * 4 + 8 + 4) + (n + 1) * 4
    return n * (3 * f * 4 + 8 + 4 + 4 + 16 + 4) + slots * (4 + 16 + f * 4) + n * (f * 4 + 4 + 4 + f * 4 + 4) + (n + 1) * 4


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


def loop_policy_for(layer_name):
    from graphgym_b200 import ops
    return {'gcnconv': ops.LOOPS_ADD_REMAINING, 'gcnidconv': ops.LOOPS_ADD_REMAINING,
            'gatconv': ops.LOOPS_REMOVE_ADD, 'gatidconv': ops.LOOPS_REMOVE_ADD,
            'ginidconv': ops.LOOPS_REMOVE}.get(layer_name, ops.LOOPS_KEEP)


def _event_ms(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(steps):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / steps


def gen_ba_batch(spec, device, seed=0):
    """Block-diagonal batch of small BA graphs (the reference's synthetic datasets are 64-node graphs,
    ref: syn_graph.py): -> n, edge_index [2,E] int64 symmetric, graph_ptr [G+1]."""
    G, nn_, m0 = spec['graphs'], spec['nodes_per_graph'], spec['m']
    g = torch.Generator(device=device).manual_seed(seed)
    t = torch.arange(m0, nn_, device=device).repeat_interleave(m0)            # arriving node of every edge
    # preferential attachment approximated per graph by sampling an earlier node with weight ~ (1 + index^-0.5)
    r = torch.rand((G, t.numel()), device=device, generator=g)
    tgt = (r * r * t.unsqueeze(0)).long().clamp(max=nn_ - 1)                  # skewed towards early (high-degree) nodes
    tgt = torch.minimum(tgt, t.unsqueeze(0) - 1)
    off = (torch.arange(G, device=device) * nn_).unsqueeze(1)
    a = (t.unsqueeze(0) + off).reshape(-1)
    b = (tgt + off).reshape(-1)
    code = torch.unique(torch.minimum(a, b) * (G * nn_) + torch.maximum(a, b))   # simple graphs: no duplicate edges
    a, b = code // (G * nn_), code % (G * nn_)
    ei = torch.stack([torch.cat([a, b]), torch.cat([b, a])]).contiguous()
    return G * nn_, ei, torch.arange(G + 1, device=device, dtype=torch.int32) * nn_


def _aux_dist(world, dev):
    """Secondary workloads shard by independent units (SURVEY §8e): no data-path collective; the process group only
    carries the timing barrier, the max-over-ranks reduction and, for the trained stack, the dW all-reduce."""
    import torch.distributed as dist
    if world > 1 and not dist.is_initialized():
        dist.init_process_group('nccl', device_id=dev)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def reduce(v, op):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=op)
        return float(t.item())
    return sync_all, (lambda v: reduce(v, dist.ReduceOp.MAX)), (lambda v: reduce(v, dist.ReduceOp.SUM))


def _timed_steps(fn, steps, warmup, sync_all, max_over_ranks):
    for _ in range(warmup):
        fn()
    sync_all()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(steps):
        fn()
    e.record()
    sync_all()
    return max_over_ranks(s.elapsed_time(e)) / steps


DUMP_BYTES = 60_000_000   # --dump-outputs writes at most this much (array data; each .npy header adds 128 bytes)


def dump_outputs(path, rows=None, whole=None):
    """--dump-outputs: write every array as path/<name>.npy in float32 (float64 stays float64).  ``whole`` arrays are
    written whole; the per-node arrays in ``rows`` keep one seeded sample of their rows, as many as fit DUMP_BYTES, so that
    two builds run with the same arguments write files that compare element for element."""
    rows, whole = rows or {}, whole or {}
    host = lambda t: t.detach().cpu().numpy() if t.dtype == torch.float64 else t.detach().float().cpu().numpy()
    out = {name: host(t) for name, t in whole.items()}
    if rows:
        n = next(iter(rows.values())).size(0)
        row_bytes = sum(t[0].numel() * (8 if t.dtype == torch.float64 else 4) for t in rows.values())
        keep = min(n, (DUMP_BYTES - sum(a.nbytes for a in out.values())) // row_bytes)
        pick = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:keep].sort().values
        out.update({name: host(t[pick.to(t.device)]) for name, t in rows.items()})
    os.makedirs(path, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(path, name + '.npy'), a)


def cpu_cycles_baseline(seconds):
    """The reference algorithm itself (identity.py:25-35: dense A_hat, k-1 dense matmuls) on BA graphs of growing size; at
    1M nodes it is infeasible (n^2 floats = 4 TB)."""
    from oracle import identity as oid
    torch.set_num_threads(os.cpu_count() or 1)
    out, t_all = [], time.time()
    for n in (64, 2708, 8192, 16384):
        if n > 8192 and seconds < 120:
            out.append({'nodes': n, 'skipped': 'about 60 s of dense matmul on 16 cores: run with --cpu-seconds >= 120'})
            continue
        _, ei = gen_graph(dict(graph='ba', n=n, m=5), torch.device('cpu'), seed=0)
        t0 = time.time()
        oid.compute_identity(ei, n, 10)
        dt = time.time() - t0
        out.append({'nodes': n, 'seconds': round(dt, 4), 'nodes_per_s': round(n / dt, 1)})
    return {'kind': 'port', 'cores': os.cpu_count() or 1, 'unit': 'nodes/s', 'value': out[2].get('nodes_per_s'),
            'sample': 'oracle/identity.py = dense compute_identity of the reference (k = 10) on BA graphs (m = 5) of '
                      '64 / 2708 / 8192 / 16384 nodes; the 1M-node workload graph is out of reach for it (O(n^3), 4 TB)',
            'sizes': out, 'wall_s': round(time.time() - t_all, 1)}


def cpu_ego_baseline(ei_cpu, n, radius, graph_ptr=None, max_centres=512):
    """nx.ego_graph per centre + induced-subgraph copy, as the reference's ego_nets does (transform.py:11-38), on the
    workload's own graphs (a bounded number of centres)."""
    import networkx as nx
    G = nx.Graph()
    G.add_nodes_from(range(n))
    G.add_edges_from(ei_cpu.t().tolist())
    centres = list(range(0, n, max(1, n // max_centres)))[:max_centres]
    t0 = time.time()
    nodes = edges = 0
    for c in centres:
        ego = nx.ego_graph(G, c, radius=radius)
        sub = nx.Graph(ego)       # the reference copies every ego into the output graph with fresh ids
        nodes += sub.number_of_nodes()
        edges += sub.number_of_edges()
    dt = time.time() - t0
    return {'kind': 'reference-algorithm (networkx)', 'cores': 1, 'unit': 'centres/s', 'value': round(len(centres) / dt, 1),
            'ms_per_centre': round(1e3 * dt / len(centres), 3), 'output_edges_per_s': round(edges / dt, 1),
            'sample': f'{len(centres)} of {n} centres, radius {radius}, nx.ego_graph + subgraph copy (transform.py:20-36)'}


def cpu_stack_baseline(spec, x_cpu, ei_cpu, ids_cpu, dims, layer_name, seconds):
    """fwd+bwd of the layer stack with the oracle layers + torch BN / ReLU / normalize on the host (the reference's own
    module sequence, layer.py:26-46), all host threads."""
    import torch.nn.functional as Fn
    from oracle import layers as olayers
    torch.set_num_threads(os.cpu_count() or 1)
    g = torch.Generator().manual_seed(0)
    params = []
    for din, dout in zip(dims[:-1], dims[1:]):
        mk = lambda *s: (torch.randn(*s, generator=g) * 0.1).requires_grad_(True)
        if layer_name == 'gcnidconv':
            params.append((mk(din, dout), mk(din, dout)))
        else:   # ginidconv: nn / nn_id = Linear, ReLU, Linear
            params.append(tuple(mk(*s) for s in ((dout, din), (dout,), (dout, dout), (dout,)) * 2))
    bns = [torch.nn.BatchNorm1d(d) for d in dims[1:]]
    gy = torch.randn(x_cpu.size(0), dims[-1], generator=g)

    def step():
        h = x_cpu
        for i, p in enumerate(params):
            if layer_name == 'gcnidconv':
                h = olayers.gcn_idconv(h, ei_cpu, ids_cpu, p[0], p[1], None)
                h = torch.relu(bns[i](h))
            else:
                h = torch.relu(olayers.gin_idconv(h, ei_cpu, ids_cpu, p[:4], p[4:]))
        if layer_name == 'gcnidconv':
            h = Fn.normalize(h, p=2, dim=1)
        h.backward(gy)
    t, done = _time_cpu_steps(step, seconds, None, 1)
    return t, done


def run_aux(args, spec, dev, rank=0, world=1):
    """Secondary hot-path rows (SURVEY §8a rows 10-11, Cfg-A / Cfg-C / Cfg-E): their own units, same JSON shape.  With
    --gpus N every rank works on its own units (source blocks / graphs): weak scaling, no data-path collective."""
    from graphgym_b200 import ops, parallel
    from graphgym_b200.contrib.transform import identity as gid
    from graphgym_b200.models import transform as gtr
    from graphgym_b200.models.layer import Batch, layer_dict
    peak, peak_src = load_peaks()
    clocks = ClockSampler(dev.index or 0, enabled=(rank == 0))
    sync_all, max_over_ranks, sum_over_ranks = _aux_dist(world, dev)
    par = 'single GPU' if world == 1 else f'{world} GPUs, independent units per rank (no data-path collective)'
    if spec['aux'] == 'cycles':
        n, ei = gen_graph(spec, dev, seed=0)
        k = spec['k']
        csr = ops.layout_build(ei, n, ops.LOOPS_ADD_REMAINING, ops.BY_TARGET)
        csc = ops.layout_build(ei, n, ops.LOOPS_ADD_REMAINING, ops.BY_SOURCE)
        w = ops.gcn_norm(csr, ops.segment_degree(csc))
        L = ops.lib()
        item_row, item_slot, items = csr.plan
        use_mp = gid.MP_STEP
        use_sell = gid.CYCLE_STEP == 'sell'
        if use_sell:
            sl = ops.sell_layout(csr)
            w_sell = sl.weights(w)
            ws = torch.empty(int(L.gg_cycle_diag_sell_workspace_bytes(n, sl.partial_rows)), dtype=torch.uint8, device=dev)
        else:
            ws = torch.empty(int(L.gg_cycle_diag_mp_workspace_bytes(n, items)), dtype=torch.uint8, device=dev)
        out = torch.empty((128, k), dtype=torch.float32, device=dev)
        blk = [rank]

        def one_block():   # 128 consecutive sources: 5 hops over the whole graph + 10 dot products; rank r takes blocks r, r+P, ...
            sb = (blk[0] * 128) % (n - 128)
            blk[0] += world
            if use_sell:
                ops.check(L.gg_cycle_diag_sell_f32(ops._ptr(csr.rowptr), ops._ptr(sl.chunk_ptr), sl.chunks, ops._ptr(sl.idx),
                                                   ops._ptr(w_sell), ops._ptr(sl.vdst), ops._ptr(sl.hub_rows),
                                                   ops._ptr(sl.hub_pptr), sl.hubs, sl.partial_rows, n, k, 1, sb, 128,
                                                   ops._ptr(out), k, ops._ptr(ws), ws.numel(), ops._stream()),
                          'gg_cycle_diag_sell_f32')
            elif use_mp:
                ops.check(L.gg_cycle_diag_mp_f32(ops._ptr(csr.rowptr), ops._ptr(csr.nbr), ops._ptr(w), ops._ptr(item_row),
                                                 ops._ptr(item_slot), items, n, k, 1, sb, 128, ops._ptr(out), k,
                                                 ops._ptr(ws), ws.numel(), ops._stream()), 'gg_cycle_diag_mp_f32')
            else:
                ops.check(L.gg_cycle_diag_f32(ops._ptr(csr.rowptr), ops._ptr(csr.nbr), ops._ptr(w), 0, n, k, 1, sb, 128,
                                              ops._ptr(out), k, ops._ptr(ws), ws.numel(), ops._stream()), 'gg_cycle_diag_f32')
        launches0 = ops.launch_count()
        with clocks:
            ms = _timed_steps(one_block, args.steps, args.warmup, sync_all, max_over_ranks)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, whole={'diag': out})   # the last timed block's diag(A_hat^1..k)
        launches = int(sum_over_ranks((ops.launch_count() - launches0) * args.steps // (args.steps + args.warmup)))
        hops = (k + 1) // 2
        slots = csr.num_slots
        visits = slots * 128 * hops * world
        step_bytes = hops * (slots * 512 + n * 512 + slots * 8 + (n + 1) * 4) + k * 2 * n * 512
        ach = step_bytes / (ms * 1e-3) / 1e9
        cpu = cpu_cycles_baseline(args.cpu_seconds) if (rank == 0 and not args.no_cpu and world == 1) else None
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
            dist.destroy_process_group()
        return {'metric': 'cycle-feature edge-visits/s (one visit = one slot x one source column x one hop)',
                'value': round(visits / (ms * 1e-3) / 1e9, 3), 'unit': 'G edge-visits/s', 'n_gpus': world,
                'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': round(ms, 4), 'higher_is_better': True,
                'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic (seeded BA generator in bench.py)',
                'config': {'workload': spec['desc'], 'nodes': n, 'slots': slots, 'k': k, 'sources_per_step_per_gpu': 128,
                           'parallelism': par,
                           'whole_graph_seconds': round(ms * 1e-3 * (n / 128) / world, 1),
                           'l2_policy': 'inputs larger than L2 (two 512 MB walk matrices)'},
                'clocks': clocks.summary(), 'e2e': None, 'gpu_launches': launches,
                'roofline': {'bound': 'hbm', 'kernel': ('spmm_sell_kernel' if use_sell else 'spmm_mpg_kernel' if use_mp else 'walk_step_kernel') + ' (+ walk_dot) over one block of 128 sources (per GPU)',
                             'achieved': round(ach, 1), 'peak': peak, 'unit': 'GB/s', 'frac': round(ach / peak, 4),
                             'traffic': None, 'peak_source': peak_src, 'algorithmic_bytes_per_step': step_bytes},
                'cpu_baseline': cpu}
    # ---- ID-GNN Full: ego-net extraction + a stack of ID layers (Cfg-E: synthetic BA batch + ginidconv; Cfg-A: fixture + gcnidconv)
    cfg_a = spec['aux'] == 'cfg_a'
    if cfg_a:
        d = np.load(os.path.join(ROOT, spec['fixture']))
        ei = torch.from_numpy(d['edge_index']).to(dev)
        gptr = torch.from_numpy(d['graph_ptr']).to(dev).int()
        n = int(d['graph_ptr'][-1])
        layer_name, dims = 'gcnidconv', [1] + [spec['hidden']] * spec['layers']
    else:
        n, ei, gptr = gen_ba_batch(spec, dev, seed=rank)      # every rank its own graphs (data parallel over graphs)
        layer_name, dims = 'ginidconv', [spec['hidden']] * (spec['layers'] + 1)
    radius, nl = spec['radius'], spec['layers']
    res = gtr.ego_nets_batch(ei, n, radius, gptr)     # warm + sizes
    torch.cuda.synchronize()
    n_out, e_out = res['num_nodes'], int(res['edge_index'].size(1))
    checks = None
    if cfg_a:   # sizes of the reference's own ego expansion (transform.py run by tests/golden/make_golden.py)
        per_graph = (res['out_node_ptr'][1:] - res['out_node_ptr'][:-1]).cpu().numpy()
        checks = {'ego_nodes_equal_reference': bool(np.array_equal(per_graph, d['ego_nodes'])),
                  'ego_edges_equal_reference': bool(e_out == 2 * int(d['ego_undirected_edges'].sum()))}
    from graphgym_b200.config import cfg as gg_cfg, reset_cfg
    from graphgym_b200.models.gnn import GNNStackStage
    reset_cfg()
    with clocks:
        ego_ms = _timed_steps(lambda: gtr.ego_nets_batch(ei, n, radius, gptr), max(3, args.steps // 2), 2, sync_all,
                              max_over_ranks)
        torch.manual_seed(0)
        eo, ids = res['edge_index'], res['node_id_index']
        if cfg_a:
            stages = [GNNStackStage(1, spec['hidden'], nl, 'gcnidconv').to(dev)]
            x = torch.ones(n_out, 1, device=dev)                                  # node_feature = tensor([1.]) per node
        else:
            stages = [layer_dict['ginidconv'](dims[i], dims[i + 1], bias=True).to(dev) for i in range(nl)]
            x = gen_features(n_out, dims[0], dev, seed=rank)
        gy = gen_features(n_out, dims[-1], dev, seed=7 + rank)
        keep = {} if args.dump_outputs else None   # the latest step's results, held only to be dumped

        def step():
            for l in stages:
                l.zero_grad(set_to_none=True)
            h = x.detach().requires_grad_(True)
            b = Batch(h, eo, ids)
            for l in stages:
                b = l(b)
                if not cfg_a:
                    b.node_feature = torch.relu(b.node_feature)   # GeneralLayer's activation (ref: layer.py:31-33)
            b.node_feature.backward(gy)
            if world > 1:
                for l in stages:
                    parallel.allreduce_grads(l)
            if keep is not None:
                keep.update(rows={'out': b.node_feature.detach(), 'grad_x': h.grad},
                            whole={f'grad_{i}.{k}': p.grad for i, l in enumerate(stages)
                                   for k, p in l.named_parameters() if p.grad is not None})
        launches0 = ops.launch_count()
        ms = _timed_steps(step, args.steps, args.warmup, sync_all, max_over_ranks)
    if keep is not None:
        dump_outputs(args.dump_outputs, **keep)
    launches = int(sum_over_ranks((ops.launch_count() - launches0) * args.steps // (args.steps + args.warmup)))
    slots_per_layer = e_out + (n_out if cfg_a else 0)      # gcnidconv adds the remaining self loops
    ef_rank = sum(slots_per_layer * (dims[i + 1] if cfg_a else dims[i]) * 2 for i in range(nl))
    ef = sum_over_ranks(ef_rank)
    ego_bytes = e_out * 8 + n_out * 8 + int(ei.size(1)) * 4   # output edges (2 x int64 written) + ids + adjacency read
    cpu = None
    if rank == 0 and not args.no_cpu and world == 1:
        ei_cpu = ei.cpu()
        cpu_ego = cpu_ego_baseline(ei_cpu, n, radius)
        t_cpu, done = cpu_stack_baseline(spec, x.cpu(), eo.cpu(), ids.cpu(), dims, layer_name, min(args.cpu_seconds, 20.0))
        cpu = {'value': round(ef_rank / t_cpu / 1e9, 4), 'unit': 'GEdge-feat/s', 'cores': os.cpu_count() or 1, 'kind': 'port',
               'ms_per_step': round(t_cpu * 1e3, 2), 'steps': done,
               'sample': f'the same ego batch ({n_out} nodes, {e_out} directed edges), {nl} x {layer_name} fwd+bwd with the '
                         'oracle layers + torch BN / ReLU / normalize on the host, all threads',
               'ego_extraction': cpu_ego}
    out = {'metric': 'layer fwd+bwd GEdge-feat/s', 'value': round(ef / (ms * 1e-3) / 1e9, 3), 'unit': 'GEdge-feat/s',
           'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': round(ms, 4),
           'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
           'data': ('bundled reference fixture (datasets/scalefree.pkl graphs [0:16], committed as tests/golden/scalefree16.npz)'
                    if cfg_a else 'synthetic (seeded BA-batch generator in bench.py)') + '; random-init weights',
           'config': {'workload': spec['desc'], 'centres_per_gpu': n, 'ego_batch_nodes_per_gpu': n_out,
                      'ego_batch_edges_directed_per_gpu': e_out, 'dims': dims, 'layers': nl, 'layer': layer_name,
                      'parallelism': par + ('' if world == 1 else '; dW all-reduced every step (data parallel over graphs)'),
                      'l2_policy': ('inputs larger than L2 (feature matrix %.0f MB)' % (n_out * dims[-1] * 4 / 1e6))
                      if n_out * dims[-1] * 4 > 126e6 else 'working set fits L2 (%.0f MB): launch / latency bound' % (n_out * dims[-1] * 4 / 1e6)},
           'clocks': clocks.summary(), 'e2e': None, 'gpu_launches': launches,
           'ego_extraction': {'ms': round(ego_ms, 3), 'centres_per_s': round(n * world / (ego_ms * 1e-3), 1),
                              'output_edges_per_s': round(e_out * world / (ego_ms * 1e-3), 1),
                              'output_GBps_per_gpu': round(ego_bytes / (ego_ms * 1e-3) / 1e9, 2),
                              'includes': 'adjacency layout build, sizes pass, fill pass (two kernel launches + scans)'},
           'roofline': None, 'cpu_baseline': cpu, 'reference_checks': checks}
    reset_cfg()
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    return out


def gpu_comparators(name, n, ei, x, gy, fin, fout, lay, policy, ef, dev):
    """GPU library formulations of the same layer step on the same box and shape (SURVEY §2b: the bar to beat):
    torch index_select + index_add_ (the reference's own op sequence on the GPU), torch.sparse CSR @ dense (cuSPARSE),
    and torch.matmul (cuBLAS) for the dense transforms.  Library kernels only; nothing of this runs on the product path."""
    from graphgym_b200 import ops
    if name != 'gcnconv':
        return None
    out = {}
    try:
        torch.manual_seed(0)
        w = torch.randn(fin, fout, device=dev) * 0.1
        csr, csc = lay.csr, lay.csc
        w_csr, w_csc = lay.weights('gcn_tgt')
        src, tgt = csr.nbr.long(), csr.rowid.long()

        def scatter_step():
            h = x @ w
            o = torch.zeros_like(h).index_add_(0, tgt, h.index_select(0, src) * w_csr.view(-1, 1))
            gh = torch.zeros_like(h).index_add_(0, src, gy.index_select(0, tgt) * w_csr.view(-1, 1))
            return o, gh @ w.t(), x.t() @ gh
        ms = _event_ms(scatter_step, 3, 1)
        out['torch_index_select_index_add'] = {'ms_per_step': round(ms, 3), 'value': round(ef / (ms * 1e-3) / 1e9, 2)}
        del src, tgt
        a = torch.sparse_csr_tensor(csr.rowptr.long(), csr.nbr.long(), w_csr, (n, n))
        at = torch.sparse_csr_tensor(csc.rowptr.long(), csc.nbr.long(), w_csc, (n, n))

        def sparse_step():
            h = x @ w
            o = a @ h
            gh = at @ gy
            return o, gh @ w.t(), x.t() @ gh
        ms = _event_ms(sparse_step, 3, 1)
        h = x @ w
        ms_spmm = _event_ms(lambda: a @ h, 5, 2)
        out['torch_sparse_csr_cusparse'] = {'ms_per_step': round(ms, 3), 'value': round(ef / (ms * 1e-3) / 1e9, 2),
                                            'spmm_ms': round(ms_spmm, 3)}
        ms_ours = _event_ms(lambda: ops.spmm(csr, h, w_csr), 5, 2)
        out['ours_spmm_ms'] = round(ms_ours, 3)
        ms_mm = _event_ms(lambda: x @ w, 10, 3)
        ms_ours_mm = _event_ms(lambda: ops.id_gemm([(x, w, None)], n, fout), 10, 3)
        out['torch_matmul_cublas_fp32'] = {'gemm_ms': round(ms_mm, 3), 'ours_tc_gemm_ms': round(ms_ours_mm, 3),
                                           'allow_tf32': bool(torch.backends.cuda.matmul.allow_tf32)}
        out['unit'] = 'GEdge-feat/s for `value` (same E\' x F x 2 numerator as the headline)'
    except Exception as exc:  # noqa: BLE001 - a comparator must never take the bench line down
        out['error'] = f'{type(exc).__name__}: {exc}'
    return out


def run_ours(args, spec, rank, world, dev):
    import torch.distributed as dist

    from graphgym_b200 import ops, parallel
    from graphgym_b200.graph import clear_cache, get_layout
    from graphgym_b200.models.layer import Batch, layer_dict
    name, fin, fout = spec['layer'], spec['fin'], spec['fout']
    multi = world > 1
    from graphgym_b200.config import cfg as gg_cfg
    gg_cfg.b200.gather_dtype = args.gather_dtype
    half = args.gather_dtype == 'bf16' and not multi
    if multi:
        if name not in parallel.ROW_PARTITIONED:
            raise SystemExit(f'--gpus {world}: the row-partitioned path serves {sorted(parallel.ROW_PARTITIONED)} '
                             f'(got {name}); run this workload with --gpus 1')
        dist.init_process_group('nccl', device_id=dev)
    t0 = time.time()
    n, ei = gen_graph(spec, dev, seed=0)
    x = gen_features(n, fin, dev)
    gy = gen_features(n, fout, dev, seed=7)
    if multi:  # every rank must see the same bits: rank 0's draw wins
        for t in (ei, x, gy):
            dist.broadcast(t, src=0)
    torch.manual_seed(0)
    part = parallel.RowPartition(n, world, rank)
    if multi:
        layer = parallel.ROW_PARTITIONED[name][0](fin, fout, bias=True).to(dev)
        x_loc, gy_loc = x[part.lo:part.hi].contiguous(), gy[part.lo:part.hi].contiguous()
    else:
        layer = layer_dict[name](fin, fout, bias=True).to(dev)
        x_loc, gy_loc = x, gy
    ids = torch.arange(0, n, 64, device=dev) if 'id' in name else None
    torch.cuda.synchronize()
    gen_s = time.time() - t0
    policy = loop_policy_for(name)

    def sync_all():
        torch.cuda.synchronize()
        if multi:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(v):
        if not multi:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(v):
        if not multi:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---- device-resident steps -------------------------------------------------------------
    spmm_events = []
    orig_spmm = ops.spmm

    def timed_spmm(*a, **k):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        out = orig_spmm(*a, **k)
        e.record()
        spmm_events.append((s, e))
        return out

    # the fused GAT passes (single GPU, heads = 1) do not go through ops.spmm: time them the same way
    gat_events = {'fwd': [], 'bwd': []}
    orig_gat = (ops.gat_sell_forward, ops.gat_sell_backward_one)

    def _timed(fn, key):
        def run(*a, **k):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            out = fn(*a, **k)
            e.record()
            gat_events[key].append((s, e))
            return out
        return run

    def bias_grad():  # the small result read back by the e2e leg: the gradient of the layer's bias
        for pname, prm in layer.named_parameters():
            if pname.endswith('bias'):
                return prm.grad
        return next(layer.parameters()).grad

    keep = {} if args.dump_outputs else None   # the latest step's results, held only until the timed steps are dumped

    def step(x_dev, ei_dev, playout=None):
        layer.zero_grad(set_to_none=True)
        # the layer input needs its gradient: message-passing layers sit behind pre_mp / earlier layers
        # (ref: gnn.py:165-168), so the backward includes dX = dH W^T as well as dW, dbias
        x_dev = x_dev.detach().requires_grad_(True)
        if multi:
            y = layer(x_dev, playout, ids) if ids is not None else layer(x_dev, playout)
            y.backward(gy_loc)
            parallel.allreduce_grads(layer)
        else:
            b = layer(Batch(x_dev, ei_dev, ids))
            y = b.node_feature
            y.backward(gy_loc)
        if keep is not None:
            keep.update(rows={'out': y.detach(), 'grad_x': x_dev.grad},
                        whole={'grad_' + k: p.grad for k, p in layer.named_parameters() if p.grad is not None})
        return bias_grad()

    t0 = time.time()
    # allgather | pipelined (per-peer send/recv rounds) | sliced (feature-sliced transposition over peer memory,
    # SpMM epilogue stores to the owners) | sliced_nccl (same over all_to_all)
    halo = os.environ.get('GG_HALO', DEFAULT_HALO)
    agg_kind = parallel.ROW_PARTITIONED[name][2] if multi else None
    f_exchanged = fout if name in ('gcnconv', 'gatconv') else fin
    if multi and halo.startswith('sliced') and not parallel.sliced_width(f_exchanged, world):
        halo = 'allgather'
    if multi and halo == 'sliced':
        # peer memory needs CUDA IPC between the ranks' processes: probe it once, all ranks agree on the outcome
        ok = 1
        try:
            parallel.PeerPool.shared(part).barrier()
            torch.cuda.synchronize()
        except Exception as exc:  # noqa: BLE001
            print(f'[bench] rank {rank}: peer memory unavailable ({type(exc).__name__}: {exc}); '
                  'falling back to the NCCL all-to-all form', file=sys.stderr)
            ok = 0
        flag = torch.tensor([ok], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0:
            halo = 'sliced_nccl'
    mk_layout = lambda e: parallel.PartitionedLayout(e, n, policy, part, exchange=halo)
    warm_weights = lambda pl: pl.sub_weights(agg_kind) if pl.pipelined else pl.weights(agg_kind)
    if multi:
        playout = mk_layout(ei)
        warm_weights(playout)
        slots_local, rows_local = playout.csr.num_slots, part.rows
        if playout.sliced:   # every rank aggregates F/P columns of ALL rows
            rows_local = n
    else:
        playout = None
        lay = get_layout(ei, n, policy)
        slots_local, rows_local = lay.csr.num_slots, n
        _ = lay.csc
    slots = slots_local if (multi and playout.sliced) else int(sum_over_ranks(slots_local))
    torch.cuda.synchronize()
    layout_first_s = time.time() - t0
    clocks = ClockSampler(dev.index or 0, enabled=(rank == 0))
    clocks.__enter__()   # sampled at 20 ms from the warm-up on: short timed regions still get samples under load
    for _ in range(args.warmup):
        step(x_loc, ei, playout)
    sync_all()
    ops.spmm = timed_spmm
    ops.gat_sell_forward, ops.gat_sell_backward_one = _timed(orig_gat[0], 'fwd'), _timed(orig_gat[1], 'bwd')
    if multi:
        parallel.trace_report()   # GG_PEER_TRACE: only the timed steps are reported
    launches0 = ops.launch_count()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    start.record()
    t_host = time.perf_counter()
    for _ in range(args.steps):
        step(x_loc, ei, playout)
    host_ms = (time.perf_counter() - t_host) * 1e3 / args.steps    # time to ENQUEUE a step: ~ms_per_step => host bound
    end.record()
    sync_all()
    ops.spmm = orig_spmm
    ops.gat_sell_forward, ops.gat_sell_backward_one = orig_gat
    exchange_trace = parallel.trace_report() if (multi and parallel._TRACE) else None
    launches = int(sum_over_ranks(ops.launch_count() - launches0))
    ms = max_over_ranks(start.elapsed_time(end)) / args.steps
    clocks.__exit__(None, None, None)
    if keep is not None:
        dump_outputs(args.dump_outputs, **keep)
        keep = None
    ef, f_agg = edge_feat_per_step(name, n, slots, fin, fout)
    value = ef / (ms * 1e-3) / 1e9

    spmm_ms = [s.elapsed_time(e) for s, e in spmm_events]
    weighted = name in ('gcnconv', 'gcnidconv', 'gatconv', 'gatidconv')
    f_launch = f_agg // world if (multi and playout.sliced) else f_agg
    per_launch_bytes = spmm_bytes(rows_local, slots_local, f_launch, weighted, 2 if half else 4)
    avg_spmm_ms = float(np.mean(spmm_ms)) if spmm_ms else float('nan')
    peak, peak_src = load_peaks()
    achieved = per_launch_bytes / (avg_spmm_ms * 1e-3) / 1e9
    roofline = {'bound': 'hbm',
                'kernel': ('spmm_h_kernel (bf16 gather)' if half else 'spmm_sell_kernel (degree-sorted sliced-ELL)' if f_launch <= ops.SELL_MAX_F and ops.SPMM_ALGO == 'auto' else 'spmm_mpg_kernel (merge-path)' if f_launch <= 128 else 'spmm_mp_kernel (merge-path)') + ' + fixup (CSR aggregation; fwd on CSR and bwd on CSC)'
                          + ((' — rank 0 of %d, ' % world) + ('all rows x F/%d columns (sub-warp-group kernel, rows stored '
                             'to their owners over NVLink)' % world if playout.sliced else 'rank-local rows') if multi else ''),
                'achieved': round(achieved, 1), 'peak': peak, 'unit': 'GB/s',
                'frac': round(achieved / peak, 4),
                'traffic': NCU_TRAFFIC.get((args.workload, 'sell' if ops.SPMM_ALGO == 'auto' else ops.SPMM_ALGO)) if not (multi or half) else None,
                'peak_source': peak_src,
                'algorithmic_bytes_per_launch': per_launch_bytes,
                'avg_launch_ms': round(avg_spmm_ms, 4), 'launches_timed': len(spmm_ms),
                'frac_dram': None,   # filled below: ncu DRAM traffic / this run's launch time / peak
                'share_of_step': round(sum(spmm_ms) / args.steps / ms, 3)}

    if gat_events['bwd'] and not spmm_ms:
        # fused GAT: the dominant launch group is the one-pass backward (per-node record + walk over the CSC layout +
        # split-row fix-up); the training forward is reported beside it
        fb = [s.elapsed_time(e) for s, e in gat_events['bwd']]
        ff = [s.elapsed_time(e) for s, e in gat_events['fwd']]
        bytes_b = gat_pass_bytes('bwd', rows_local, slots_local, f_agg)
        bytes_f = gat_pass_bytes('fwd', rows_local, slots_local, f_agg)
        ach_b, ach_f = bytes_b / (np.mean(fb) * 1e-3) / 1e9, bytes_f / (np.mean(ff) * 1e-3) / 1e9
        roofline.update({'kernel': 'gat_tstat_d_kernel + gat_sell_bwd_one_kernel + fixup (the whole edge-softmax / '
                                   'aggregation backward in one walk over the CSC sliced-ELL layout)',
                         'achieved': round(ach_b, 1), 'frac': round(ach_b / peak, 4), 'traffic': NCU_TRAFFIC.get((args.workload, 'bwd_one')),
                         'algorithmic_bytes_per_launch': bytes_b, 'avg_launch_ms': round(float(np.mean(fb)), 4),
                         'launches_timed': len(fb), 'share_of_step': round(sum(fb) / args.steps / ms, 3),
                         'also': {'kernel': 'gat_sell_fwd_train_kernel + fixup (online softmax fused into the CSR '
                                            'aggregation, writes out and out_pos)',
                                  'achieved': round(ach_f, 1), 'frac': round(ach_f / peak, 4),
                                  'algorithmic_bytes_per_launch': bytes_f, 'avg_launch_ms': round(float(np.mean(ff)), 4),
                                  'launches_timed': len(ff), 'share_of_step': round(sum(ff) / args.steps / ms, 3),
                                  'traffic': NCU_TRAFFIC.get((args.workload, 'fwd_train'))}})
        if roofline['also']['traffic']:
            roofline['also']['frac_dram'] = round(roofline['also']['traffic'] / (np.mean(ff) * 1e-3) / 1e9 / peak, 4)
        avg_spmm_ms = float(np.mean(fb))
    if roofline['traffic']:
        roofline['frac_dram'] = round(roofline['traffic'] / (avg_spmm_ms * 1e-3) / 1e9 / peak, 4)
    # ---- layout build alone (amortised over layers/epochs in training; reported, not in `value`) ---
    clear_cache()
    sync_all()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    if multi:
        pl2 = mk_layout(ei)
        warm_weights(pl2)
        del pl2
    else:
        lay = get_layout(ei, n, policy)
        _ = lay.csr, lay.csc
        lay.weights('gcn_tgt' if name == 'gcnconv' else 'sum')
    e.record()
    torch.cuda.synchronize()
    layout_ms = max_over_ranks(s.elapsed_time(e))

    # ---- end to end: host buffers in, result out, every step ------------------------------------
    x_host = x_loc.cpu().pin_memory()
    # N > 1: every rank uploads only ITS 1/N of the edge list (columns [rank*epr, (rank+1)*epr)); the pieces are
    # all-gathered over NVLink on the device (the layout needs the whole graph in the sliced exchange)
    e_total = int(ei.size(1))
    epr = (e_total + world - 1) // world
    if multi:
        pad = torch.full((2, epr * world - e_total), -1, dtype=ei.dtype, device=dev)
        ei_piece = torch.cat([ei, pad], 1)[:, rank * epr:(rank + 1) * epr].contiguous()
        ei_host = ei_piece.cpu().pin_memory()
        del pad, ei_piece
    else:
        ei_host = ei.cpu().pin_memory()
    e2e_steps = max(5, min(args.steps, 10))
    res_host = torch.empty(fout, dtype=torch.float32).pin_memory()

    side = torch.cuda.Stream(device=dev)

    def issue_copies():
        # this step's inputs, pinned host -> device, on the copy stream: edge_index first (the layout build needs only
        # the graph), then the node features
        with torch.cuda.stream(side):
            eid = ei_host.to(dev, non_blocking=True)
            e_ready = torch.cuda.Event()
            e_ready.record(side)
            xd = x_host.to(dev, non_blocking=True)
            x_ready = torch.cuda.Event()
            x_ready.record(side)
        return eid, xd, e_ready, x_ready

    def compute(eid, xd, e_ready, x_ready):
        cur = torch.cuda.current_stream()
        cur.wait_event(e_ready)
        eid.record_stream(cur)
        if multi:
            pieces = torch.empty((world, 2, epr), dtype=eid.dtype, device=dev)
            dist.all_gather_into_tensor(pieces, eid)
            eid = pieces.permute(1, 0, 2).reshape(2, world * epr)[:, :e_total].contiguous()
            pl = mk_layout(eid)
            warm_weights(pl)
        else:
            pl = None
            lay = get_layout(eid, n, policy)          # public API: builds + caches CSR, CSC and weights
            _ = lay.csr, lay.csc
        cur.wait_event(x_ready)                        # the layer waits for the features right before its first GEMM
        xd.record_stream(cur)
        r = step(xd, eid, pl)
        res_host.copy_(r.detach().reshape(-1)[:fout], non_blocking=True)

    def e2e_run(k):
        # a loader's prefetch: the copies of step i+1 are in flight while step i computes; every step's copies, layout
        # build, fwd+bwd and result read-back happen inside the timed region
        nxt = issue_copies()
        for i in range(k):
            cur_in = nxt
            if i + 1 < k:
                nxt = issue_copies()
            compute(*cur_in)

    e2e_run(4)   # the prefetch pipeline keeps two steps' buffers alive: let the caching allocator reach its steady state
    sync_all()
    clear_cache()
    stats0 = torch.cuda.memory_stats(dev)
    s.record()
    e2e_run(e2e_steps)
    e.record()
    sync_all()
    stats1 = torch.cuda.memory_stats(dev)
    e2e_ms = max_over_ranks(s.elapsed_time(e)) / e2e_steps
    h2d = int(sum_over_ranks(x_host.numel() * 4 + ei_host.numel() * 8))
    e2e = {'value': round(ef / (e2e_ms * 1e-3) / 1e9, 3), 'unit': 'GEdge-feat/s',
           'ms_per_step': round(e2e_ms, 3), 'steps': e2e_steps,
           'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': int(fout * 4 * world),
           'stats': {k: stats1.get(k, 0) - stats0.get(k, 0) for k in ('num_device_alloc', 'num_device_free', 'num_alloc_retries')}
           if os.environ.get('GG_E2E_STATS') else None,
           'includes': 'every step: H2D of this rank\'s 1/N of edge_index, then of its node_feature rows, from pinned memory '
                       '(copy stream; the copies of step i+1 overlap the compute of step i, as a prefetching loader does), '
                       + ('NCCL all-gather of the edge list pieces over NVLink, ' if multi else '') +
                       'CSR+CSC layout build, layer fwd+bwd (dX, dW, dbias) via the layer API, D2H of the bias gradient'}
    del x_host, ei_host

    parity = None
    if multi:
        # correctness of the driver-run multi-GPU path: this rank's rows of the output and of dX, and the all-reduced
        # parameter gradients, against the single-GPU layer (same parameters: the partitioned module wraps it) on the
        # same inputs; max over ranks
        fwd_m = (lambda t: layer(t, playout, ids)) if ids is not None else (lambda t: layer(t, playout))
        xg = x_loc.detach().requires_grad_(True)
        layer.zero_grad(set_to_none=True)
        y_m = fwd_m(xg)
        y_m.backward(gy_loc)
        y_m = y_m.detach()
        parallel.allreduce_grads(layer)
        gm = {k: v.grad.detach().clone() for k, v in layer.named_parameters() if v.grad is not None}
        dx_m = xg.grad.detach().clone()
        layer.zero_grad(set_to_none=True)
        x1 = x.detach().requires_grad_(True)
        y1 = layer.model(x1, ei, ids) if ids is not None else layer.model(x1, ei)
        y1.backward(gy)
        rel = lambda a, r: float((a.double() - r.double()).abs().max() / r.double().abs().max().clamp(min=1e-30))
        errs = {'out': rel(y_m, y1.detach()[part.lo:part.hi]), 'dx': rel(dx_m, x1.grad[part.lo:part.hi])}
        for k, v in layer.model.named_parameters():
            if v.grad is not None and ('model.' + k) in gm:
                errs['d' + k] = rel(gm['model.' + k], v.grad)
        parity = {k: max_over_ranks(v) for k, v in sorted(errs.items())}
        parity['tolerance'] = 1e-5
        parity['ok'] = all(v <= 1e-5 for k, v in parity.items() if k not in ('tolerance', 'ok'))
        parity['metric'] = 'max|a - b| / max|b| against the single-GPU layer on the same inputs, max over ranks'
        del y_m, dx_m, x1, y1, gm
        layer.zero_grad(set_to_none=True)
    comparators = None
    if not multi and not args.no_comparators and rank == 0:
        comparators = gpu_comparators(name, n, ei, x, gy, fin, fout, lay, policy, ef, dev)
    cpu = None
    if rank == 0 and not args.no_cpu and not multi:
        cpu = cpu_baseline(spec, seconds=args.cpu_seconds, warmup=1, graph=(n, ei.cpu(), x.cpu(), gy.cpu()), extras=True)
    out = {
        'metric': 'layer fwd+bwd GEdge-feat/s', 'value': round(value, 3), 'unit': 'GEdge-feat/s',
        'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': round(ms, 4),
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None,
        'dtype': 'f32' if not half else 'f32 arithmetic, gathered operand stored in bf16 (1e-2 mode)',
        'data': 'synthetic (seeded power-law / BA / uniform generators in bench.py; random-init glorot weights)',
        'config': {'workload': spec['desc'], 'layer': name, 'nodes': n, 'edges_directed': int(ei.size(1)),
                   'slots_after_loop_policy': slots, 'f_in': fin, 'f_out': fout, 'f_aggregated': f_agg,
                   'parallelism': ('row-partitioned x%d, exchange fwd and bwd: %s' % (world, HALO_DESC[halo])) if multi
                   else 'single GPU',
                   'l2_policy': 'inputs larger than L2 (feature matrix %.0f MB vs 126 MB L2)' % (n * f_agg * 4 / 1e6)
                   if n * f_agg * 4 > 126e6 else 'inputs fit L2: launch-bound workload, no flush',
                   'layout_cached_across_steps': True},
        'clocks': clocks.summary(), 'e2e': e2e, 'gpu_launches': int(launches),
        'roofline': roofline, 'cpu_baseline': cpu,
        'host_enqueue_ms_per_step': round(host_ms, 3),
        'parity_vs_1gpu': parity, 'comparators': comparators,
        'exchange_trace_ms': exchange_trace,   # GG_PEER_TRACE=1: mean ms between the exchange's phase marks, rank 0, timed steps
        # the reference re-runs its COO edits + normalisation on every forward (idconv.py:69-87); `value` caches the layout
        'value_with_layout_build_every_step': round(ef / ((ms + layout_ms) * 1e-3) / 1e9, 3),
        'layout_build_ms': round(layout_ms, 3), 'graph_gen_s': round(gen_s, 2),
        'layout_first_call_s': round(layout_first_s, 3),
    }
    if multi:
        if playout.pool is not None:
            playout.pool.close()
        dist.barrier()
        dist.destroy_process_group()
    return out


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle restatement of the reference's op sequence, all host threads
# ------------------------------------------------------------------------------------------------
CPU_CHUNK = 1 << 22   # edges per chunk of the CPU arm (the [E, F] message tensor of the full graph would be 33 GB)


def cpu_params(fin, fout):
    g = torch.Generator().manual_seed(0)
    mk = lambda *s: torch.randn(*s, generator=g) * 0.1
    return {'weight': mk(fin, fout), 'bias': mk(fout), 'w_l': mk(fout, fin), 'w_r': mk(fout, fin),
            'att': mk(1, 1, 2 * fout)}


def cpu_layer_step(name, x, ei, p, gy, chunk=CPU_CHUNK):
    """One forward+backward of the reference's CPU op sequence (ref: layer.py:135-162 -> pyg.nn.*, idconv.py:89-92):
    oracle/chunked.py = oracle/layers.py + autograd, evaluated over edge chunks (SURVEY §8d)."""
    from oracle import chunked
    if name == 'gcnconv':
        return chunked.gcnconv_step(x, ei, p['weight'], p['bias'], gy, chunk)
    if name == 'sageconv':
        return chunked.sageconv_step(x, ei, p['w_l'], p['bias'], p['w_r'], gy, chunk)
    if name == 'gatconv':
        return chunked.gatconv_step(x, ei, p['weight'], p['att'], p['bias'], gy, chunk=chunk)
    raise KeyError(name)


def _time_cpu_steps(fn, seconds, steps, warmup):
    """Median wall time of `steps` calls (or as many as fit `seconds`, at least one) after `warmup` untimed calls."""
    for _ in range(warmup):
        fn()
    times, t_end = [], time.time() + seconds
    while True:
        t0 = time.time()
        fn()
        times.append(time.time() - t0)
        if (steps is not None and len(times) >= steps) or (steps is None and (time.time() >= t_end or len(times) >= 50)):
            break
    return float(np.median(times)), len(times)


def cpu_baseline(spec, seconds=15.0, steps=None, warmup=1, graph=None, extras=False, scale=1.0):
    """Oracle (kind 'port': PyG is not installable here) on the FULL graph of the workload (`scale` = 1; the per-edge
    tensors are chunked), all host threads.  `graph` = (n, edge_index, x, gy) CPU tensors to reuse (the bits the GPU arm
    ran on); otherwise the same generator runs on the CPU.  `extras`: also the reference's default thread count
    (cfg.num_threads = 6, ref: config.py:57) and a torch.sparse CSR (MKL) formulation of the same layer."""
    name, fin, fout = spec['layer'], spec['fin'], spec['fout']
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cpu = torch.device('cpu')
    if graph is None:
        n, ei = gen_graph(spec, cpu, seed=0, scale=scale)
        x = gen_features(n, fin, cpu)
        gy = gen_features(n, fout, cpu, seed=7)
    else:
        n, ei, x, gy = graph
    params = cpu_params(fin, fout)
    slots = int(ei.size(1)) + (n if name in ('gcnconv', 'gatconv') else 0)   # upper bound; exact E' needs the loop count
    if name in ('gcnconv', 'gatconv'):
        slots -= int((ei[0] == ei[1]).sum())
    ef, _ = edge_feat_per_step(name, n, slots, fin, fout)
    with torch.no_grad():
        t, done = _time_cpu_steps(lambda: cpu_layer_step(name, x, ei, params, gy), seconds, steps, warmup)
        out = {'value': round(ef / t / 1e9, 4), 'unit': 'GEdge-feat/s', 'cores': cores, 'kind': 'port',
               'ms_per_step': round(t * 1e3, 2), 'steps': done, 'torch_threads': torch.get_num_threads(),
               'sample': f'the whole workload graph ({n} nodes, {int(ei.size(1))} directed edges, {name} {fin}->{fout}, '
                         f'fwd+bwd, fp32), {done} step(s) after {warmup} warm-up: oracle restatement of the PyG op sequence '
                         f'(index_select gather, per-edge scale, index_add_ scatter, matmul) over edge chunks of {CPU_CHUNK}'
                         + ('' if scale == 1.0 else f' — generator scaled x{scale:.4f}')}
        if extras:
            torch.set_num_threads(min(6, cores))
            t6, d6 = _time_cpu_steps(lambda: cpu_layer_step(name, x, ei, params, gy), 0.0, 1, 0)
            out['six_threads'] = {'value': round(ef / t6 / 1e9, 4), 'ms_per_step': round(t6 * 1e3, 2), 'steps': d6,
                                  'torch_threads': torch.get_num_threads(),
                                  'note': 'the reference default cfg.num_threads = 6 (config.py:57, main_zd.py:284)'}
            torch.set_num_threads(cores)
            if name == 'gcnconv':
                out['torch_sparse_csr'] = cpu_sparse_gcn(n, ei, x, gy, params, ef)
    return out


def cpu_sparse_gcn(n, ei, x, gy, p, ef):
    """Secondary CPU line (SURVEY §8d): the same GCN layer as A_hat @ (X W) with torch.sparse CSR (MKL), fwd + bwd."""
    from oracle import layers as olayers
    t0 = time.time()
    ei2, norm = olayers.gcn_norm_tgt(ei, n, x.dtype)
    a = torch.sparse_coo_tensor(torch.stack([ei2[1], ei2[0]]), norm, (n, n)).coalesce()
    a_csr, at_csr = a.to_sparse_csr(), a.t().coalesce().to_sparse_csr()
    build = time.time() - t0

    def step():
        h = x @ p['weight']
        out = a_csr @ h + p['bias']
        gh = at_csr @ gy
        return out, gh @ p['weight'].t(), x.t() @ gh, gy.sum(0)
    step()
    t, done = _time_cpu_steps(step, 0.0, 2, 0)
    return {'value': round(ef / t / 1e9, 4), 'ms_per_step': round(t * 1e3, 2), 'steps': done,
            'csr_build_s': round(build, 2), 'note': 'torch.sparse CSR @ dense (MKL), adjacency built once outside the step'}


def run_reference(args, spec, rank, world):
    if rank != 0:
        return None
    t0 = time.time()
    # the whole workload graph; K timed steps after one warm-up (a step is ~10 s of CPU at 62 M edges)
    cpu = cpu_baseline(spec, steps=args.steps, warmup=1 if args.warmup > 0 else 0, scale=args.cpu_scale)
    return {'impl': 'reference', 'metric': 'layer fwd+bwd GEdge-feat/s', 'value': cpu['value'],
            'unit': 'GEdge-feat/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': cpu['ms_per_step'], 'higher_is_better': True, 'scaling': 'strong',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic (seeded generators in bench.py, run on the CPU)',
            'config': {'workload': spec['desc'], 'layer': spec['layer'], 'same_graph_family_and_size_as_the_gpu_arm': args.cpu_scale == 1.0,
                       'warmup_steps_run': 1 if args.warmup > 0 else 0},
            'cpu_baseline': cpu, 'wall_s': round(time.time() - t0, 1),
            'e2e': {'value': cpu['value'], 'unit': 'GEdge-feat/s', 'h2d_bytes_per_step': 0,
                    'd2h_bytes_per_step': 0},
            'note': 'torch_geometric / torch_scatter are not installable offline: this is the oracle '
                    'restatement of the reference CPU path (oracle/chunked.py == oracle/layers.py + autograd), all host threads'}


def main():
    # stdout carries exactly one JSON line: libraries that print there (NCCL's version banner at NCCL_DEBUG=VERSION
    # and above) are sent to stderr for the whole run, the line goes to the saved descriptor
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(obj) + '\n').encode())

    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument('--cpu-seconds', type=float, default=15.0)
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--cpu-scale', type=float, default=1.0,
                    help='--impl reference: shrink the generator (nodes and edges together); 1.0 = the whole workload graph')
    ap.add_argument('--no-comparators', action='store_true', help='skip the GPU library comparators (N=1)')
    ap.add_argument('--gather-dtype', default='f32', choices=['f32', 'bf16'],
                    help="storage of the aggregation's gathered operand: f32 (reference arithmetic, the default and "
                         "the headline) or bf16 (the north star's 1e-2 mode; single GPU)")
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last one computed (layer output, input gradient, '
                         'parameter gradients; a seeded sample of the rows of per-node arrays, %d bytes at most) as '
                         'DIR/<name>.npy, to compare two builds output for output (single GPU)' % DUMP_BYTES)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    spec = WORKLOADS[args.workload]
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    if args.dump_outputs and (world > 1 or args.impl == 'reference'):
        ap.error('--dump-outputs dumps the single-GPU timed path (--impl ours, one process)')
    if args.impl == 'reference':
        if spec.get('aux'):
            raise SystemExit('--impl reference covers the layer workloads')
        out = run_reference(args, spec, rank, world)
        if out is not None:
            emit(out)
        return
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device: the product path has no CPU fallback '
                         '(use --impl reference for the CPU arm)')
    local = int(os.environ.get('LOCAL_RANK', 0))
    dev = torch.device('cuda', local)
    torch.cuda.set_device(dev)
    if spec.get('aux'):
        out = run_aux(args, spec, dev, rank, world)
    else:
        out = run_ours(args, spec, rank, world, dev)
    if rank == 0:
        emit(out)


if __name__ == '__main__':
    main()
