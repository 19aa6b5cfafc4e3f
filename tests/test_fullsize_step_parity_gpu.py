"""One single-GPU bench step against float64 at the size bench.py times it, element by element.

Every single-GPU layer workload of ``bench.py`` draws its inputs here exactly as ``bench.run_ours`` does
(``gen_graph(spec, dev, seed=0)``, ``gen_features(n, fin)``, ``gen_features(n, fout, seed=7)``, ``torch.manual_seed(0)``
before ``layer_dict[name](fin, fout, bias=True)``) and runs one forward + backward through ``forward(Batch)``.  ``out``,
``grad_x`` and every parameter gradient are compared with ``oracle/chunked.py`` evaluated in float64 on the device, once
with the layer's initial bias and once with the bias drawn from U(-0.3, 0.3) so that the bias term is not zero.

Bounds, all of which apply:
  norm-wise     max|got - ref| / max|ref| < 1e-5 on every array (``tests/util.py::rel_err``).
  element-wise  GCN and SAGE are multilinear in (x, W, b, gy): the same chunked step on (|x|, |W|, |b|, |gy|) gives
                ``mag``, an upper bound on the sum of the absolute values of the terms behind each element, and
                |got - ref| <= 1e-5 mag must hold for every element of every array, so that isolated and low-degree rows
                are held to their own scale rather than to the hubs'.  GAT ``out``: |got - ref| <= 1e-5 (sum_e alpha_e
                (|x_src| |W|) + |b|) with the float64 alpha (|x| |W| rather than |h|: see ``gat_out_magnitude``).
  fp32 floor    the same chunked oracle run in float32 on the device is measured against float64; where that run itself
                misses 1e-5 the quantity is ill-conditioned, and the kernel must be within twice the float32 oracle's
                error instead.  A kernel worse than that is a bug, not a tolerance problem.

The kernels that ran are read from a profile of the checked step: they must be the ones ``bench.py`` times.

Where the floor applies (measured on one B200, power limit 1000 W): products_gat's grad_x, dW and datt.  The float32
oracle itself misses 1e-5 there (grad_x 1.79e-4, dW 1.76e-5, datt 2.88e-5 norm-wise; the kernels: 1.79e-4, 1.41e-5,
3.36e-5).  The cause is not cancellation but the leaky ReLU's gate: 5 of the 64.3 M logits lie within float32 rounding
of zero (|z| down to 9.4e-9) and take the other slope in float32 than in float64, which changes those edges' dz by a
factor of 5; the worst row of grad_x is an endpoint of one of them.  Everywhere else every array is within 1e-5 (1e-2 in
the bf16-gather mode) both norm-wise and element-wise; DESIGN.md section 5 lists the numbers.
"""
import math
import re
from collections import Counter

import pytest
import torch

import bench
from oracle import chunked
from oracle import identity as oid
from oracle import pyg_utils as U
from util import FP32_TOL, powerlaw_graph, rel_err

gpu = pytest.mark.gpu


def norm_err(got, ref):
    """``rel_err`` evaluated where the arrays live (no host copy of a 2.5 GB array)."""
    d = (got.double() - ref.double()).abs()
    return float(d.max() / ref.double().abs().max().clamp(min=1e-30)) if d.numel() else 0.0


def elementwise_err(got, ref, mag, where=False):
    """max over the elements of |got - ref| / mag; an element with mag = 0 has only zero terms and must be exact.
    ``where``: also the index of that element."""
    d = (got.double() - ref.double()).abs()
    if not d.numel():
        return (0.0, None) if where else 0.0
    r = d / mag.double().clamp(min=1e-300)
    i = int(r.argmax())
    return (float(r.view(-1)[i]), tuple(int(v) for v in torch.unravel_index(torch.tensor(i), r.shape))) if where else \
        float(r.view(-1)[i])


def check_arrays(tag, got, ref, mag=None, ref32=None, tol=FP32_TOL):
    """Every bound on every array of ``ref``; reports all measurements, fails on any.  -> {array: measurements}."""
    mag, ref32 = mag or {}, ref32 or {}
    report, failures = {}, []
    for k, r in ref.items():
        g = got[k].reshape(r.shape)
        ne = norm_err(g, r)
        ee, at = elementwise_err(g, r, mag[k], where=True) if k in mag else (None, None)
        n32 = norm_err(ref32[k], r) if k in ref32 else None
        e32 = elementwise_err(ref32[k], r, mag[k]) if (k in ref32 and k in mag) else None
        bn = tol if n32 is None or n32 < tol else 2 * n32
        be = tol if e32 is None or e32 < tol else 2 * e32
        report[k] = dict(norm=ne, elem=ee, norm32=n32, elem32=e32)
        line = (f'{tag} {k}: norm-wise {ne:.2e} (bound {bn:.2e}), element-wise '
                + ('-' if ee is None else f'{ee:.2e} (bound {be:.2e}, worst at {at})')
                + f'; fp32 oracle {"-" if n32 is None else f"{n32:.2e}"} / {"-" if e32 is None else f"{e32:.2e}"}')
        print(line)
        if not ne < bn or (ee is not None and not ee <= be):
            failures.append(line)
    assert not failures, '\n'.join(failures)
    return report


def kernels_of(fn):
    """Run ``fn`` under the CUDA profiler -> (its result, Counter of kernel name -> launches)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    return res, Counter({e.key: e.count for e in prof.key_averages()})


def launches(kern, name):
    pat = re.compile(r'\b%s\b' % re.escape(name))
    return sum(c for k, c in kern.items() if pat.search(k))


def check_path(tag, kern, want, never=()):
    """``want``: kernel -> least launches; ``never``: kernels that must not have run."""
    seen = {k: launches(kern, k) for k in list(want) + list(never)}
    bad = [k for k, c in want.items() if seen[k] < c] + [k for k in never if seen[k]]
    assert not bad, f'{tag}: kernels {bad} ran other than expected; launches {seen}'


# ------------------------------------------------------------------------------------------------
# the bench step
# ------------------------------------------------------------------------------------------------
CASES = {   # case -> (bench workload, gather dtype, tolerance)
    'products_gcn': ('products_gcn', 'f32', FP32_TOL),
    'products_gcn_bf16': ('products_gcn', 'bf16', 1e-2),
    'products_gat': ('products_gat', 'f32', FP32_TOL),
    'ba1m_gcn': ('ba1m_gcn', 'f32', FP32_TOL),
    'ba1m_sage': ('ba1m_sage', 'f32', FP32_TOL),
    'cora_gcn': ('cora_gcn', 'f32', FP32_TOL),
}
SIMT = ('id_gemm_kernel', 'gemm_tn_kernel')           # CUDA-core GEMMs: never on the tensor-core build's path
NARROW = ('tc_gemm_kernel', 'tc_gemm_tn_kernel', 'spmm_mp_kernel', 'spmm_mpg_kernel') + SIMT
PATHS = {   # case -> (kernel -> least launches in one step, kernels that must not run, python entry point -> calls)
    'products_gcn': ({'spmm_sell_kernel': 2, 'tc_gemm_persist_kernel': 2, 'tc_gemm_tn_persist_kernel': 1}, NARROW,
                     {'spmm': 2}),
    'products_gcn_bf16': ({'spmm_h_kernel': 2, 'tc_gemm_persist_kernel': 2, 'tc_gemm_tn_persist_kernel': 1},
                          NARROW + ('spmm_sell_kernel',), {'spmm': 2}),
    'products_gat': ({'gat_sell_fwd_train_kernel': 1, 'gat_tstat_d_kernel': 1, 'gat_sell_bwd_one_kernel': 1,
                      'gat_att_partial_kernel': 1, 'tc_gemm_persist_kernel': 2, 'tc_gemm_tn_persist_kernel': 1},
                     NARROW + ('gat_sell_bwd_edge_kernel', 'gat_fwd_kernel', 'gat_bwd_edge_kernel'),
                     {'spmm': 0, 'gat_sell_forward': 1, 'gat_sell_backward_one': 1}),
    'ba1m_gcn': ({'spmm_mp_kernel': 2, 'tc_gemm_kernel': 2, 'tc_gemm_tn_kernel': 1},
                 ('spmm_sell_kernel', 'spmm_mpg_kernel', 'tc_gemm_persist_kernel', 'tc_gemm_tn_persist_kernel') + SIMT,
                 {'spmm': 2}),
    'ba1m_sage': ({'spmm_mp_kernel': 2, 'tc_gemm_kernel': 3, 'tc_gemm_tn_kernel': 2},
                  ('spmm_sell_kernel', 'spmm_mpg_kernel', 'tc_gemm_persist_kernel', 'tc_gemm_tn_persist_kernel') + SIMT,
                  {'spmm': 2}),
    # K = 1433: X W runs as ceil(1433 / 256) = 6 launches accumulating into out, dX as one more
    'cora_gcn': ({'tc_gemm_kernel': 7, 'tc_gemm_tn_kernel': 1}, ('tc_gemm_persist_kernel',) + SIMT, {'spmm': 2}),
}
BIAS = {'gcnconv': 'model.bias', 'gatconv': 'model.bias', 'sageconv': 'model.lin_l.bias'}
_INPUTS = {}


def bench_inputs(spec, dev):
    """bench.run_ours's graph, features and output gradient (kept for the next case on the same graph)."""
    key = (spec['graph'], spec['n'], spec['fin'], spec['fout'])
    if key not in _INPUTS:
        _INPUTS.clear()
        torch.cuda.empty_cache()
        n, ei = bench.gen_graph(spec, dev, seed=0)
        _INPUTS[key] = (n, ei, bench.gen_features(n, spec['fin'], dev), bench.gen_features(n, spec['fout'], dev, seed=7))
    return _INPUTS[key]


def oracle_step(layer, p, x, ei, gy, dtype, absolute=False):
    """The chunked oracle of ``layer`` in ``dtype`` -> {array name: value} named like the layer's parameters (+ alpha
    [E'] for GAT).  ``absolute``: on |x|, |W|, |b|, |gy| (the term magnitudes of a multilinear layer)."""
    c = (lambda t: t.detach().to(dtype).abs()) if absolute else (lambda t: t.detach().to(dtype))
    if layer == 'gcnconv':
        out, dx, dw, db = chunked.gcnconv_step(c(x), ei, c(p['model.weight']), c(p['model.bias']), c(gy))
        return {'out': out, 'grad_x': dx, 'model.weight': dw, 'model.bias': db}
    if layer == 'sageconv':
        out, dx, dwl, dbl, dwr = chunked.sageconv_step(c(x), ei, c(p['model.lin_l.weight']), c(p['model.lin_l.bias']),
                                                       c(p['model.lin_r.weight']), c(gy))
        return {'out': out, 'grad_x': dx, 'model.lin_l.weight': dwl, 'model.lin_l.bias': dbl, 'model.lin_r.weight': dwr}
    out, dx, dw, datt, db, alpha = chunked.gatconv_step(c(x), ei, c(p['model.weight']), c(p['model.att']),
                                                        c(p['model.bias']), c(gy), return_alpha=True)
    return {'out': out, 'grad_x': dx, 'model.weight': dw, 'model.att': datt, 'model.bias': db, 'alpha': alpha}


def gat_out_magnitude(x, ei, weight, bias, alpha, chunk=1 << 22):
    """sum_e alpha_e (|x_src| |W|) + |b| per element of GAT's out (float64, alpha over the layer's edge list).  The terms
    behind out[i, c] are alpha_e x[src, k] W[k, c]: h = x W is itself a sum, and where it cancels (|h| << |x| |W|) its own
    float32 rounding is larger than |h|, so sum_e alpha_e |h_src| would not bound the rounding of a correct kernel."""
    e2, _ = U.remove_self_loops(ei)
    e2, _ = U.add_self_loops(e2, num_nodes=x.size(0))
    h = x.double().abs() @ weight.double().abs()
    return chunked._scatter_messages(torch.zeros_like(h), h, e2[0], e2[1], alpha, chunk) + bias.double().abs()


@gpu
@pytest.mark.parametrize('bias_draw', ['init', 'uniform'])
@pytest.mark.parametrize('case', list(CASES))
def test_bench_step_equals_fp64_at_full_size(cuda, case, bias_draw):
    """The documented numbers are in DESIGN.md section 5; the fp32 floor is taken only where the float32 oracle itself
    misses 1e-5 (GAT's datt, a sum of about 64 M cancelling terms, is the expected case)."""
    from graphgym_b200 import ops
    from graphgym_b200.config import cfg
    from graphgym_b200.models.layer import Batch, layer_dict
    workload, gather, tol = CASES[case]
    spec = bench.WORKLOADS[workload]
    name = spec['layer']
    n, ei, x, gy = bench_inputs(spec, cuda)
    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(cfg.b200, 'gather_dtype', gather)
        torch.manual_seed(0)
        layer = layer_dict[name](spec['fin'], spec['fout'], bias=True).to(cuda)
        if bias_draw == 'uniform':
            with torch.no_grad():
                dict(layer.named_parameters())[BIAS[name]].uniform_(
                    -0.3, 0.3, generator=torch.Generator(device=cuda).manual_seed(11))

        def step():
            layer.zero_grad(set_to_none=True)
            xg = x.detach().requires_grad_(True)
            y = layer(Batch(xg, ei)).node_feature
            y.backward(gy)
            return y.detach(), xg.grad
        step()                                       # bench's warm-up: the layout is built here
        calls = Counter()

        def counted(fn, key):
            def run(*a, **k):
                calls[key] += 1
                return fn(*a, **k)
            return run
        for key in ('spmm', 'gat_sell_forward', 'gat_sell_backward_one'):
            mp.setattr(ops, key, counted(getattr(ops, key), key))
        (out, gx), kern = kernels_of(step)
    want, never, entry = PATHS[case]
    check_path(case, kern, want, never)
    assert {k: calls[k] for k in entry} == entry, (case, dict(calls))
    got = {'out': out, 'grad_x': gx, **{k: p.grad for k, p in layer.named_parameters()}}
    p = {k: v.detach() for k, v in layer.named_parameters()}
    del layer, out, gx

    ref = oracle_step(name, p, x, ei, gy, torch.float64)
    alpha = ref.pop('alpha', None)
    if name == 'gatconv':
        mag = {'out': gat_out_magnitude(x, ei, p['model.weight'], p['model.bias'], alpha)}
        del alpha
    else:
        mag = oracle_step(name, p, x, ei, gy, torch.float64, absolute=True)
    ref32 = None
    if gather == 'f32':
        ref32 = oracle_step(name, p, x, ei, gy, torch.float32)
        ref32.pop('alpha', None)
    check_arrays(f'{case}[{bias_draw}]', got, ref, mag, ref32, tol)
    del got, ref, mag, ref32
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------
# cycle features: bench's ba1m_cycles call, each entry against its own value
# ------------------------------------------------------------------------------------------------
def check_per_entry(tag, got, want, tol=FP32_TOL):
    """|got - want| / want per entry (every entry is a sum of non-negative terms: no cancellation), max per column."""
    rel = ((got.double() - want).abs() / want).amax(0)
    print(f'{tag}: per-entry relative error by power p = 1..{rel.numel()}: ' + ' '.join(f'{v:.2e}' for v in rel.tolist()))
    assert bool((want > 0).all()), tag
    assert float(rel.max()) <= tol, (tag, rel.tolist())


@gpu
@pytest.mark.parametrize('step', ['sell', 'mp'])
def test_cycle_feature_blocks_equal_fp64_per_entry(cuda, step):
    """gg_cycle_diag_{sell,mp}_f32 called as bench.run_aux calls it, on block 0, the block holding the highest-degree
    node (block 0 itself on this BA graph) and the last 128 nodes (where bench's wrap-around (blk * 128) % (n - 128)
    ends)."""
    from graphgym_b200 import ops
    spec = bench.WORKLOADS['ba1m_cycles']
    _INPUTS.clear()
    torch.cuda.empty_cache()
    n, ei = bench.gen_graph(spec, cuda, seed=0)
    k = spec['k']
    csr = ops.layout_build(ei, n, ops.LOOPS_ADD_REMAINING, ops.BY_TARGET)
    csc = ops.layout_build(ei, n, ops.LOOPS_ADD_REMAINING, ops.BY_SOURCE)
    w = ops.gcn_norm(csr, ops.segment_degree(csc))
    L = ops.lib()
    hub = int(torch.bincount(ei[0], minlength=n).argmax())
    blocks = sorted({0, min(hub // 128 * 128, n - 128), n - 128})
    if step == 'sell':
        sl = ops.sell_layout(csr)
        w_sell = sl.weights(w)
        ws = torch.empty(int(L.gg_cycle_diag_sell_workspace_bytes(n, sl.partial_rows)), dtype=torch.uint8, device=cuda)
    else:
        item_row, item_slot, items = csr.plan
        ws = torch.empty(int(L.gg_cycle_diag_mp_workspace_bytes(n, items)), dtype=torch.uint8, device=cuda)
    out = torch.empty((128, k), dtype=torch.float32, device=cuda)
    for sb in blocks:
        if step == 'sell':
            ops.check(L.gg_cycle_diag_sell_f32(ops._ptr(csr.rowptr), ops._ptr(sl.chunk_ptr), sl.chunks, ops._ptr(sl.idx),
                                               ops._ptr(w_sell), ops._ptr(sl.vdst), ops._ptr(sl.hub_rows),
                                               ops._ptr(sl.hub_pptr), sl.hubs, sl.partial_rows, n, k, 1, sb, 128,
                                               ops._ptr(out), k, ops._ptr(ws), ws.numel(), ops._stream()),
                      'gg_cycle_diag_sell_f32')
        else:
            ops.check(L.gg_cycle_diag_mp_f32(ops._ptr(csr.rowptr), ops._ptr(csr.nbr), ops._ptr(w), ops._ptr(item_row),
                                             ops._ptr(item_slot), items, n, k, 1, sb, 128, ops._ptr(out), k,
                                             ops._ptr(ws), ws.numel(), ops._stream()), 'gg_cycle_diag_mp_f32')
        want = oid.diag_powers_sparse(ei, n, k, torch.arange(sb, sb + 128, device=cuda))
        check_per_entry(f'ba1m_cycles {step} block at {sb}' + (' (hub)' if sb <= hub < sb + 128 else ''), out, want)


# ------------------------------------------------------------------------------------------------
# peaky softmax: logits up to ~100 (an unshifted exp overflows), every GAT path
# ------------------------------------------------------------------------------------------------
GAT_PATHS = {   # name -> (GAT_ALGO, GAT_BWD, SELL_SEG, kernels that must run)
    'sell_one': ('sell', 'one', 256, ('gat_sell_fwd_train_kernel', 'gat_sell_bwd_one_kernel')),
    'sell_two': ('sell', 'two', 256, ('gat_sell_fwd_eval_kernel', 'gat_sell_bwd_edge_kernel', 'gat_sell_bwd_src_kernel')),
    'sell_seg8': ('sell', 'one', 8, ('gat_sell_fwd_train_kernel', 'gat_sell_bwd_one_kernel')),
    'mp': ('mp', 'one', 256, ('gat_sddmm_mp_kernel',)),
    'row': ('row', 'one', 256, ('gat_fwd_kernel', 'gat_bwd_edge_kernel', 'gat_bwd_src_kernel')),
}


@pytest.fixture(scope='module')
def peaky(cuda):
    """A 50 k-node power-law graph (hub rows far longer than one 256-slot virtual row) plus 100 isolated nodes; h small
    integers, att integers times a power of two: every logit is exact in fp32 and the largest pass log(FLT_MAX)."""
    n0, iso, f = 50_000, 100, 128
    N = n0 + iso
    perm = torch.randperm(N, generator=torch.Generator().manual_seed(3))
    ei = perm[powerlaw_graph(21, n0, 10, max_deg=3000)]          # nodes perm[n0:] have no edge
    g = torch.Generator().manual_seed(4)
    h = torch.randint(-4, 5, (N, f), generator=g).float()
    att_i = torch.randint(-3, 4, (1, 1, 2 * f), generator=g).float()
    e2, _ = U.remove_self_loops(ei)
    e2, _ = U.add_self_loops(e2, num_nodes=N)
    z_int = (h @ att_i[0, 0, :f])[e2[1]] + (h @ att_i[0, 0, f:])[e2[0]]
    scale = 2.0 ** math.ceil(math.log2(90.0 / float(z_int.max())))
    att = att_i * scale
    z = z_int * scale
    assert float(z.max()) > math.log(torch.finfo(torch.float32).max), float(z.max())
    bias = torch.empty(f).uniform_(-0.3, 0.3, generator=g)
    gy = torch.randn(N, f, generator=g)
    return dict(N=N, ei=ei.to(cuda), iso=perm[n0:].to(cuda), h=h.to(cuda), att=att.to(cuda), bias=bias.to(cuda),
                gy=gy.to(cuda), z=z)


@gpu
@pytest.mark.parametrize('path', list(GAT_PATHS))
def test_gat_paths_on_peaky_logits_equal_fp64(cuda, peaky, path):
    from graphgym_b200 import ops
    from graphgym_b200.graph import GraphLayout
    algo, bwd, seg, kernels = GAT_PATHS[path]
    N, ei, h, att, bias, gy = (peaky[k] for k in ('N', 'ei', 'h', 'att', 'bias', 'gy'))
    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(ops, 'GAT_ALGO', algo)
        mp.setattr(ops, 'GAT_BWD', bwd)
        mp.setattr(ops, 'SELL_SEG', seg)
        lay = GraphLayout(ei, N, ops.LOOPS_REMOVE_ADD)
        csr = lay.csr
        if path == 'sell_one':      # the input claim, on the layer's own layout
            rp, nbr = csr.rowptr.long().cpu(), csr.nbr.long().cpu()
            a_t = (h @ att[0, 0, :h.size(1)]).cpu()
            a_s = (h @ att[0, 0, h.size(1):]).cpu()
            deg = rp[1:] - rp[:-1]
            late = 0
            for i in torch.nonzero(deg > seg).flatten().tolist():
                z = a_t[i] + a_s[nbr[rp[i]:rp[i + 1]]]
                late += int(int(torch.argmax(z)) // seg > 0)
            assert late >= 8, late

        def run():
            out, alpha, a_tgt, a_src, pos = ops.gat_forward(csr, h, att, 1, 0.2, bias, need_grad=True)
            dh, datt = ops.gat_backward(csr, lay.csc, lay.csc2csr, h, att, 1, 0.2, bias, alpha, a_tgt, a_src, out, gy,
                                        pos)
            return out, dh, datt
        (out, dh, datt), kern = kernels_of(run)
        if algo == 'sell':
            assert ops.sell_layout(csr).seg == seg and ops.sell_layout(csr).hubs > 0
    check_path(path, kern, {k: 1 for k in kernels})
    # an isolated node aggregates its self loop alone: alpha = 1 exactly
    iso = peaky['iso']
    assert torch.equal(out[iso], h[iso] + bias), path
    eye = torch.eye(h.size(1), device=cuda)
    ref = chunked.gatconv_step(h.double(), ei, eye.double(), att.double(), bias.double(), gy.double(), return_alpha=True)
    r32 = chunked.gatconv_step(h, ei, eye, att, bias, gy)
    mag = {'out': gat_out_magnitude(h, ei, eye, bias, ref[5])}
    check_arrays(f'peaky {path}', {'out': out, 'dh': dh, 'datt': datt},
                 {'out': ref[0], 'dh': ref[1], 'datt': ref[3]}, mag, {'out': r32[0], 'dh': r32[1], 'datt': r32[3]})


# ------------------------------------------------------------------------------------------------
# compute_identity at the size of tests/test_identity_gpu.py, per power
# ------------------------------------------------------------------------------------------------
@gpu
def test_compute_identity_per_column_per_entry(cuda):
    from graphgym_b200.contrib.transform.identity import compute_identity
    n, k = 20000, 10
    ei = powerlaw_graph(11, n, 8).to(cuda)
    got = compute_identity(ei, n, k)
    want = torch.cat([oid.diag_powers_sparse(ei, n, k, torch.arange(s, min(n, s + 2048), device=cuda))
                      for s in range(0, n, 2048)])
    check_per_entry('compute_identity n=20000', got, want)


# ------------------------------------------------------------------------------------------------
# CPU: the element-wise bound sees what the norm-wise bound does not
# ------------------------------------------------------------------------------------------------
def test_elementwise_bound_rejects_what_rel_err_accepts():
    """On a power-law graph with sum aggregation the hub rows set max|ref|: an error of 1e-4 relative confined to the
    degree-1 rows passes rel_err < 1e-5 and fails the element-wise bound."""
    spec = bench.WORKLOADS['products_gcn']
    cpu = torch.device('cpu')
    n, ei = bench.gen_graph(spec, cpu, scale=1e-3)
    x = torch.rand(n, 16, generator=torch.Generator().manual_seed(0), dtype=torch.float64)
    src, tgt = ei
    ref = chunked._scatter_messages(torch.zeros_like(x), x, src, tgt, None, 1 << 12)
    mag = chunked._scatter_messages(torch.zeros_like(x), x.abs(), src, tgt, None, 1 << 12)
    deg1 = torch.bincount(tgt, minlength=n) == 1
    assert int(deg1.sum()) > 0
    got = ref.clone()
    got[deg1] *= 1 + 1e-4
    assert rel_err(got, ref) < FP32_TOL
    assert elementwise_err(got, ref, mag) > FP32_TOL
    assert elementwise_err(ref, ref, mag) == 0.0
