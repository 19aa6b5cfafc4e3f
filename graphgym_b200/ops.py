"""Tensor-level wrappers over the C-ABI (include/gg_b200.h).

torch is used for device memory and streams only: every function checks its tensors, pulls raw
device pointers and calls one ``gg_*`` entry point on the current CUDA stream.  CPU tensors are
rejected — there is no CPU path in this package.
"""
import ctypes

import torch

from . import _lib
from ._lib import GemmSegment, check, lib

LOOPS_KEEP, LOOPS_ADD_REMAINING, LOOPS_REMOVE_ADD, LOOPS_REMOVE, LOOPS_ADD = range(5)
BY_TARGET, BY_SOURCE = 0, 1
SUM, MEAN = 0, 1
ACT_NONE, ACT_RELU, ACT_LRELU = 0, 1, 2


import os as _os
SPMM_ALGO = _os.environ.get("GG_SPMM_ALGO", "auto")    # auto | mp | mpg (grouped slots, f <= 128) | sell (sliced ELL, f <= 128) | row
SPMM_STAGE = _os.environ.get("GG_SPMM_STAGE", "tma")   # tma | ldg
SPMM_DEEP = _os.environ.get("GG_SPMM_DEEP", "0") == "1"  # 16 instead of 8 gathers per lane and batch
SPMM_L2HINT = _os.environ.get("GG_SPMM_L2HINT", "1") == "1"  # gathers evict_last, streams evict_first in L2


def _spmm_flags():
    return (1 if SPMM_STAGE == "ldg" else 0) | (2 if SPMM_DEEP else 0) | (4 if SPMM_L2HINT else 0)
GEMM_MODE = _os.environ.get("GG_GEMM", "tc")           # tc (tcgen05 3xTF32) | simt (fp32 CUDA cores)


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _need_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("graphgym_b200 ops run on CUDA tensors only (no CPU fallback); "
                               f"got a tensor on {t.device}")


def _rows(t, name):
    """(tensor, leading dimension) of a 2-D fp32 matrix with unit inner stride."""
    if t.dtype != torch.float32 or t.dim() != 2:
        raise ValueError(f"{name}: expected a 2-D float32 tensor, got {tuple(t.shape)} {t.dtype}")
    if t.size(1) > 1 and t.stride(1) != 1:
        t = t.contiguous()
    if t.size(0) > 1 and t.stride(0) < t.size(1):
        t = t.contiguous()
    ld = t.stride(0) if t.size(0) > 1 else max(t.size(1), 1)
    return t, ld


def launch_count():
    return int(lib().gg_launch_count())


# --------------------------------------------------------------------------------------------
# layout
# --------------------------------------------------------------------------------------------
class Csr:
    """One compressed layout of an (edited) edge list: segments grouped by target or by source."""
    __slots__ = ("rowptr", "nbr", "perm", "rowid", "num_slots", "num_nodes", "num_edges", "policy",
                 "group_by", "_plan", "_sell")

    def __init__(self, rowptr, nbr, perm, rowid, num_slots, num_nodes, num_edges, policy, group_by):
        self.rowptr, self.nbr, self.perm, self.rowid = rowptr, nbr, perm, rowid
        self.num_slots, self.num_nodes, self.num_edges = num_slots, num_nodes, num_edges
        self.policy, self.group_by = policy, group_by
        self._plan = None
        self._sell = None

    def _build_plan(self, units):
        if self._plan is None:
            self._plan = {}
        if units not in self._plan:
            L = lib()
            items = int(L.gg_spmm_plan_items(self.num_nodes, self.num_slots, units))
            item_row = torch.empty(items + 1, dtype=torch.int32, device=self.rowptr.device)
            item_slot = torch.empty(items + 1, dtype=torch.int32, device=self.rowptr.device)
            check(L.gg_spmm_plan_build(_ptr(self.rowptr), self.num_nodes, self.num_slots, units,
                                       _ptr(item_row), _ptr(item_slot), _stream()), "gg_spmm_plan_build")
            self._plan[units] = (item_row, item_slot, items)
        return self._plan[units]

    @property
    def plan(self):
        """Merge-path work plan of the load-balanced SpMM: (item_row, item_slot, items), built once."""
        return self._build_plan(int(lib().gg_spmm_plan_units(self.num_nodes, self.num_slots)))


def layout_build(edge_index, num_nodes, policy=LOOPS_KEEP, group_by=BY_TARGET, row_range=None, nbr_range=None):
    """COO ``edge_index[2,E]`` (int64, row 0 = source, row 1 = target) -> Csr.  One host sync to
    read E' (self-loop removal makes it data dependent).

    ``row_range=(lo, hi)``: rank-local layout of a row partition — only groups in [lo, hi) are kept,
    the returned Csr has hi-lo rows (rowptr is the [lo, hi] slice) and GLOBAL ids in ``nbr`` / ``rowid``.
    ``nbr_range=(lo, hi)`` additionally keeps only slots whose neighbour lies in that block."""
    _need_cuda(edge_index)
    if edge_index.dtype != torch.int64 or edge_index.dim() != 2 or edge_index.size(0) != 2:
        raise ValueError(f"edge_index must be int64 [2,E], got {tuple(edge_index.shape)} {edge_index.dtype}")
    ei = edge_index.contiguous()
    E, N = ei.size(1), int(num_nodes)
    L = lib()
    cap = int(L.gg_layout_capacity(E, N, policy))
    dev = ei.device
    rowptr = torch.empty(N + 1, dtype=torch.int32, device=dev)
    nbr = torch.empty(max(cap, 1), dtype=torch.int32, device=dev)
    perm = torch.empty(max(cap, 1), dtype=torch.int32, device=dev)
    rowid = torch.empty(max(cap, 1), dtype=torch.int32, device=dev)
    ws_bytes = int(L.gg_layout_build_workspace_bytes(E, N, policy))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    lo, hi = (0, N) if row_range is None else (int(row_range[0]), int(row_range[1]))
    nlo, nhi = (0, N) if nbr_range is None else (int(nbr_range[0]), int(nbr_range[1]))
    check(L.gg_layout_build_range(_ptr(ei), E, N, policy, group_by, lo, hi, nlo, nhi, _ptr(rowptr), _ptr(nbr),
                                  _ptr(perm), _ptr(rowid), _ptr(ws), ws_bytes, _stream()),
          "gg_layout_build_range")
    bad = int(ws[:4].view(torch.int32).item())
    if bad:
        raise ValueError(f"edge_index holds {bad} edge(s) with an endpoint outside [0, {N})")
    num_slots = int(rowptr[N].item())
    if row_range is not None:
        rowptr = rowptr[lo:hi + 1]   # rows before lo are empty, so rowptr[lo] == 0
    return Csr(rowptr, nbr[:num_slots], perm[:num_slots], rowid[:num_slots], num_slots, hi - lo, E, policy,
               group_by)


def sort_pairs(keys, vals, key_bits):
    """Stable sort of u32 pairs (int32 tensors reinterpret as u32)."""
    _need_cuda(keys, vals)
    n = keys.numel()
    L = lib()
    ko, vo = torch.empty_like(keys), torch.empty_like(keys)
    ws_bytes = int(L.gg_sort_pairs_workspace_bytes(n))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=keys.device)
    check(L.gg_sort_pairs_u32(_ptr(keys), _ptr(vals), _ptr(ko), _ptr(vo), n, key_bits, _ptr(ws),
                              ws_bytes, _stream()), "gg_sort_pairs_u32")
    return ko, vo


def slot_map(a, b):
    """map[t] = slot of layout ``a`` that holds the same edge as slot t of layout ``b``."""
    assert a.num_slots == b.num_slots
    scratch = torch.empty(a.num_edges + a.num_nodes + 1, dtype=torch.int32, device=a.perm.device)
    out = torch.empty(max(b.num_slots, 1), dtype=torch.int32, device=a.perm.device)[:b.num_slots]
    check(lib().gg_layout_slot_map(_ptr(a.perm), _ptr(b.perm), a.num_slots, a.num_edges, a.num_nodes,
                                   _ptr(scratch), _ptr(out), _stream()), "gg_layout_slot_map")
    return out


def slot_weights(csr, edge_index=None, edge_weight=None, loop_fill=1.0):
    dev = csr.perm.device
    out = torch.empty(max(csr.num_slots, 1), dtype=torch.float32, device=dev)[:csr.num_slots]
    scratch = None
    ei = None
    if edge_weight is not None:
        _need_cuda(edge_weight, edge_index)
        edge_weight = edge_weight.contiguous().float()
        ei = edge_index.contiguous()
        scratch = torch.empty(max(csr.num_nodes, 1), dtype=torch.int32, device=dev)
    check(lib().gg_layout_slot_weights(_ptr(csr.perm), csr.num_slots, _ptr(ei), _ptr(edge_weight),
                                       csr.num_edges, csr.num_nodes, csr.policy, float(loop_fill),
                                       _ptr(scratch), _ptr(out), _stream()), "gg_layout_slot_weights")
    return out


def segment_degree(csr, w_slot=None):
    deg = torch.empty(max(csr.num_nodes, 1), dtype=torch.float32, device=csr.rowptr.device)[:csr.num_nodes]
    check(lib().gg_segment_degree(_ptr(csr.rowptr), _ptr(w_slot), csr.num_nodes, _ptr(deg), _stream()),
          "gg_segment_degree")
    return deg


def gcn_norm(csr, deg, w_slot=None):
    out = torch.empty(max(csr.num_slots, 1), dtype=torch.float32, device=deg.device)[:csr.num_slots]
    check(lib().gg_gcn_norm(_ptr(csr.rowid), _ptr(csr.nbr), _ptr(w_slot), _ptr(deg), csr.num_slots,
                            _ptr(out), _stream()), "gg_gcn_norm")
    return out


def mean_weights(csr_t, deg):
    """1/deg[nbr[s]] per slot of the transposed layout (backward of a mean aggregation)."""
    out = torch.empty(max(csr_t.num_slots, 1), dtype=torch.float32, device=deg.device)[:csr_t.num_slots]
    check(lib().gg_mean_weights(_ptr(csr_t.nbr), _ptr(deg), csr_t.num_slots, _ptr(out), _stream()),
          "gg_mean_weights")
    return out


def id_count(ids, num_nodes):
    _need_cuda(ids)
    ids = ids.contiguous().long()
    cnt = torch.empty(max(num_nodes, 1), dtype=torch.float32, device=ids.device)[:num_nodes]
    check(lib().gg_id_count(_ptr(ids), ids.numel(), num_nodes, _ptr(cnt), _stream()), "gg_id_count")
    return cnt


# --------------------------------------------------------------------------------------------
# aggregation
# --------------------------------------------------------------------------------------------
def cast_bf16(x):
    """fp32 [n, f] -> bf16 [n, f], round to nearest even (f % 4 == 0)."""
    _need_cuda(x)
    x, ld = _rows(x, "x")
    n, f = x.shape
    out = torch.empty((n, f), dtype=torch.bfloat16, device=x.device)
    check(lib().gg_cast_f32_bf16(_ptr(x), ld, n, f, _ptr(out), max(f, 1), _stream()), "gg_cast_f32_bf16")
    return out


def bf16_gather_ok(f):
    return f % 8 == 0 and 0 < f <= 256


def _spmm_bf16(csr, x, w_slot, reduce, x_self, self_scale, bias):
    if x.dim() != 2 or not x.is_contiguous():
        x = x.contiguous()
    n, f = csr.num_nodes, x.size(1)
    if not bf16_gather_ok(f):
        raise ValueError(f"bf16-gather aggregation needs f % 8 == 0 and f <= 256, got f={f}")
    out = torch.empty((n, f), dtype=torch.float32, device=x.device)
    if n == 0:
        return out
    ld_self = 0
    if x_self is not None:
        x_self, ld_self = _rows(x_self, "x_self")
    if bias is not None:
        bias = bias.contiguous()
    L = lib()
    item_row, item_slot, items = csr.plan
    ws_bytes = int(L.gg_spmm_mp_workspace_bytes(items, f))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
    check(L.gg_spmm_mp_bf16(_ptr(csr.rowptr), _ptr(csr.nbr), _ptr(w_slot), _ptr(item_row), _ptr(item_slot), items,
                            _ptr(x), f, _ptr(out), f, n, f, reduce, _ptr(x_self), ld_self, float(self_scale),
                            _ptr(bias), _ptr(ws), ws_bytes, _spmm_flags(), _stream()), "gg_spmm_mp_bf16")
    return out


SELL_SEG = int(_os.environ.get("GG_SELL_SEG", "256"))   # rows longer than this are cut into virtual rows (multiple of 4)
SELL_MAX_F = int(_os.environ.get("GG_SELL_MAX_F", "128"))
# hub hint of the sliced-ELL aggregation: rows of the ~SELL_HUB_BYTES / (4 f) most referenced source nodes are kept in L2,
# the rest is streamed (0 = off).  Only used when the gathered matrix does not fit the L2 anyway.
SELL_HUB_BYTES = int(_os.environ.get("GG_SELL_HUB_MB", "32")) << 20
SELL_HUB_MIN_F = 64   # below this width the kernel is latency bound, not DRAM bound: the hint measures as noise   # auto: widths up to this run on the sliced-ELL kernel


class SellLayout:
    """Degree-sorted sliced-ELL re-layout of a Csr for the narrow-row aggregation (csrc/spmm_sell.cu): built once per
    layout by ``gg_sell_build``; one host read of the sizes (layout-build level, like ``layout_build``'s E')."""

    def __init__(self, csr, seg=None):
        L = lib()
        seg = int(seg or SELL_SEG)
        n, slots, dev = csr.num_nodes, csr.num_slots, csr.rowptr.device
        vcap = int(L.gg_sell_vrow_capacity(n, slots, seg))
        ucap = int(L.gg_sell_unit_capacity(n, slots, seg))
        hcap = int(L.gg_sell_split_capacity(slots, seg))
        i32 = lambda k: torch.empty(max(int(k), 1), dtype=torch.int32, device=dev)
        self.chunk_ptr, self.idx, self.slot_of = i32(vcap // 8 + 1), i32(4 * ucap), i32(4 * ucap)
        self.vdst, self.hub_rows, self.hub_pptr = i32(vcap), i32(hcap), i32(hcap + 1)
        info = torch.zeros(8, dtype=torch.int32, device=dev)
        ws = torch.empty(int(L.gg_sell_build_workspace_bytes(n, slots, seg)), dtype=torch.uint8, device=dev)
        check(L.gg_sell_build(_ptr(csr.rowptr), _ptr(csr.nbr), n, slots, seg, _ptr(self.chunk_ptr), _ptr(self.idx),
                              _ptr(self.slot_of), _ptr(self.vdst), _ptr(self.hub_rows), _ptr(self.hub_pptr), _ptr(info),
                              _ptr(ws), ws.numel(), _stream()), "gg_sell_build")
        self.vrows, self.chunks, self.units, self.hubs, self.partial_rows = (int(v) for v in info[:5].tolist())
        self.seg = seg      # (no back-reference to the Csr: a csr <-> layout cycle would keep ~3 GB per products-sized
        # layout alive until Python's cycle collector runs — measured as +3.5 GiB of HBM per e2e step)
        self.total = 4 * self.units        # entries of idx / slot_of in use (the arrays keep their capacity)
        self._w = None
        self._hint = {}                    # hubs -> idx with the hub bit (gg_sell_hub_hint)
        self._nbr, self._n, self._slots = csr.nbr, n, slots

    def idx_hint(self, hubs):
        """idx with bit 30 marking the `hubs` most referenced sources (built once per hub count)."""
        hit = self._hint.get(hubs)
        if hit is None:
            L = lib()
            dev = self.idx.device
            hit = torch.empty_like(self.idx)
            ws_bytes = int(L.gg_sell_hub_hint_workspace_bytes(self._n))
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            check(L.gg_sell_hub_hint(_ptr(self._nbr), self._slots, self._n, _ptr(self.idx), self.total, int(hubs), _ptr(hit),
                                     _ptr(ws), ws_bytes, _stream()), "gg_sell_hub_hint")
            self._hint = {hubs: hit}
        return hit

    def weights(self, w_slot):
        """Per-slot weights re-laid in unit order (padding = 0).  The last permutation is kept (a cached GCN norm hits
        every step; a per-step array such as GAT's alpha is permuted per call and replaces the entry)."""
        if w_slot is None:
            return None
        hit = self._w
        if hit is not None and hit[0] is w_slot and hit[1] == w_slot._version:
            return hit[2]
        src = w_slot.contiguous()
        dst = torch.empty(max(self.total, 4), dtype=torch.float32, device=src.device)
        check(lib().gg_sell_permute_f32(_ptr(self.slot_of), self.total, _ptr(src), _ptr(dst), _stream()),
              "gg_sell_permute_f32")
        self._w = (w_slot, w_slot._version, dst)
        return dst


def sell_layout(csr):
    if csr._sell is None:
        csr._sell = SellLayout(csr)
    return csr._sell


def _sell_hub_idx(sl, n_src, f, flags):
    """(idx, flags) of a sliced-ELL aggregation call gathering ``n_src`` rows of width ``f``."""
    # hub hint: only when the gathered matrix is (much) larger than what the hint keeps resident
    if SELL_HUB_BYTES and f >= SELL_HUB_MIN_F and n_src * f * 4 > 2 * SELL_HUB_BYTES and (flags & 4):
        # hub count in powers of two: the hint array is rebuilt only when the width class changes
        hubs = 1 << max(10, (SELL_HUB_BYTES // (4 * f)).bit_length() - 1)
        return sl.idx_hint(hubs), flags | 8
    return sl.idx, flags


def _spmm_sell(csr, x, ldx, x_ptr, w_slot, reduce, x_self, ld_self, self_scale, bias, r1, out, ldo, out_peers):
    sl = sell_layout(csr)
    L = lib()
    f = x.size(1)
    ws_bytes = int(L.gg_spmm_sell_workspace_bytes(sl.partial_rows, f))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
    peers = (out_peers._arr, len(out_peers.ptrs), out_peers.rows_per_rank) if out_peers is not None else (None, 1, max(csr.num_nodes, 1))
    idx, flags = _sell_hub_idx(sl, x.size(0), f, _spmm_flags())
    check(L.gg_spmm_sell_f32(_ptr(sl.chunk_ptr), sl.chunks, _ptr(idx), _ptr(sl.weights(w_slot)), _ptr(sl.vdst),
                             _ptr(csr.rowptr), _ptr(sl.hub_rows), _ptr(sl.hub_pptr), sl.hubs, sl.partial_rows, x_ptr, ldx,
                             _ptr(out), ldo, peers[0], peers[1], peers[2], csr.num_nodes, f, reduce, _ptr(x_self), ld_self,
                             float(self_scale), _ptr(bias), _ptr(r1[0]), _ptr(r1[1]), _ptr(r1[2]), _ptr(r1[3]), _ptr(ws),
                             ws_bytes, flags, _stream()), "gg_spmm_sell_f32")


def _al16(t):
    return t is None or t.data_ptr() % 16 == 0


def spmm_max(csr, x, w_slot=None, x_self=None, self_scale=0.0, bias=None, algo=None):
    """Max aggregation -> (out [n, f], arg int32 [n, f]):
    out[i,:] = max_{s in segment i} w[s]*x[nbr[s],:] (0 for an empty segment) + self_scale*x_self[i,:] + bias;
    arg[i,c] = the first slot (in slot order) reaching the maximum, -1 for an empty segment (csrc/spmm_max.cu).
    The sliced-ELL kernel runs where ``spmm`` would run its sliced-ELL path (f % 4 == 0, 16-byte rows, n + slots >=
    2**14; wider rows as column tiles of 128), the warp-per-row kernel otherwise.  ``algo`` ('sell' | 'row') overrides the
    choice for this call."""
    _need_cuda(x, w_slot, x_self, bias, csr.rowptr)
    x, ldx = _rows(x, "x")
    n, f = csr.num_nodes, x.size(1)
    dev = x.device
    out = torch.empty((n, f), dtype=torch.float32, device=dev)
    arg = torch.empty((n, f), dtype=torch.int32, device=dev)
    if n == 0 or f == 0:
        return out, arg
    ld_self = 0
    if x_self is not None:
        x_self, ld_self = _rows(x_self, "x_self")
    if bias is not None:
        bias = bias.contiguous()
    L = lib()
    aligned = f % 4 == 0 and ldx % 4 == 0 and _al16(x) and _al16(bias) and (x_self is None or (ld_self % 4 == 0 and _al16(x_self)))
    if algo is None:
        algo = "sell" if aligned and n + csr.num_slots >= 1 << 14 else "row"
    if algo == "sell":
        if not aligned:
            raise ValueError("spmm_max: the sliced-ELL kernel needs f % 4 == 0 and 16-byte aligned rows")
        sl = sell_layout(csr)
        ws_bytes = int(L.gg_spmm_sell_max_workspace_bytes(sl.partial_rows, f))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        idx, flags = _sell_hub_idx(sl, x.size(0), min(f, 128), _spmm_flags())
        check(L.gg_spmm_sell_max_f32(_ptr(sl.chunk_ptr), sl.chunks, _ptr(idx), _ptr(sl.slot_of), _ptr(sl.weights(w_slot)),
                                     _ptr(sl.vdst), _ptr(sl.hub_rows), _ptr(sl.hub_pptr), sl.hubs, sl.partial_rows, _ptr(x),
                                     ldx, _ptr(out), f, _ptr(arg), f, n, f, _ptr(x_self), ld_self, float(self_scale),
                                     _ptr(bias), _ptr(ws), ws_bytes, flags, _stream()), "gg_spmm_sell_max_f32")
    elif algo == "row":
        check(L.gg_spmm_row_max_f32(_ptr(csr.rowptr), _ptr(csr.nbr), _ptr(w_slot), _ptr(x), ldx, _ptr(out), f, _ptr(arg), f,
                                    n, f, _ptr(x_self), ld_self, float(self_scale), _ptr(bias), _stream()),
              "gg_spmm_row_max_f32")
    else:
        raise ValueError(f"spmm_max: algo={algo!r}")
    return out, arg


def spmm_max_bwd(csc, csc2csr, g, arg, w_slot_csc=None, self_scale=0.0, algo=None):
    """Backward of ``spmm_max`` wrt x: dx[j,:] = sum over the CSC slots t of row j whose edge won its column
    (arg[target, c] == CSR slot of the edge) of w_csc[t] * g[target, :], + self_scale * g[j, :].  Path choice as in
    ``spmm_max``."""
    _need_cuda(g, arg, w_slot_csc, csc.rowptr)
    g, ldg = _rows(g, "g")
    arg = arg.contiguous()
    n, f = csc.num_nodes, g.size(1)
    dev = g.device
    dx = torch.empty((n, f), dtype=torch.float32, device=dev)
    if n == 0 or f == 0:
        return dx
    L = lib()
    aligned = f % 4 == 0 and ldg % 4 == 0 and _al16(g) and _al16(arg)
    if algo is None:
        algo = "sell" if aligned and n + csc.num_slots >= 1 << 14 else "row"
    if algo == "sell":
        if not aligned:
            raise ValueError("spmm_max_bwd: the sliced-ELL kernel needs f % 4 == 0 and 16-byte aligned rows")
        sl = sell_layout(csc)
        emap = _sell_edge_map(csc, csc2csr)
        ws_bytes = int(L.gg_spmm_sell_max_workspace_bytes(sl.partial_rows, f))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        check(L.gg_spmm_sell_max_bwd_f32(_ptr(sl.chunk_ptr), sl.chunks, _ptr(sl.idx), _ptr(emap), _ptr(sl.weights(w_slot_csc)),
                                         _ptr(sl.vdst), _ptr(sl.hub_rows), _ptr(sl.hub_pptr), sl.hubs, sl.partial_rows,
                                         _ptr(g), ldg, _ptr(arg), f, n, f, float(self_scale), _ptr(dx), f, _ptr(ws), ws_bytes,
                                         _spmm_flags(), _stream()), "gg_spmm_sell_max_bwd_f32")
    elif algo == "row":
        check(L.gg_spmm_row_max_bwd_f32(_ptr(csc.rowptr), _ptr(csc.nbr), _ptr(csc2csr), _ptr(w_slot_csc), _ptr(g), ldg,
                                        _ptr(arg), f, n, f, float(self_scale), _ptr(dx), f, _stream()),
              "gg_spmm_row_max_bwd_f32")
    else:
        raise ValueError(f"spmm_max_bwd: algo={algo!r}")
    return dx


def spmm_max_heads(csr, x, w, heads, bias=None):
    """``spmm_max`` with one weight per (slot, head): column c of x uses w[s, c // (f / heads)] (w [E', heads]); the
    warp-per-row kernel (csrc/attn_agg.cu).  -> (out [n, f], arg int32 [n, f])."""
    _need_cuda(x, w, bias, csr.rowptr)
    x, ldx = _rows(x, "x")
    n, f = csr.num_nodes, x.size(1)
    out = torch.empty((n, f), dtype=torch.float32, device=x.device)
    arg = torch.empty((n, f), dtype=torch.int32, device=x.device)
    if bias is not None:
        bias = bias.contiguous()
    check(lib().gg_spmm_row_max_heads_f32(_ptr(csr.rowptr), _ptr(csr.nbr), _ptr(w.contiguous()), int(heads), _ptr(x), ldx,
                                          _ptr(out), f, _ptr(arg), f, n, f, _ptr(bias), _stream()),
          "gg_spmm_row_max_heads_f32")
    return out, arg


def spmm_max_heads_bwd(csc, csc2csr, g, arg, w, heads):
    """Backward of ``spmm_max_heads`` wrt x; ``w`` in CSR slot order [E', heads]."""
    _need_cuda(g, arg, w, csc.rowptr)
    g, ldg = _rows(g, "g")
    arg = arg.contiguous()
    n, f = csc.num_nodes, g.size(1)
    dx = torch.empty((n, f), dtype=torch.float32, device=g.device)
    check(lib().gg_spmm_row_max_heads_bwd_f32(_ptr(csc.rowptr), _ptr(csc.nbr), _ptr(csc2csr), _ptr(w.contiguous()),
                                              int(heads), _ptr(g), ldg, _ptr(arg), f, n, f, _ptr(dx), f, _stream()),
          "gg_spmm_row_max_heads_bwd_f32")
    return dx


def max_winner_sddmm(csr, arg, g, h, heads=1):
    """dalpha [E', heads]: dalpha[s, k] = sum over the columns c of head k that slot s won (arg[i, c] == s) of
    g[i, c] * h[nbr[s], c] — the gradient of per-slot weights through ``spmm_max`` / ``spmm_max_heads``; bitwise
    deterministic (csrc/attn_agg.cu)."""
    _need_cuda(g, h, arg, csr.rowptr)
    g, ldg = _rows(g, "g")
    h, ldh = _rows(h, "h")
    arg = arg.contiguous()
    f = g.size(1)
    dalpha = _f32((csr.num_slots, heads), g.device)
    check(lib().gg_max_winner_sddmm_f32(_ptr(csr.rowptr), _ptr(csr.nbr), _ptr(arg), f, _ptr(g), ldg, _ptr(h), ldh,
                                        csr.num_nodes, int(heads), f, _ptr(dalpha), _stream()), "gg_max_winner_sddmm_f32")
    return dalpha


EDGE_MAX_KD = 256   # edge_dim limit of edge_max (its W_a column tile is staged in shared memory)


def _edge_rows(a, name):
    if a.dtype != torch.float32 or a.dim() != 2:
        raise ValueError(f"{name}: expected a 2-D float32 tensor, got {tuple(a.shape)} {a.dtype}")
    return _rows(a, name)


def edge_row_reduce(csr, a, mean=False):
    """[n, kd]: out[i] = sum over the CSR slots s of row i of a[perm[s]] (slot order), / indeg(i) with ``mean``; rows
    without slots 0.  ``a``: [E, kd] in edge order (csrc/edge_agg.cu)."""
    _need_cuda(a, csr.rowptr)
    a, lda = _edge_rows(a, "edge_feature")
    n, k = csr.num_nodes, a.size(1)
    out = _f32((n, k), a.device)
    check(lib().gg_edge_row_reduce_f32(_ptr(csr.rowptr), _ptr(csr.perm), n, _ptr(a), lda, k, int(bool(mean)), _ptr(out),
                                       max(k, 1), _stream()), "gg_edge_row_reduce_f32")
    return out


def edge_rows_self(csr, h=None, y=None, z=None, mean=False):
    """y + r * h + z per row (each term optional), r = indeg(i) or, with ``mean``, [indeg(i) > 0]; written into ``y``
    when given."""
    _need_cuda(h, y, z, csr.rowptr)
    n = csr.num_nodes
    ldh = ldy = ldz = 0
    if h is not None:
        h, ldh = _rows(h, "h")
    if z is not None:
        z, ldz = _rows(z, "z")
    f = next(t.size(1) for t in (h, y, z) if t is not None)
    if y is not None:
        y_t, ldy = _rows(y, "y")
        assert y_t is y
        out, ldo = y, ldy
    else:
        out, ldo = _f32((n, f), csr.rowptr.device), max(f, 1)
    check(lib().gg_edge_rows_self_f32(_ptr(csr.rowptr), n, f, int(bool(mean)), _ptr(y), ldy, _ptr(h), ldh, _ptr(z), ldz,
                                      _ptr(out), ldo, _stream()), "gg_edge_rows_self_f32")
    return out


def max_mask(g, arg):
    """g where arg >= 0, else 0."""
    _need_cuda(g, arg)
    g, ldg = _rows(g, "g")
    arg = arg.contiguous()
    n, f = g.shape
    out = _f32((n, f), g.device)
    check(lib().gg_max_mask_f32(_ptr(g), ldg, _ptr(arg), f, n, f, _ptr(out), max(f, 1), _stream()), "gg_max_mask_f32")
    return out


def edge_max(csr, h_j, h_i, a, w_a, x_self=None, self_scale=0.0, bias=None, algo=None):
    """Max aggregation with the edge term -> (out [n, f], arg int32 [n, f]):
    out[i,c] = max_{s in row i} h_j[nbr[s],c] + a[perm[s]] . w_a[c] (+ h_i[i,c] where the row has a slot; 0 for an empty
    row) + self_scale*x_self + bias; arg = the first slot reaching the maximum, -1 for an empty row.  ``h_i`` may be None;
    ``w_a``: [f, kd] (rows may be strided, e.g. a column slice of nn.Linear's weight).  Path choice as ``spmm_max``;
    ``algo`` ('sell' | 'row') overrides it."""
    _need_cuda(h_j, h_i, a, w_a, x_self, bias, csr.rowptr)
    h_j, ldj = _rows(h_j, "h_j")
    a, lda = _edge_rows(a, "edge_feature")
    w_a, ldw = _rows(w_a, "w_a")
    n, f, kd = csr.num_nodes, h_j.size(1), a.size(1)
    if kd > EDGE_MAX_KD:
        raise NotImplementedError(f"edge_max: edge_dim {kd} > {EDGE_MAX_KD}")
    dev = h_j.device
    out = _f32((n, f), dev)
    arg = torch.empty((n, f), dtype=torch.int32, device=dev)
    if n == 0 or f == 0:
        return out, arg
    ldi = ld_self = 0
    if h_i is not None:
        h_i, ldi = _rows(h_i, "h_i")
    if x_self is not None:
        x_self, ld_self = _rows(x_self, "x_self")
    if bias is not None:
        bias = bias.contiguous()
    L = lib()
    aligned = (f % 4 == 0 and ldj % 4 == 0 and _al16(h_j) and _al16(bias) and
               (h_i is None or (ldi % 4 == 0 and _al16(h_i))) and (x_self is None or (ld_self % 4 == 0 and _al16(x_self))))
    if algo is None:
        algo = "sell" if aligned and n + csr.num_slots >= 1 << 14 else "row"
    if algo == "sell":
        if not aligned:
            raise ValueError("edge_max: the sliced-ELL kernel needs f % 4 == 0 and 16-byte aligned rows")
        sl = sell_layout(csr)
        ws_bytes = int(L.gg_spmm_sell_max_workspace_bytes(sl.partial_rows, f))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        check(L.gg_edge_max_sell_f32(_ptr(sl.chunk_ptr), sl.chunks, _ptr(sl.idx), _ptr(sl.slot_of), _ptr(csr.perm),
                                     _ptr(sl.vdst), _ptr(sl.hub_rows), _ptr(sl.hub_pptr), sl.hubs, sl.partial_rows,
                                     _ptr(h_j), ldj, _ptr(h_i), ldi, _ptr(a), lda, kd, _ptr(w_a), ldw, _ptr(out), f,
                                     _ptr(arg), f, n, f, _ptr(x_self), ld_self, float(self_scale), _ptr(bias), _ptr(ws),
                                     ws_bytes, _spmm_flags(), _stream()), "gg_edge_max_sell_f32")
    elif algo == "row":
        check(L.gg_edge_max_row_f32(_ptr(csr.rowptr), _ptr(csr.nbr), _ptr(csr.perm), _ptr(h_j), ldj, _ptr(h_i), ldi, _ptr(a),
                                    lda, kd, _ptr(w_a), ldw, _ptr(out), f, _ptr(arg), f, n, f, _ptr(x_self), ld_self,
                                    float(self_scale), _ptr(bias), _stream()), "gg_edge_max_row_f32")
    else:
        raise ValueError(f"edge_max: algo={algo!r}")
    return out, arg


def edge_max_winner(csr, arg, g, w_a):
    """d edge_feature [E, kd] of ``edge_max``: row perm[s] = sum over the columns c slot s won of g[i,c] w_a[c], in
    column order; 0 for an edge that won nothing."""
    _need_cuda(arg, g, w_a, csr.rowptr)
    g, ldg = _rows(g, "g")
    w_a, ldw = _rows(w_a, "w_a")
    arg = arg.contiguous()
    n, f, kd = csr.num_nodes, g.size(1), w_a.size(1)
    da = _f32((csr.num_edges, kd), g.device)
    check(lib().gg_edge_max_winner_f32(_ptr(csr.rowptr), _ptr(csr.perm), _ptr(arg), f, _ptr(g), ldg, _ptr(w_a), ldw, n, f,
                                       kd, _ptr(da), max(kd, 1), _stream()), "gg_edge_max_winner_f32")
    return da


def edge_max_wgrad(csr, arg, g, a):
    """d w_a [f, kd] of ``edge_max``: sum_i g[i,c] a[perm[arg[i,c]]] over the rows with arg >= 0 (fixed order)."""
    _need_cuda(arg, g, a, csr.rowptr)
    g, ldg = _rows(g, "g")
    a, lda = _edge_rows(a, "edge_feature")
    arg = arg.contiguous()
    n, f, kd = csr.num_nodes, g.size(1), a.size(1)
    L = lib()
    dw = _f32((f, kd), g.device)
    ws_bytes = int(L.gg_edge_max_wgrad_workspace_bytes(n, f, kd))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=g.device)
    check(L.gg_edge_max_wgrad_f32(_ptr(csr.perm), _ptr(arg), f, _ptr(g), ldg, _ptr(a), lda, n, f, kd, _ptr(dw), max(kd, 1),
                                  _ptr(ws), ws_bytes, _stream()), "gg_edge_max_wgrad_f32")
    return dw


def _spline_u(u, csr):
    if u.dtype != torch.float32 or u.dim() != 1 or u.numel() != csr.num_edges:
        raise ValueError(f"pseudo-coordinates: expected a [{csr.num_edges}] float32 tensor, got {tuple(u.shape)} {u.dtype}")
    return u.contiguous()


def _spline_algo(csr, f, lds, tensors, algo, name):
    aligned = f % 4 == 0 and all(ld % 4 == 0 for ld in lds) and all(_al16(t) for t in tensors)
    if algo is None:
        algo = "sell" if aligned and csr.num_nodes + csr.num_slots >= 1 << 14 else "row"
    if algo == "sell" and not aligned:
        raise ValueError(f"{name}: the sliced-ELL kernel needs f % 4 == 0 and 16-byte aligned rows")
    if algo not in ("sell", "row"):
        raise ValueError(f"{name}: algo={algo!r}")
    return algo


def spline_spread(csr, x, u, w_slot=None, mean=False, algo=None):
    """[n, 2f] = [sum_s w_s c0_s x[nbr[s]] | sum_s w_s c1_s x[nbr[s]]] per row (/ indeg with ``mean``), (c0, c1) the
    degree-1 open B-spline coefficients of the pseudo-coordinate u[perm[s]] (kernel size 2; csrc/spline_agg.cu).
    ``u``: [E] float32 in edge order; ``w_slot``: per-slot weights of ``csr`` or None.  Path choice as ``spmm_max``;
    ``algo`` ('sell' | 'row') overrides it."""
    _need_cuda(x, u, w_slot, csr.rowptr)
    x, ldx = _rows(x, "x")
    u = _spline_u(u, csr)
    n, f = csr.num_nodes, x.size(1)
    out = _f32((n, 2 * f), x.device)
    if n == 0 or f == 0:
        return out
    L = lib()
    if _spline_algo(csr, f, (ldx,), (x,), algo, "spline_spread") == "sell":
        sl = sell_layout(csr)
        ws_bytes = int(L.gg_spmm_sell_max_workspace_bytes(sl.partial_rows, f))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
        check(L.gg_spline_spread_sell_f32(_ptr(sl.chunk_ptr), sl.chunks, _ptr(sl.idx), _ptr(sl.slot_of),
                                          _ptr(sl.weights(w_slot)), _ptr(csr.perm), _ptr(u), _ptr(sl.vdst), _ptr(csr.rowptr),
                                          _ptr(sl.hub_rows), _ptr(sl.hub_pptr), sl.hubs, sl.partial_rows, _ptr(x), ldx,
                                          _ptr(out), 2 * f, n, f, int(bool(mean)), _ptr(ws), ws_bytes, _spmm_flags(),
                                          _stream()), "gg_spline_spread_sell_f32")
    else:
        check(L.gg_spline_spread_row_f32(_ptr(csr.rowptr), _ptr(csr.nbr), _ptr(csr.perm), _ptr(w_slot), _ptr(u), _ptr(x), ldx,
                                         _ptr(out), 2 * f, n, f, int(bool(mean)), _stream()), "gg_spline_spread_row_f32")
    return out


def spline_blend(csr, y, u, w_slot=None, mean=False, residual=None, bias=None, algo=None):
    """[n, f]: sum_s w_s (c0_s y[nbr[s], :f] + c1_s y[nbr[s], f:]) per row (/ indeg with ``mean``) + residual + bias;
    ``y``: [*, 2f].  Coefficients, ``u``, ``w_slot`` and the path choice as ``spline_spread``."""
    _need_cuda(y, u, w_slot, residual, bias, csr.rowptr)
    y, ldy = _rows(y, "y")
    u = _spline_u(u, csr)
    n, f = csr.num_nodes, y.size(1) // 2
    if y.size(1) != 2 * f:
        raise ValueError(f"spline_blend: y must have an even width, got {tuple(y.shape)}")
    out = _f32((n, f), y.device)
    if n == 0 or f == 0:
        return out
    ld_res = 0
    if residual is not None:
        residual, ld_res = _rows(residual, "residual")
    if bias is not None:
        bias = bias.contiguous()
    L = lib()
    if _spline_algo(csr, f, (ldy, ld_res), (y, residual, bias), algo, "spline_blend") == "sell":
        sl = sell_layout(csr)
        ws_bytes = int(L.gg_spmm_sell_max_workspace_bytes(sl.partial_rows, f))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=y.device)
        check(L.gg_spline_blend_sell_f32(_ptr(sl.chunk_ptr), sl.chunks, _ptr(sl.idx), _ptr(sl.slot_of),
                                         _ptr(sl.weights(w_slot)), _ptr(csr.perm), _ptr(u), _ptr(sl.vdst), _ptr(csr.rowptr),
                                         _ptr(sl.hub_rows), _ptr(sl.hub_pptr), sl.hubs, sl.partial_rows, _ptr(y), ldy,
                                         _ptr(out), f, n, f, int(bool(mean)), _ptr(residual), ld_res, _ptr(bias), _ptr(ws),
                                         ws_bytes, _spmm_flags(), _stream()), "gg_spline_blend_sell_f32")
    else:
        check(L.gg_spline_blend_row_f32(_ptr(csr.rowptr), _ptr(csr.nbr), _ptr(csr.perm), _ptr(w_slot), _ptr(u), _ptr(y), ldy,
                                        _ptr(out), f, n, f, int(bool(mean)), _ptr(residual), ld_res, _ptr(bias), _stream()),
              "gg_spline_blend_row_f32")
    return out


def spline_du(csr, u, a, a_half, b, b_half, f):
    """[E] in edge order: du[perm[s]] = (dc[(t+1) mod 2] - dc[t mod 2]) / indeg(i) for the slots s of row i, t = trunc(u),
    dc_k = <a[i, k a_half : k a_half + f], b[nbr[s], k b_half : k b_half + f]> (a_half / b_half = 0: one operand for both
    matrices) — the pseudo-coordinate gradient of the mean B-spline aggregation."""
    _need_cuda(u, a, b, csr.rowptr)
    a, lda = _rows(a, "a")
    b, ldb = _rows(b, "b")
    u = _spline_u(u, csr)
    du = _f32((csr.num_edges,), u.device)
    check(lib().gg_spline_du_f32(_ptr(csr.rowptr), _ptr(csr.nbr), _ptr(csr.perm), _ptr(u), _ptr(a), lda, int(a_half),
                                 _ptr(b), ldb, int(b_half), csr.num_nodes, int(f), _ptr(du), _stream()), "gg_spline_du_f32")
    return du


def rows_epilogue(x, mean_csr=None, rank1=None, heads=1, bias=None, out=None):
    """out[i, :] = x[i, :] / indeg(i) (with ``mean_csr``; rows without in-edges unscaled) + s1[i, k] v1 + s2[i, k] v2
    (``rank1`` = (s1 [n, heads], v1 [f], s2, v2), k the column's head) + bias.  ``out`` may be ``x``."""
    _need_cuda(x, bias)
    x, ldx = _rows(x, "x")
    n, f = x.shape
    if out is None:
        out = torch.empty((n, f), dtype=torch.float32, device=x.device)
    out_t, ldo = _rows(out, "out")
    assert out_t is out, "out must have unit inner stride"
    r1 = [t.contiguous() if t is not None else None for t in (rank1 or (None, None, None, None))]
    if bias is not None:
        bias = bias.contiguous()
    check(lib().gg_rows_epilogue_f32(_ptr(x), ldx, n, f, _ptr(mean_csr.rowptr if mean_csr is not None else None),
                                     int(heads), _ptr(r1[0]), _ptr(r1[1]), _ptr(r1[2]), _ptr(r1[3]), _ptr(bias), _ptr(out),
                                     ldo, _stream()), "gg_rows_epilogue_f32")
    return out


class PeerRows:
    """Where the rows of a peer-output SpMM go: ``ptrs[o]`` = device pointer (peer memory, already offset
    to this rank's column slice) of rank o's [rows_per_rank, ld] block."""
    __slots__ = ("ptrs", "rows_per_rank", "ld", "_arr")

    def __init__(self, ptrs, rows_per_rank, ld):
        self.ptrs, self.rows_per_rank, self.ld = [int(p) for p in ptrs], int(rows_per_rank), int(ld)
        self._arr = (ctypes.c_void_p * len(self.ptrs))(*self.ptrs)


def spmm(csr, x, w_slot=None, reduce=SUM, x_self=None, self_scale=0.0, bias=None, out=None, rank1=None,
         x_row_base=0, out_peers=None, algo=None):
    """out[i,:] = reduce_{s in segment i} w[s]*x[nbr[s],:] + self_scale*x_self[i,:] + bias.

    ``rank1`` = (s1 [n], v1 [f], s2 [n], v2 [f]) adds s1[i]*v1 + s2[i]*v2 in the epilogue (merge-path
    kernel only; used by the GAT backward).  ``x_row_base``: ``x`` holds rows [x_row_base, x_row_base +
    x.size(0)) of the matrix the neighbour ids index (a peer's block in the halo pipeline).
    ``out_peers`` (PeerRows): rows are stored into the owning ranks' memory instead of ``out``
    (feature-sliced exchange of the row-partitioned path); returns None."""
    _need_cuda(x, w_slot, x_self, bias, csr.rowptr)
    if x.dtype == torch.bfloat16:
        if out is not None or rank1 is not None or out_peers is not None or x_row_base:
            raise ValueError("bf16-gather aggregation: out / rank1 / out_peers / x_row_base are fp32-only")
        return _spmm_bf16(csr, x, w_slot, reduce, x_self, self_scale, bias)
    x, ldx = _rows(x, "x")
    n, f = csr.num_nodes, x.size(1)
    x_ptr = ctypes.c_void_p(x.data_ptr() - int(x_row_base) * ldx * 4)
    ld_self = 0
    if x_self is not None:
        x_self, ld_self = _rows(x_self, "x_self")
    if bias is not None:
        bias = bias.contiguous()
    L = lib()
    r1 = [t.contiguous() if t is not None else None for t in (rank1 or (None, None, None, None))]
    algo = algo or SPMM_ALGO   # ``algo`` overrides the module setting for this call
    sell_ok = f % 4 == 0 and 0 < f <= 128 and n > 0 and (ldx * 4) % 16 == 0
    if out_peers is not None:
        if out is not None:
            raise ValueError("out_peers excludes out")
        if sell_ok and (algo == "sell" or (algo == "auto" and f <= SELL_MAX_F)):
            _spmm_sell(csr, x, ldx, x_ptr, w_slot, reduce, x_self, ld_self, self_scale, bias, r1, None, out_peers.ld,
                       out_peers)
            return None
        item_row, item_slot, items = csr.plan
        ws_bytes = int(L.gg_spmm_mp_workspace_bytes(items, f))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
        check(L.gg_spmm_mpg_f32(_ptr(csr.rowptr), _ptr(csr.nbr), _ptr(w_slot), _ptr(item_row), _ptr(item_slot),
                                items, x_ptr, ldx, None, out_peers.ld, out_peers._arr, len(out_peers.ptrs),
                                out_peers.rows_per_rank, n, f, reduce, _ptr(x_self), ld_self, float(self_scale),
                                _ptr(bias), _ptr(r1[0]), _ptr(r1[1]), _ptr(r1[2]), _ptr(r1[3]), _ptr(ws), ws_bytes,
                                _spmm_flags(), _stream()), "gg_spmm_mpg_f32")
        return None
    if out is None:
        out = torch.empty((n, f), dtype=torch.float32, device=x.device)
    out_t, ldo = _rows(out, "out")
    assert out_t is out, "out must have unit inner stride"
    big = n + csr.num_slots >= 1 << 14
    if sell_ok and (algo == "sell" or (algo == "auto" and big and f <= SELL_MAX_F)):
        _spmm_sell(csr, x, ldx, x_ptr, w_slot, reduce, x_self, ld_self, self_scale, bias, r1, out, ldo, None)
        return out
    if algo == "sell":
        algo = "auto"
    if algo == "auto":
        # merge-path kernels on graphs big enough to need balancing: the grouped-slot kernel up to 128 columns (at 128 it
        # measures 4.17 ms vs 4.55 ms for the whole-warp TMA kernel on the products graph), whole warps per item with
        # several vectors per lane beyond; one-warp-per-row (odd f, tiny graphs) otherwise
        algo = "row"
        if f % 4 == 0 and big:
            algo = "mpg" if f <= 128 else ("mp" if f <= 1024 else "row")
    if rank1 is not None and algo == "row":
        algo = "mp"
    if algo == "mpg" and f % 4 == 0 and f <= 128 and n > 0:
        item_row, item_slot, items = csr.plan
        ws_bytes = int(L.gg_spmm_mp_workspace_bytes(items, f))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
        check(L.gg_spmm_mpg_f32(_ptr(csr.rowptr), _ptr(csr.nbr), _ptr(w_slot), _ptr(item_row), _ptr(item_slot),
                                items, x_ptr, ldx, _ptr(out), ldo, None, 1, max(n, 1), n, f, reduce,
                                _ptr(x_self), ld_self, float(self_scale), _ptr(bias), _ptr(r1[0]), _ptr(r1[1]),
                                _ptr(r1[2]), _ptr(r1[3]), _ptr(ws), ws_bytes, _spmm_flags(), _stream()),
              "gg_spmm_mpg_f32")
        return out
    if algo in ("mp", "mpg") and f % 4 == 0 and f <= 1024 and n > 0:
        item_row, item_slot, items = csr.plan
        ws_bytes = int(L.gg_spmm_mp_workspace_bytes(items, f))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
        check(L.gg_spmm_mp_f32(_ptr(csr.rowptr), _ptr(csr.nbr), _ptr(w_slot), _ptr(item_row), _ptr(item_slot),
                               items, x_ptr, ldx, _ptr(out), ldo, n, f, reduce, _ptr(x_self), ld_self,
                               float(self_scale), _ptr(bias), _ptr(r1[0]), _ptr(r1[1]), _ptr(r1[2]), _ptr(r1[3]),
                               _ptr(ws), ws_bytes, _spmm_flags(), _stream()),
              "gg_spmm_mp_f32")
        return out
    if rank1 is not None:
        raise ValueError("rank-1 epilogue terms need the merge-path kernel (f % 4 == 0, f <= 1024)")
    check(L.gg_spmm_f32(_ptr(csr.rowptr), _ptr(csr.nbr), _ptr(w_slot), x_ptr, ldx, _ptr(out), ldo,
                        n, f, reduce, _ptr(x_self), ld_self, float(self_scale), _ptr(bias),
                        _stream()), "gg_spmm_f32")
    return out


# --------------------------------------------------------------------------------------------
# dense transform
# --------------------------------------------------------------------------------------------
def id_gemm(segments, n, f, b_trans=False, bias=None, act=ACT_NONE, relu_mask=None, out=None):
    """out = act(sum_g diag(scale_g) A_g B_g + bias) .* (relu_mask > 0).

    ``segments``: list of (a [n,k], b [k,f] or [f,k] if b_trans, scale [n] or None)."""
    if not 1 <= len(segments) <= _lib.GG_GEMM_MAX_SEGMENTS:
        raise ValueError("id_gemm takes 1..4 K-segments")
    arr = (GemmSegment * len(segments))()
    keep = []
    dev = None
    for i, (a, b, scale) in enumerate(segments):
        _need_cuda(a, b, scale)
        a, lda = _rows(a, "a")
        b, ldb = _rows(b, "b")
        k = a.size(1)
        if a.size(0) != n or (b.size(1) if b_trans else b.size(0)) != k or \
                (b.size(0) if b_trans else b.size(1)) != f:
            raise ValueError(f"id_gemm segment {i}: a {tuple(a.shape)} b {tuple(b.shape)} "
                             f"b_trans={b_trans} do not give [{n},{f}]")
        if scale is not None:
            scale = scale.contiguous()
            assert scale.dtype == torch.float32 and scale.numel() == n
        keep += [a, b, scale]
        arr[i] = GemmSegment(a.data_ptr(), lda, b.data_ptr(), ldb,
                             scale.data_ptr() if scale is not None else None, k)
        dev = a.device
    if out is None:
        out = torch.empty((n, f), dtype=torch.float32, device=dev)
    out_t, ldo = _rows(out, "out")
    assert out_t is out
    ld_mask = 0
    if relu_mask is not None:
        relu_mask, ld_mask = _rows(relu_mask, "relu_mask")
    if bias is not None:
        bias = bias.contiguous()
    L = lib()
    if GEMM_MODE == "tc" and n > 0 and f > 0:
        ws_bytes = int(L.gg_id_gemm_tc_workspace_bytes(arr, len(segments), f))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        check(L.gg_id_gemm_tc_f32(arr, len(segments), int(b_trans), n, f, _ptr(bias), act, _ptr(relu_mask),
                                  ld_mask, _ptr(out), ldo, _ptr(ws), ws_bytes, _stream()), "gg_id_gemm_tc_f32")
        return out
    check(L.gg_id_gemm_f32(arr, len(segments), int(b_trans), n, f, _ptr(bias), act, _ptr(relu_mask),
                           ld_mask, _ptr(out), ldo, _stream()), "gg_id_gemm_f32")
    return out


def gemm_tn(a, g, row_index=None):
    """out[K,F] = sum_r a[row(r),:]^T g[row(r),:]."""
    _need_cuda(a, g, row_index)
    a, lda = _rows(a, "a")
    g, ldg = _rows(g, "g")
    k, f = a.size(1), g.size(1)
    if row_index is not None:
        row_index = row_index.contiguous().long()
        n = row_index.numel()
    else:
        n = a.size(0)
        assert g.size(0) == n
    L = lib()
    out = torch.empty((k, f), dtype=torch.float32, device=a.device)
    if GEMM_MODE == "tc" and n >= 512:   # below a couple of 256-row segments the CUDA-core kernel is as fast
        ws_bytes = int(L.gg_gemm_tn_tc_workspace_bytes(n, k, f))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=a.device)
        check(L.gg_gemm_tn_tc_f32(_ptr(a), lda, _ptr(row_index), _ptr(g), ldg, n, k, f, _ptr(out), max(f, 1),
                                  _ptr(ws), ws_bytes, _stream()), "gg_gemm_tn_tc_f32")
        return out
    ws_bytes = int(L.gg_gemm_tn_workspace_bytes(n, k, f))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=a.device)
    check(L.gg_gemm_tn_f32(_ptr(a), lda, _ptr(row_index), _ptr(g), ldg, n, k, f, _ptr(out), max(f, 1),
                           _ptr(ws), ws_bytes, _stream()), "gg_gemm_tn_f32")
    return out


def colsum(g):
    _need_cuda(g)
    g, ldg = _rows(g, "g")
    n, f = g.shape
    L = lib()
    out = torch.empty(f, dtype=torch.float32, device=g.device)
    ws_bytes = int(L.gg_colsum_workspace_bytes(n, f))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=g.device)
    check(L.gg_colsum_f32(_ptr(g), ldg, n, f, _ptr(out), _ptr(ws), ws_bytes, _stream()), "gg_colsum_f32")
    return out


def gather_rows(x, ids):
    _need_cuda(x, ids)
    x, ldx = _rows(x, "x")
    ids = ids.contiguous().long()
    m, f = ids.numel(), x.size(1)
    out = torch.empty((m, f), dtype=torch.float32, device=x.device)
    check(lib().gg_gather_rows_f32(_ptr(x), ldx, _ptr(ids), m, f, _ptr(out), max(f, 1), _stream()),
          "gg_gather_rows_f32")
    return out


def scatter_add_rows_(out, ids, x):
    """out[ids[r],:] += x[r,:] in place."""
    _need_cuda(out, ids, x)
    x, ldx = _rows(x, "x")
    out_t, ldo = _rows(out, "out")
    assert out_t is out
    ids = ids.contiguous().long()
    check(lib().gg_scatter_add_rows_f32(_ptr(x), ldx, _ptr(ids), ids.numel(), x.size(1), _ptr(out), ldo,
                                        _stream()), "gg_scatter_add_rows_f32")
    return out


def relu_grad(g, y):
    _need_cuda(g, y)
    g, ldg = _rows(g, "g")
    y, ldy = _rows(y, "y")
    n, f = g.shape
    out = torch.empty((n, f), dtype=torch.float32, device=g.device)
    check(lib().gg_relu_grad_f32(_ptr(g), ldg, _ptr(y), ldy, n, f, _ptr(out), max(f, 1), _stream()),
          "gg_relu_grad_f32")
    return out


# --------------------------------------------------------------------------------------------
# fused layer post-ops (BatchNorm1d -> activation -> row L2 normalise)
# --------------------------------------------------------------------------------------------
def bn_stats(y, eps, running_mean=None, running_var=None, momentum=0.0):
    """-> (mean [f], invstd [f]) of the columns of ``y`` (biased variance); updates the running statistics in place."""
    _need_cuda(y, running_mean, running_var)
    y, ld = _rows(y, "y")
    n, f = y.shape
    if n < 1:
        raise ValueError("bn_stats: empty batch")
    mean = torch.empty(f, dtype=torch.float32, device=y.device)
    invstd = torch.empty(f, dtype=torch.float32, device=y.device)
    L = lib()
    ws_bytes = int(L.gg_postops_workspace_bytes(n, f))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=y.device)
    check(L.gg_bn_stats_f32(_ptr(y), ld, n, f, float(eps), _ptr(mean), _ptr(invstd), _ptr(running_mean), _ptr(running_var),
                            float(momentum), _ptr(ws), ws_bytes, _stream()), "gg_bn_stats_f32")
    return mean, invstd


def postops_fwd(y, mean, invstd, gamma, beta, act, slope, l2norm):
    """-> (out, rownorm or None)"""
    _need_cuda(y, mean, invstd, gamma, beta)
    y, ld = _rows(y, "y")
    n, f = y.shape
    out = torch.empty((n, f), dtype=torch.float32, device=y.device)
    rownorm = torch.empty(max(n, 1), dtype=torch.float32, device=y.device)[:n] if l2norm else None
    check(lib().gg_postops_fwd_f32(_ptr(y), ld, n, f, _ptr(mean), _ptr(invstd), _ptr(gamma), _ptr(beta), int(act),
                                   float(slope), int(bool(l2norm)), _ptr(out), max(f, 1), _ptr(rownorm), _stream()),
          "gg_postops_fwd_f32")
    return out, rownorm


def postops_bwd(go, out, y, mean, invstd, gamma, train, act, slope, l2norm, rownorm):
    """-> (dy, dgamma or None, dbeta or None)"""
    _need_cuda(go, out, y)
    go, ld_go = _rows(go, "go")
    out, ld_o = _rows(out, "out")
    y, ld_y = _rows(y, "y")
    n, f = go.shape
    dev = go.device
    dy = torch.empty((n, f), dtype=torch.float32, device=dev)
    dgamma = dbeta = ws = None
    ws_bytes = 0
    L = lib()
    if mean is not None:
        dgamma = torch.empty(f, dtype=torch.float32, device=dev)
        dbeta = torch.empty(f, dtype=torch.float32, device=dev)
        ws_bytes = int(L.gg_postops_workspace_bytes(n, f))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    check(L.gg_postops_bwd_f32(_ptr(go), ld_go, _ptr(out), ld_o, _ptr(y), ld_y, n, f, _ptr(mean), _ptr(invstd), _ptr(gamma),
                               int(bool(train)), int(act), float(slope), int(bool(l2norm)), _ptr(rownorm), _ptr(dy),
                               max(f, 1), _ptr(dgamma), _ptr(dbeta), _ptr(ws), ws_bytes, _stream()), "gg_postops_bwd_f32")
    return dy, dgamma, dbeta


SKIP_SUM, SKIP_PREFIX = 1, 2   # gg_skip: out = act(BN(y) + res) | out = act([res | BN(y)])


def postops_skip_fwd(y, res, mode, mean, invstd, gamma, beta, act, slope, l2norm):
    """The skip epilogue -> (out, rownorm or None).  SKIP_SUM: res [n, f], out [n, f]; SKIP_PREFIX: res [n, p],
    out [n, p + f] with act(res) in the first p columns; the L2 (``l2norm``) over the whole output row."""
    _need_cuda(y, res, mean, invstd, gamma, beta)
    y, ld = _rows(y, "y")
    res, ld_res = _rows(res, "res")
    n, f = y.shape
    if res.size(0) != n:
        raise ValueError(f"postops_skip_fwd: res has {res.size(0)} rows, y {n}")
    if mode == SKIP_SUM:
        if res.size(1) != f:
            raise ValueError(f"postops_skip_fwd: a sum skip needs res [n, {f}], got {tuple(res.shape)}")
        p = 0
    elif mode == SKIP_PREFIX:
        p = res.size(1)
    else:
        raise ValueError(f"postops_skip_fwd: mode={mode}")
    out = torch.empty((n, p + f), dtype=torch.float32, device=y.device)
    rownorm = torch.empty(max(n, 1), dtype=torch.float32, device=y.device)[:n] if l2norm else None
    check(lib().gg_postops_skip_fwd_f32(_ptr(y), ld, _ptr(res), ld_res, n, f, p, int(mode), _ptr(mean), _ptr(invstd),
                                        _ptr(gamma), _ptr(beta), int(act), float(slope), int(bool(l2norm)), _ptr(out),
                                        max(p + f, 1), _ptr(rownorm), _stream()), "gg_postops_skip_fwd_f32")
    return out, rownorm


def postops_skip_bwd(go, out, y, mode, mean, invstd, gamma, train, act, slope, l2norm, rownorm):
    """-> (dy, dres, dgamma or None, dbeta or None) of ``postops_skip_fwd``; the prefix width is out's width - y's."""
    _need_cuda(go, out, y)
    go, ld_go = _rows(go, "go")
    out, ld_o = _rows(out, "out")
    y, ld_y = _rows(y, "y")
    n, f = y.shape
    p = out.size(1) - f if mode == SKIP_PREFIX else 0
    dev = go.device
    dy = torch.empty((n, f), dtype=torch.float32, device=dev)
    dres = torch.empty((n, p if mode == SKIP_PREFIX else f), dtype=torch.float32, device=dev)
    dgamma = dbeta = ws = None
    ws_bytes = 0
    L = lib()
    if mean is not None:
        dgamma = torch.empty(f, dtype=torch.float32, device=dev)
        dbeta = torch.empty(f, dtype=torch.float32, device=dev)
        ws_bytes = int(L.gg_postops_workspace_bytes(n, f))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    check(L.gg_postops_skip_bwd_f32(_ptr(go), ld_go, _ptr(out), ld_o, _ptr(y), ld_y, n, f, p, int(mode), _ptr(mean),
                                    _ptr(invstd), _ptr(gamma), int(bool(train)), int(act), float(slope),
                                    int(bool(l2norm)), _ptr(rownorm), _ptr(dy), max(f, 1), _ptr(dres),
                                    max(dres.size(1), 1), _ptr(dgamma), _ptr(dbeta), _ptr(ws), ws_bytes, _stream()),
          "gg_postops_skip_bwd_f32")
    return dy, dres, dgamma, dbeta


# --------------------------------------------------------------------------------------------
# GAT
# --------------------------------------------------------------------------------------------
def _f32(shape, dev):
    n = 1
    for d in shape:
        n *= d
    return torch.empty(max(n, 1), dtype=torch.float32, device=dev)[:n].view(*shape)


GAT_ALGO = _os.environ.get("GG_GAT_ALGO", "auto")   # auto | sell (fused, sliced ELL) | mp (split passes, merge-path) | row
GAT_BWD = _os.environ.get("GG_GAT_BWD", "one")      # fused backward: one (single CSC pass) | two (edge pass + source pass)


def _gat_use_sell(csr, f, heads):
    if heads != 1 or f % 4 != 0 or f > 128 or GAT_ALGO in ("row", "mp"):
        return False
    return GAT_ALGO == "sell" or csr.num_nodes + csr.num_slots >= 1 << 14


def gat_sell_forward(csr, h, ldh, a_tgt, a_src, slope, bias, need_grad=False):
    """-> (out, rowstat [n, 2] = per-row (max, sum of exp), pos); alpha is never materialised (csrc/gat_sell.cu).
    ``pos`` = (out_pos [n, f], a_pos [n]) when ``need_grad`` (the sums over the positive-logit slots that the one-pass
    backward turns into da_tgt), else None."""
    sl = sell_layout(csr)
    n, f = h.shape
    L = lib()
    out = torch.empty((n, f), dtype=torch.float32, device=h.device)
    rowstat = torch.empty((max(n, 1), 2), dtype=torch.float32, device=h.device)[:n]
    pos = None
    if need_grad and GAT_BWD == "one":
        pos = (torch.empty((n, f), dtype=torch.float32, device=h.device), _f32((n,), h.device))
    ws_bytes = int(L.gg_gat_sell_workspace_bytes(sl.partial_rows, f))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=h.device)
    if bias is not None:
        bias = bias.contiguous()
    check(L.gg_gat_sell_fwd_f32(_ptr(sl.chunk_ptr), sl.chunks, _ptr(sl.idx), _ptr(sl.vdst), _ptr(sl.hub_rows),
                                _ptr(sl.hub_pptr), sl.hubs, sl.partial_rows, _ptr(h), ldh, _ptr(a_tgt), _ptr(a_src), n, f,
                                float(slope), _ptr(bias), _ptr(out), f, _ptr(rowstat), _ptr(pos[0]) if pos else None, f,
                                _ptr(pos[1]) if pos else None, _ptr(ws), ws_bytes, _stream()),
          "gg_gat_sell_fwd_f32")
    return out, rowstat, pos


def _sell_edge_map(csc, csc2csr):
    """CSR slot of the edge behind every entry of the CSC sliced-ELL layout (-1 for padding); built once per layout."""
    sl = sell_layout(csc)
    hit = getattr(sl, "_edge_map", None)
    if hit is None or hit[0] is not csc2csr:
        out = torch.empty(max(sl.total, 4), dtype=torch.int32, device=csc2csr.device)
        check(lib().gg_sell_compose_map(_ptr(sl.slot_of), sl.total, _ptr(csc2csr), _ptr(out), _stream()),
              "gg_sell_compose_map")
        sl._edge_map = hit = (csc2csr, out)
    return hit[1]


def gat_sell_backward(csr, csc, csc2csr, h, att, slope, bias, rowstat, a_tgt, a_src, out, g, pos=None):
    """-> dh [n, f], datt [1, 2c] (heads = 1)."""
    h, ldh = _rows(h, "h")
    g, ldg = _rows(g, "g")
    out, ldo = _rows(out, "out")
    n, f = h.shape
    dev = h.device
    att = att.contiguous().view(1, 2 * f)
    L = lib()
    s1, s2 = sell_layout(csr), sell_layout(csc)
    if bias is not None:
        bias = bias.contiguous()
    da_tgt, da_src = _f32((n,), dev), _f32((n,), dev)
    ws_bytes = int(L.gg_gat_sell_workspace_bytes(max(s1.partial_rows, s2.partial_rows), f))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    if pos is not None:
        dh = gat_sell_backward_one(s2, h, ldh, g, ldg, out, ldo, bias, pos, a_tgt, a_src, rowstat, att, slope, da_tgt,
                                   da_src, ws, ws_bytes)
        return dh, _gat_att_grad(h, ldh, da_tgt, da_src, n, f)
    dz = _f32((csr.num_slots,), dev)
    check(L.gg_gat_sell_bwd_edge_f32(_ptr(s1.chunk_ptr), s1.chunks, _ptr(s1.idx), _ptr(s1.slot_of), _ptr(s1.vdst),
                                     _ptr(s1.hub_rows), _ptr(s1.hub_pptr), s1.hubs, s1.partial_rows, _ptr(h), ldh, _ptr(g),
                                     ldg, _ptr(out), ldo, _ptr(bias), _ptr(a_tgt), _ptr(a_src), _ptr(rowstat), n, f,
                                     float(slope), _ptr(dz), _ptr(da_tgt), _ptr(ws), ws_bytes, _stream()),
          "gg_gat_sell_bwd_edge_f32")
    emap = _sell_edge_map(csc, csc2csr)
    dh = torch.empty((n, f), dtype=torch.float32, device=dev)
    tstat = torch.empty((max(n, 1), 4), dtype=torch.float32, device=dev)
    att_tgt, att_src = att[0, :f].contiguous(), att[0, f:].contiguous()
    check(L.gg_gat_sell_bwd_src_f32(_ptr(s2.chunk_ptr), s2.chunks, _ptr(s2.idx), _ptr(emap), _ptr(s2.vdst),
                                    _ptr(s2.hub_rows), _ptr(s2.hub_pptr), s2.hubs, s2.partial_rows, _ptr(g), ldg,
                                    _ptr(a_tgt), _ptr(a_src), _ptr(rowstat), _ptr(dz), _ptr(da_tgt), _ptr(att_src),
                                    _ptr(att_tgt), n, f, float(slope), _ptr(dh), f, _ptr(da_src), _ptr(tstat), _ptr(ws),
                                    ws_bytes, _stream()), "gg_gat_sell_bwd_src_f32")
    return dh, _gat_att_grad(h, ldh, da_tgt, da_src, n, f)


def gat_sell_backward_one(s2, h, ldh, g, ldg, out, ldo, bias, pos, a_tgt, a_src, rowstat, att, slope, da_tgt, da_src, ws,
                          ws_bytes):
    """The one-pass backward's launches (per-node record, the walk over the CSC layout, split-row fix-up) -> dh."""
    out_pos, a_pos = pos
    n, f = h.shape
    dh = torch.empty((n, f), dtype=torch.float32, device=h.device)
    tstat = torch.empty((max(n, 1), 4), dtype=torch.float32, device=h.device)
    att_tgt, att_src = att[0, :f].contiguous(), att[0, f:].contiguous()
    check(lib().gg_gat_sell_bwd_one_f32(_ptr(s2.chunk_ptr), s2.chunks, _ptr(s2.idx), _ptr(s2.vdst), _ptr(s2.hub_rows),
                                        _ptr(s2.hub_pptr), s2.hubs, s2.partial_rows, _ptr(h), ldh, _ptr(g), ldg, _ptr(out),
                                        ldo, _ptr(bias), _ptr(out_pos), out_pos.stride(0), _ptr(a_pos), _ptr(a_tgt),
                                        _ptr(a_src), _ptr(rowstat), _ptr(att_src), _ptr(att_tgt), n, f, float(slope),
                                        _ptr(dh), f, _ptr(da_tgt), _ptr(da_src), _ptr(tstat), _ptr(ws), ws_bytes,
                                        _stream()), "gg_gat_sell_bwd_one_f32")
    return dh


def _gat_att_grad(h, ldh, da_tgt, da_src, n, f):
    L = lib()
    datt = torch.empty((1, 2 * f), dtype=torch.float32, device=h.device)
    ws2_bytes = int(L.gg_gat_att_grad_workspace_bytes(n, 1, f))
    ws2 = torch.empty(ws2_bytes, dtype=torch.uint8, device=h.device)
    check(L.gg_gat_att_grad_f32(_ptr(h), ldh, _ptr(da_tgt), _ptr(da_src), n, 1, f, _ptr(datt), _ptr(ws2), ws2_bytes,
                                _stream()), "gg_gat_att_grad_f32")
    return datt


def _gat_use_mp(csr, f, heads):
    if heads != 1 or f % 4 != 0 or f > 1024 or GAT_ALGO == "row":
        return False
    return GAT_ALGO == "mp" or csr.num_nodes + csr.num_slots >= 1 << 14


def gat_forward(csr, h, att, heads, slope, bias, need_grad=False):
    """-> out [n, heads*c], alpha [E', heads], a_tgt, a_src [n, heads], pos (fused path with ``need_grad``: the extra
    record of the one-pass backward, else None; hand it back to gat_backward)."""
    _need_cuda(h, att, bias)
    h, ldh = _rows(h, "h")
    n, f = h.shape
    c = f // heads
    att = att.contiguous().view(heads, 2 * c)
    a_tgt, a_src = _f32((n, heads), h.device), _f32((n, heads), h.device)
    L = lib()
    check(L.gg_gat_scores_f32(_ptr(h), ldh, _ptr(att), n, heads, c, _ptr(a_tgt), _ptr(a_src), _stream()),
          "gg_gat_scores_f32")
    if _gat_use_sell(csr, f, heads) and ldh % 4 == 0:
        out, rowstat, pos = gat_sell_forward(csr, h, ldh, a_tgt, a_src, slope, bias, need_grad)
        return out, rowstat, a_tgt, a_src, pos     # rowstat [n, 2] stands in for alpha [E', 1]
    alpha = _f32((csr.num_slots, heads), h.device)
    if _gat_use_mp(csr, f, heads):
        check(L.gg_gat_alpha_f32(_ptr(csr.rowptr), _ptr(csr.nbr), _ptr(a_tgt), _ptr(a_src), n, float(slope),
                                 _ptr(alpha), _stream()), "gg_gat_alpha_f32")
        out = spmm(csr, h, alpha.view(-1), SUM, None, 0.0, bias)
        return out, alpha, a_tgt, a_src, None
    out = torch.empty((n, f), dtype=torch.float32, device=h.device)
    if bias is not None:
        bias = bias.contiguous()
    check(L.gg_gat_fwd_f32(_ptr(csr.rowptr), _ptr(csr.nbr), _ptr(h), ldh, _ptr(a_tgt), _ptr(a_src), n,
                           heads, c, float(slope), _ptr(bias), _ptr(alpha), _ptr(out), max(f, 1),
                           _stream()), "gg_gat_fwd_f32")
    return out, alpha, a_tgt, a_src, None


def gat_backward(csr, csc, csc2csr, h, att, heads, slope, bias, alpha, a_tgt, a_src, out, g, pos=None):
    """-> dh [n, f], datt [heads, 2c].  ``alpha`` is the per-row (max, sum) record when the forward ran fused; ``pos`` is
    gat_forward's fifth result (None: the fused backward runs as two passes)."""
    if alpha.dim() == 2 and alpha.size(0) == h.size(0) and alpha.size(1) == 2 and _gat_use_sell(csr, h.size(1), heads):
        return gat_sell_backward(csr, csc, csc2csr, h, att, slope, bias, alpha, a_tgt, a_src, out, g, pos)
    h, ldh = _rows(h, "h")
    g, ldg = _rows(g, "g")
    out, ldo = _rows(out, "out")
    n, f = h.shape
    c = f // heads
    att = att.contiguous().view(heads, 2 * c)
    dev = h.device
    dz = _f32((csr.num_slots, heads), dev)
    da_tgt, da_src = _f32((n, heads), dev), _f32((n, heads), dev)
    L = lib()
    if _gat_use_mp(csr, f, heads):
        item_row, item_slot, items = csr.plan
        dalpha = _f32((csr.num_slots,), dev)
        counter = torch.empty(64, dtype=torch.int32, device=dev)
        check(L.gg_gat_sddmm_mp_f32(_ptr(csr.rowptr), _ptr(csr.nbr), _ptr(item_row), _ptr(item_slot), items,
                                    _ptr(h), ldh, _ptr(g), ldg, n, f, _ptr(dalpha), _ptr(counter), _stream()),
              "gg_gat_sddmm_mp_f32")
        check(L.gg_gat_dz_f32(_ptr(csr.rowptr), _ptr(csr.nbr), _ptr(a_tgt), _ptr(a_src), _ptr(alpha), _ptr(dalpha),
                              n, float(slope), _ptr(dz), _ptr(da_tgt), _stream()), "gg_gat_dz_f32")
        alpha_t = _f32((csc.num_slots,), dev)
        check(L.gg_gat_csc_gather_f32(_ptr(csc.rowptr), _ptr(csc2csr), _ptr(alpha), _ptr(dz), n, _ptr(alpha_t),
                                      _ptr(da_src), _stream()), "gg_gat_csc_gather_f32")
        # dH = A_alpha^T g + da_src att_src + da_tgt att_tgt  (att = [a_tgt half | a_src half])
        dh = spmm(csc, g, alpha_t, SUM, None, 0.0, None,
                  rank1=(da_src.view(-1), att[0, c:], da_tgt.view(-1), att[0, :c]))
        datt = torch.empty((heads, 2 * c), dtype=torch.float32, device=dev)
        ws_bytes = int(L.gg_gat_att_grad_workspace_bytes(n, heads, c))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        check(L.gg_gat_att_grad_f32(_ptr(h), ldh, _ptr(da_tgt), _ptr(da_src), n, heads, c, _ptr(datt), _ptr(ws),
                                    ws_bytes, _stream()), "gg_gat_att_grad_f32")
        return dh, datt
    check(L.gg_gat_bwd_edge_f32(_ptr(csr.rowptr), _ptr(csr.nbr), _ptr(h), ldh, _ptr(a_tgt), _ptr(a_src),
                                _ptr(alpha), _ptr(g), ldg, _ptr(out), ldo, _ptr(bias), n, heads, c,
                                float(slope), _ptr(dz), _ptr(da_tgt), _stream()), "gg_gat_bwd_edge_f32")
    dh = torch.empty((n, f), dtype=torch.float32, device=dev)
    check(L.gg_gat_bwd_src_f32(_ptr(csc.rowptr), _ptr(csc.nbr), _ptr(csc2csr), _ptr(alpha), _ptr(dz),
                               _ptr(g), ldg, _ptr(da_tgt), _ptr(att), n, heads, c, _ptr(da_src), _ptr(dh),
                               max(f, 1), _stream()), "gg_gat_bwd_src_f32")
    datt = torch.empty((heads, 2 * c), dtype=torch.float32, device=dev)
    ws_bytes = int(L.gg_gat_att_grad_workspace_bytes(n, heads, c))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    check(L.gg_gat_att_grad_f32(_ptr(h), ldh, _ptr(da_tgt), _ptr(da_src), n, heads, c, _ptr(datt), _ptr(ws),
                                ws_bytes, _stream()), "gg_gat_att_grad_f32")
    return dh, datt


def gat_sddmm_slice(csr, h_slice, g_slice):
    """This rank's share of dalpha over its column slice: [E'] = <g_slice[row(s)], h_slice[nbr[s]]> (f <= 128)."""
    _need_cuda(h_slice, g_slice)
    h_slice, ldh = _rows(h_slice, "h_slice")
    g_slice, ldg = _rows(g_slice, "g_slice")
    n, f = csr.num_nodes, h_slice.size(1)
    item_row, item_slot, items = csr.plan
    dalpha = _f32((csr.num_slots,), h_slice.device)
    counter = torch.empty(64, dtype=torch.int32, device=h_slice.device)
    check(lib().gg_gat_sddmm_mpg_f32(_ptr(csr.rowptr), _ptr(csr.nbr), _ptr(item_row), _ptr(item_slot), items,
                                     _ptr(h_slice), ldh, _ptr(g_slice), ldg, n, f, _ptr(dalpha), _ptr(counter),
                                     _stream()), "gg_gat_sddmm_mpg_f32")
    return dalpha


def sddmm(csr, h, g):
    """z[s] = <g[row(s), :], h[nbr[s], :]> over the layout's slots (merge-path SDDMM, f % 4 == 0, f <= 1024)."""
    _need_cuda(h, g)
    h, ldh = _rows(h, "h")
    g, ldg = _rows(g, "g")
    n, f = csr.num_nodes, h.size(1)
    item_row, item_slot, items = csr.plan
    z = _f32((csr.num_slots,), h.device)
    counter = torch.empty(64, dtype=torch.int32, device=h.device)
    check(lib().gg_gat_sddmm_mp_f32(_ptr(csr.rowptr), _ptr(csr.nbr), _ptr(item_row), _ptr(item_slot), items, _ptr(h), ldh,
                                    _ptr(g), ldg, n, f, _ptr(z), _ptr(counter), _stream()), "gg_gat_sddmm_mp_f32")
    return z


def segment_softmax(csr, z, scale=1.0):
    alpha = _f32((csr.num_slots,), z.device)
    check(lib().gg_segment_softmax_f32(_ptr(csr.rowptr), _ptr(z.contiguous()), csr.num_nodes, float(scale), _ptr(alpha),
                                       _stream()), "gg_segment_softmax_f32")
    return alpha


def segment_softmax_bwd(csr, alpha, dalpha, scale=1.0):
    dz = _f32((csr.num_slots,), alpha.device)
    check(lib().gg_segment_softmax_bwd_f32(_ptr(csr.rowptr), _ptr(alpha), _ptr(dalpha.contiguous()), csr.num_nodes,
                                           float(scale), _ptr(dz), _stream()), "gg_segment_softmax_bwd_f32")
    return dz


# ---- the GAT passes one by one (heads = 1), as the row-partitioned layer composes them ------------------
def gat_scores(h, att_row):
    """a_tgt[i] = <att[:c], h_i>, a_src[i] = <att[c:], h_i> for the rows of ``h``; ``att_row``: [1, 2c]."""
    _need_cuda(h, att_row)
    h, ldh = _rows(h, "h")
    n, c = h.shape
    a_tgt, a_src = _f32((n, 1), h.device), _f32((n, 1), h.device)
    check(lib().gg_gat_scores_f32(_ptr(h), ldh, _ptr(att_row.contiguous()), n, 1, c, _ptr(a_tgt), _ptr(a_src),
                                  _stream()), "gg_gat_scores_f32")
    return a_tgt.view(-1), a_src.view(-1)


def gat_alpha(csr, a_tgt, a_src, slope):
    alpha = _f32((csr.num_slots,), a_tgt.device)
    check(lib().gg_gat_alpha_f32(_ptr(csr.rowptr), _ptr(csr.nbr), _ptr(a_tgt.contiguous()), _ptr(a_src.contiguous()),
                                 csr.num_nodes, float(slope), _ptr(alpha), _stream()), "gg_gat_alpha_f32")
    return alpha


def gat_dz(csr, a_tgt, a_src, alpha, dalpha, slope):
    """-> dz [E'] (gradient of the pre-softmax logits), da_tgt [n]."""
    dev = alpha.device
    dz, da_tgt = _f32((csr.num_slots,), dev), _f32((csr.num_nodes,), dev)
    check(lib().gg_gat_dz_f32(_ptr(csr.rowptr), _ptr(csr.nbr), _ptr(a_tgt), _ptr(a_src), _ptr(alpha), _ptr(dalpha),
                              csr.num_nodes, float(slope), _ptr(dz), _ptr(da_tgt), _stream()), "gg_gat_dz_f32")
    return dz, da_tgt


def gat_csc_gather(csc, csc2csr, alpha, dz):
    """-> alpha in CSC slot order, da_src [n] = per-source sums of dz."""
    dev = alpha.device
    alpha_t, da_src = _f32((csc.num_slots,), dev), _f32((csc.num_nodes,), dev)
    check(lib().gg_gat_csc_gather_f32(_ptr(csc.rowptr), _ptr(csc2csr), _ptr(alpha), _ptr(dz), csc.num_nodes,
                                      _ptr(alpha_t), _ptr(da_src), _stream()), "gg_gat_csc_gather_f32")
    return alpha_t, da_src


def gat_att_grad(h, da_tgt, da_src, heads=1):
    """datt [heads, 2c] = per head [da_tgt^T h | da_src^T h] over the rows of ``h`` (da_* [n, heads])."""
    h, ldh = _rows(h, "h")
    n, f = h.shape
    c = f // heads
    L = lib()
    datt = torch.empty((heads, 2 * c), dtype=torch.float32, device=h.device)
    ws_bytes = int(L.gg_gat_att_grad_workspace_bytes(n, heads, c))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=h.device)
    check(L.gg_gat_att_grad_f32(_ptr(h), ldh, _ptr(da_tgt.contiguous()), _ptr(da_src.contiguous()), n, heads, c, _ptr(datt),
                                _ptr(ws), ws_bytes, _stream()), "gg_gat_att_grad_f32")
    return datt


# ---- per-(slot, head) passes of the multi-head max (csrc/attn_agg.cu) -----------------------------------
def gat_scores_heads(h, att, heads):
    """-> a_tgt, a_src [n, heads] of ``gat_forward`` (``att`` [1, heads, 2c])."""
    _need_cuda(h, att)
    h, ldh = _rows(h, "h")
    n, f = h.shape
    a_tgt, a_src = _f32((n, heads), h.device), _f32((n, heads), h.device)
    check(lib().gg_gat_scores_f32(_ptr(h), ldh, _ptr(att.contiguous()), n, heads, f // heads, _ptr(a_tgt), _ptr(a_src),
                                  _stream()), "gg_gat_scores_f32")
    return a_tgt, a_src


def gat_alpha_heads(csr, a_tgt, a_src, heads, slope):
    alpha = _f32((csr.num_slots, heads), a_tgt.device)
    check(lib().gg_gat_alpha_heads_f32(_ptr(csr.rowptr), _ptr(csr.nbr), _ptr(a_tgt.contiguous()), _ptr(a_src.contiguous()),
                                       csr.num_nodes, int(heads), float(slope), _ptr(alpha), _stream()),
          "gg_gat_alpha_heads_f32")
    return alpha


def gat_dz_heads(csr, a_tgt, a_src, alpha, dalpha, heads, slope):
    """-> dz [E', heads], da_tgt [n, heads]."""
    dev = alpha.device
    dz, da_tgt = _f32((csr.num_slots, heads), dev), _f32((csr.num_nodes, heads), dev)
    check(lib().gg_gat_dz_heads_f32(_ptr(csr.rowptr), _ptr(csr.nbr), _ptr(a_tgt), _ptr(a_src), _ptr(alpha),
                                    _ptr(dalpha.contiguous()), csr.num_nodes, int(heads), float(slope), _ptr(dz),
                                    _ptr(da_tgt), _stream()), "gg_gat_dz_heads_f32")
    return dz, da_tgt


def gat_src_sum_heads(csc, csc2csr, dz, heads):
    """-> da_src [n, heads] = per-source sums of dz."""
    da_src = _f32((csc.num_nodes, heads), dz.device)
    check(lib().gg_gat_src_sum_heads_f32(_ptr(csc.rowptr), _ptr(csc2csr), _ptr(dz), csc.num_nodes, int(heads),
                                         _ptr(da_src), _stream()), "gg_gat_src_sum_heads_f32")
    return da_src
