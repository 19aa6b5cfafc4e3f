"""Per-``edge_index`` graph layout cache (SURVEY §8b "Ownership").

The reference re-runs its COO edits and normalisation on every forward (``cached=False``,
ref: graphgym/contrib/layer/idconv.py:69-87,157-175).  We build CSR (by target, for the forward
aggregation) and CSC (by source, for the backward wrt the features) once per distinct
``edge_index`` tensor and self-loop policy; the cache key is the tensor's identity + version
counter, and each entry keeps its ``edge_index`` alive so the address cannot be recycled.
"""
from collections import OrderedDict

import torch

from . import ops

_CACHE = OrderedDict()
_CACHE_MAX = 16
# A cached layout holds its edge_index, CSR + CSC, weights and the sliced-ELL re-layouts: ~85 bytes per edge, 5 GB for the
# 62 M-edge products graph.  Sixteen of those would be 80 GB of HBM that the caching allocator has to cudaMalloc step by
# step (measured: the e2e leg of bench.py went from 38 to 104 ms per step as the cache filled).  The cache is therefore
# bounded by edges as well: the newest entries whose edge counts sum to at most _CACHE_MAX_EDGES stay (always at least two:
# the step in flight and the one being built by a prefetching loader).
_CACHE_MAX_EDGES = 1 << 27


class GraphLayout:
    def __init__(self, edge_index, num_nodes, policy):
        self.edge_index = edge_index
        self.num_nodes = int(num_nodes)
        self.policy = policy
        self._csr = None
        self._csc = None
        self._weights = {}
        self._csc2csr = None

    # ---- topology ------------------------------------------------------------------------
    @property
    def csr(self):
        """Grouped by target (edge_index[1]): the rows the forward aggregation reduces over."""
        if self._csr is None:
            self._csr = ops.layout_build(self.edge_index, self.num_nodes, self.policy, ops.BY_TARGET)
        return self._csr

    @property
    def csc(self):
        """Grouped by source (edge_index[0]): the transposed graph, used by the backward."""
        if self._csc is None:
            self._csc = ops.layout_build(self.edge_index, self.num_nodes, self.policy, ops.BY_SOURCE)
        return self._csc

    @property
    def num_slots(self):
        return self.csr.num_slots

    @property
    def csc2csr(self):
        if self._csc2csr is None:
            self._csc2csr = ops.slot_map(self.csr, self.csc)
        return self._csc2csr

    # ---- per-slot weights ----------------------------------------------------------------
    def weights(self, kind):
        """(w_csr, w_csc) for an aggregation kind:
        'sum'      no weights
        'mean'     forward divides in the kernel; backward weight = 1/indeg(target)
        'gcn_src'  D^-1/2 A D^-1/2 with the degree summed over edge_index[0] (ref: idconv.py:143-148)
        'gcn_tgt'  same with the degree summed over edge_index[1] (PyG >= 1.6 GCNConv, layer.py:138)
        'gcn_src_mean'  'gcn_src' weights reduced with a mean over the target's in-edges
        'max'      no weights, max over the in-edges (functional._AggregateMax)
        'gcn_src_max'   'gcn_src' weights, max over the target's normalised messages
        """
        if kind not in self._weights:
            if kind in ("sum", "max"):
                w = (None, None)
            elif kind == "mean":
                indeg = ops.segment_degree(self.csr)
                w = (None, ops.mean_weights(self.csc, indeg))
            elif kind in ("gcn_src", "gcn_tgt"):
                deg = ops.segment_degree(self.csc if kind == "gcn_src" else self.csr)
                w = (ops.gcn_norm(self.csr, deg), ops.gcn_norm(self.csc, deg))
            elif kind == "gcn_src_mean":
                # MessagePassing(aggr='mean') over the normalised messages (ref: idconv.py:19,89-92 with
                # cfg.gnn.agg = 'mean' and normalize_adj): forward = mean_i(w_e h_j); backward weight = w_e / indeg(target).
                # One elementwise product per layout (layout-build level, cached).
                w_csr, w_csc = self.weights("gcn_src")
                w = (w_csr, w_csc * ops.mean_weights(self.csc, ops.segment_degree(self.csr)))
            elif kind == "gcn_src_max":
                # MessagePassing(aggr='max') over the normalised messages: the backward scales by the same w_e
                w = self.weights("gcn_src")
            else:
                raise KeyError(kind)
            self._weights[kind] = w
        return self._weights[kind]


def get_layout(edge_index, num_nodes, policy):
    key = (edge_index.data_ptr(), tuple(edge_index.shape), edge_index._version, int(num_nodes), policy,
           edge_index.device.index)
    hit = _CACHE.get(key)
    if hit is not None and hit.edge_index is edge_index:
        _CACHE.move_to_end(key)
        return hit
    lay = GraphLayout(edge_index, num_nodes, policy)
    _CACHE[key] = lay
    while len(_CACHE) > _CACHE_MAX:
        _CACHE.popitem(last=False)
    while len(_CACHE) > 2 and sum(int(v.edge_index.size(1)) for v in _CACHE.values()) > _CACHE_MAX_EDGES:
        _CACHE.popitem(last=False)
    return lay


def clear_cache():
    _CACHE.clear()


class IdIndex:
    """``node_id_index`` with its per-row multiplicity (index_add_ semantics, ref: idconv.py:67)."""
    __slots__ = ("ids", "count", "num_nodes")

    def __init__(self, ids, num_nodes):
        self.ids = ids.contiguous().long()
        self.num_nodes = int(num_nodes)
        self.count = ops.id_count(self.ids, self.num_nodes)


_ID_CACHE = OrderedDict()


def get_id_index(ids, num_nodes):
    key = (ids.data_ptr(), tuple(ids.shape), ids._version, int(num_nodes), ids.device.index)
    hit = _ID_CACHE.get(key)
    if hit is not None and hit[0] is ids:
        _ID_CACHE.move_to_end(key)
        return hit[1]
    info = IdIndex(ids, num_nodes)
    _ID_CACHE[key] = (ids, info)
    while len(_ID_CACHE) > _CACHE_MAX:
        _ID_CACHE.popitem(last=False)
    return info
