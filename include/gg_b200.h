/*
 * gg_b200.h — C-ABI of the B200-native GraphGym message-passing hot path.
 *
 * This is the drop-in boundary: everything the reference's layer code obtains from
 * torch_geometric / torch_scatter / tf_geometric on the hot path is served by the
 * entry points below (plain pointers and sizes, no torch types). The Python host
 * side (graphgym_b200/) binds them with ctypes and keeps the reference's own layer
 * API (`register_layer` / `layer_dict`, `forward(batch)`) on top.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the parameter name ends in `_host`;
 *   - matrices are row-major fp32 with an explicit leading dimension (in elements);
 *   - graph indices are int32 on the device (N, E' < 2^31); the COO input is the
 *     reference's int64 `edge_index[2,E]` (row 0 = source j, row 1 = target i,
 *     PyG `source_to_target` flow, graphgym/contrib/layer/idconv.py:177);
 *   - `stream` is a `cudaStream_t` (passed as void* so C callers need no CUDA headers);
 *   - return value 0 = OK, negative = gg_status; `gg_last_error()` returns the
 *     thread-local message of the last failure; no exceptions cross the boundary;
 *   - the caller allocates all outputs and workspaces (`*_workspace_bytes` queries);
 *   - nothing here runs on the CPU: there is no fallback path.
 *
 * Citations `ref:` are relative to the reference repository root (JBanks/GraphGym).
 */
#ifndef GG_B200_H
#define GG_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default) /* the library is built with -fvisibility=hidden */
#endif

typedef void* gg_stream_t;

enum gg_status {
    GG_OK = 0,
    GG_ERR_INVALID = -1,   /* bad argument (null pointer, negative size, misaligned row) */
    GG_ERR_CUDA = -2,      /* a CUDA runtime call or launch failed                        */
    GG_ERR_WORKSPACE = -3, /* workspace too small                                          */
    GG_ERR_UNSUPPORTED = -4
};

int gg_version(void);
const char* gg_last_error(void);
/* Number of kernels this library has launched in this process (all threads). */
int64_t gg_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * Graph layout (SURVEY §8a rows 1-2).  The reference keeps COO and edits it with PyG helpers on
 * every forward; we build CSR (grouped by target) / CSC (grouped by source) once per edge_index.
 *
 * Self-loop policy = the PyG helper the reference layer calls before propagate:
 *   KEEP           nothing                                   (SAGEConv, GeneralIDConv w/o norm)
 *   ADD_REMAINING  add_remaining_self_loops                  ref: idconv.py:52-53,140-141,232-233, identity.py:14-15
 *   REMOVE_ADD     remove_self_loops + add_self_loops        ref: idconv.py:302-304 (GAT)
 *   REMOVE         remove_self_loops                         ref: idconv.py:370 (GIN-ID)
 *   ADD            add_self_loops / tfg add_self_loop_edge   ref: sparse_adj.py:58-63, TfgIDLayer.py:298
 * The edited edge list is: kept original edges in their original order, then one (i,i) per node
 * i = 0..N-1 (policies that add).  The layout is the STABLE counting sort of that list by the
 * group key (ties keep list order; duplicates are kept; nothing is coalesced).
 *
 * Outputs (caller-allocated; cap = gg_layout_capacity(E, N, policy)):
 *   rowptr[N+1]  segment offsets; rowptr[N] = E' (number of slots actually used)
 *   nbr[cap]     the other endpoint of each slot (source if grouped by target, and vice versa)
 *   perm[cap]    id of the slot's edge: e in [0,E) = original column of edge_index,
 *                E + i = the appended self loop of node i
 *   rowid[cap]   group key of each slot (nullable)
 * ------------------------------------------------------------------------------------------ */
enum gg_loop_policy {
    GG_LOOPS_KEEP = 0,
    GG_LOOPS_ADD_REMAINING = 1,
    GG_LOOPS_REMOVE_ADD = 2,
    GG_LOOPS_REMOVE = 3,
    GG_LOOPS_ADD = 4
};
enum gg_group_by { GG_BY_TARGET = 0, GG_BY_SOURCE = 1 };

int64_t gg_layout_capacity(int64_t num_edges, int64_t num_nodes, int policy);
size_t gg_layout_build_workspace_bytes(int64_t num_edges, int64_t num_nodes, int policy);
int gg_layout_build(const int64_t* edge_index, int64_t num_edges, int64_t num_nodes, int policy,
                    int group_by, int32_t* rowptr, int32_t* nbr, int32_t* perm, int32_t* rowid,
                    void* workspace, size_t workspace_bytes, gg_stream_t stream);

/* Row-partitioned variant (SURVEY §8e): only the groups in [range_begin, range_end) are kept (edges of
 * other groups and appended loops of other nodes are dropped); rowptr still has N+1 entries, so
 * rowptr + range_begin is the rank-local row pointer and nbr holds GLOBAL node ids.
 * [nbr_begin, nbr_end) additionally keeps only the slots whose neighbour lies in that block (one peer's
 * rows): the per-peer sub-layouts of the pipelined halo exchange.  Pass 0, num_nodes for no filter. */
int gg_layout_build_range(const int64_t* edge_index, int64_t num_edges, int64_t num_nodes, int policy,
                          int group_by, int64_t range_begin, int64_t range_end, int64_t nbr_begin,
                          int64_t nbr_end, int32_t* rowptr, int32_t* nbr, int32_t* perm, int32_t* rowid,
                          void* workspace, size_t workspace_bytes, gg_stream_t stream);

/* Stable LSD radix sort of (key,value) u32 pairs on keys < 2^key_bits (the engine under
 * gg_layout_build, exported for the ego-net and halo code). */
size_t gg_sort_pairs_workspace_bytes(int64_t n);
int gg_sort_pairs_u32(const uint32_t* keys_in, const uint32_t* vals_in, uint32_t* keys_out,
                      uint32_t* vals_out, int64_t n, int key_bits, void* workspace,
                      size_t workspace_bytes, gg_stream_t stream);

/* inv[perm_a[s]] = s, then map[t] = inv[perm_b[t]]: slot of layout A holding the same edge as slot t
 * of layout B (CSC slot -> CSR slot).  `scratch` holds num_edges + num_nodes int32. */
int gg_layout_slot_map(const int32_t* perm_a, const int32_t* perm_b, int64_t num_slots,
                       int64_t num_edges, int64_t num_nodes, int32_t* scratch, int32_t* map,
                       gg_stream_t stream);

/* Per-slot edge weights of the edited list: w_slot[s] = w_edge[perm[s]] for original edges (1 when
 * w_edge is null), `loop_fill` for appended loops; with ADD_REMAINING and w_edge given, an appended
 * loop inherits the weight of the LAST removed (i,i) edge (PyG add_remaining_self_loops).
 * `edge_index` may be null when w_edge is null. */
int gg_layout_slot_weights(const int32_t* perm, int64_t num_slots, const int64_t* edge_index,
                           const float* w_edge, int64_t num_edges, int64_t num_nodes, int policy,
                           float loop_fill, int32_t* scratch_nodes, float* w_slot,
                           gg_stream_t stream);

/* Weighted degree per group: deg[i] = sum_{s in segment i} w_slot[s] (w_slot null => segment length),
 * summed in slot order (deterministic).  ref: scatter_add(edge_weight,row) idconv.py:56,144;
 * SparseAdj.reduce_sum sparse_adj.py:84-85. */
int gg_segment_degree(const int32_t* rowptr, const float* w_slot, int64_t num_nodes, float* deg,
                      gg_stream_t stream);

/* Symmetric GCN normalisation per slot: w_out[s] = dis[rowid[s]] * w_in[s] * dis[nbr[s]],
 * dis = deg^-1/2 with inf -> 0.  `deg` is the degree the reference uses: summed over
 * edge_index[0] (source) in idconv.py:143-148 / identity.py:17-22, over the target in PyG>=1.6
 * GCNConv (layer.py:138); the caller passes whichever applies.  w_in null => 1. */
int gg_gcn_norm(const int32_t* rowid, const int32_t* nbr, const float* w_in, const float* deg,
                int64_t num_slots, float* w_out, gg_stream_t stream);

/* Transposed weights of a mean aggregation: w_out[s] = 1/deg[nbr[s]] (0 when deg is 0); with the
 * CSC layout and deg = in-degree this is d(mean_i)/d(x_j) per slot (ref: aggr='mean', idconv.py:195). */
int gg_mean_weights(const int32_t* nbr, const float* deg, int64_t num_slots, float* w_out,
                    gg_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Aggregation (SURVEY §8a row 4):  out[i,:] = epi( sum_{s in segment i} w[s] * x[nbr[s],:] )
 *   ref: MessagePassing.propagate + message idconv.py:89-92,177-180,235-239,371,378-379;
 *        SparseAdj.matmul sparse_adj.py:91-97.
 *   reduce: 0 = sum, 1 = mean (divide by segment length; empty segment -> 0).
 *   epilogue: out = agg + self_scale * x_self[i,:] (x_self nullable; GIN's (1+eps)*x, idconv.py:371)
 *                       + bias[:] (nullable).
 * The backward wrt x is the same call on the transposed layout (CSC) with the transposed weights.
 * Rows of x / out / x_self must be 16-byte aligned when f % 4 == 0 (vector path); any f works.
 * ------------------------------------------------------------------------------------------ */
enum gg_reduce { GG_SUM = 0, GG_MEAN = 1 };
int gg_spmm_f32(const int32_t* rowptr, const int32_t* nbr, const float* w_slot, const float* x,
                int64_t ldx, float* out, int64_t ldo, int64_t num_rows, int64_t f, int reduce,
                const float* x_self, int64_t ld_self, float self_scale, const float* bias,
                gg_stream_t stream);

/* Load-balanced variant for large / skewed graphs (merge-path over slots + row markers, persistent
 * warps, neighbour-index tiles staged in shared memory by TMA bulk copies; see csrc/spmm_mp.cu).
 * The plan depends only on rowptr and is built once per layout:
 *   units  = gg_spmm_plan_units(N, E')                  merged units (slots + rows) per work item
 *   items  = gg_spmm_plan_items(N, E', units)
 *   gg_spmm_plan_build -> item_row[items+1], item_slot[items+1]
 * gg_spmm_mp_f32 has the semantics of gg_spmm_f32; it needs f % 4 == 0, f <= 1024, 16-byte aligned rows
 * (GG_ERR_UNSUPPORTED otherwise) and a workspace of gg_spmm_mp_workspace_bytes(items, f).
 * stage_mode: bit 0 = plain loads instead of cp.async.bulk staging, bit 1 = deep (16-wide) gather batches,
 * bit 2 = L2 residency hints (feature-row gathers evict_last; index / weight / output streams evict_first).
 * Same fixed summation order per row in every mode.
 * Optional rank-1 epilogue terms (nullable): out[row,:] += r1_s[row]*r1_v[:] + r2_s[row]*r2_v[:]. */
int gg_spmm_plan_units(int64_t num_rows, int64_t num_slots);
int64_t gg_spmm_plan_items(int64_t num_rows, int64_t num_slots, int units);
int gg_spmm_plan_build(const int32_t* rowptr, int64_t num_rows, int64_t num_slots, int units,
                       int32_t* item_row, int32_t* item_slot, gg_stream_t stream);
size_t gg_spmm_mp_workspace_bytes(int64_t items, int64_t f);
int gg_spmm_mp_f32(const int32_t* rowptr, const int32_t* nbr, const float* w_slot,
                   const int32_t* item_row, const int32_t* item_slot, int64_t items, const float* x,
                   int64_t ldx, float* out, int64_t ldo, int64_t num_rows, int64_t f, int reduce,
                   const float* x_self, int64_t ld_self, float self_scale, const float* bias,
                   const float* r1_s, const float* r1_v, const float* r2_s, const float* r2_v,
                   void* workspace, size_t workspace_bytes, int stage_mode, gg_stream_t stream);

/* Narrow-row variant (f % 4 == 0, f <= 128): the warp's 32 lanes are cut into 32/G groups of
 * G = gg_spmm_group_lanes(f) lanes and one warp instruction gathers 32/G different slots of the warp's
 * item; partial sums are combined across the groups at every row end with a fixed shuffle butterfly.
 * Uses the same plan as gg_spmm_mp_f32; same semantics; the summation order per row is fixed (but is
 * not the order of gg_spmm_mp_f32).
 *
 * Peer output (row-partitioned path, SURVEY §8e; `out_peers_host` non-null, `out` ignored): this rank
 * aggregates ITS column slice for all `num_rows` global rows and stores row i into the memory of the
 * rank that owns it: out_peers_host[i / rows_per_rank] + (i % rows_per_rank) * ldo — HOST array of
 * `world` DEVICE pointers (peer memory from gg_peer_open, already offset to this rank's columns).  The
 * stores are plain global stores over NVLink: aggregation and the return leg of the exchange are ONE
 * kernel.  The caller orders it against the peers with gg_peer_barrier.  flags: bit 2 = L2 residency
 * hints as in gg_spmm_mp_f32.  r1_s/r1_v, r2_s/r2_v: the optional rank-1 epilogue terms of gg_spmm_mp_f32
 * (scalars indexed by the global row, vectors already offset to this call's columns). */
int gg_spmm_group_lanes(int64_t f);
int gg_spmm_mpg_f32(const int32_t* rowptr, const int32_t* nbr, const float* w_slot, const int32_t* item_row,
                    const int32_t* item_slot, int64_t items, const float* x, int64_t ldx, float* out,
                    int64_t ldo, float* const* out_peers_host, int world, int64_t rows_per_rank,
                    int64_t num_rows, int64_t f, int reduce, const float* x_self, int64_t ld_self,
                    float self_scale, const float* bias, const float* r1_s, const float* r1_v, const float* r2_s,
                    const float* r2_v, void* workspace, size_t workspace_bytes, int flags, gg_stream_t stream);

/* Degree-sorted sliced-ELL aggregation for narrow rows (csrc/spmm_sell.cu; f % 4 == 0, f <= 128) — same semantics and
 * epilogue as gg_spmm_mpg_f32 (incl. peer output), no row-end work in the kernel.  The layout is rebuilt once per CSR:
 *   rows longer than `seg` slots (multiple of 4, <= 4096) are cut into virtual rows of <= seg slots; virtual rows are
 *   sorted by descending length (stable) and grouped 8 to a chunk, padded to the chunk's longest row rounded up to 4;
 *   neighbour ids are stored as int4 units, (4-slot group k4)-major inside a chunk: idx[(chunk_ptr[c] + k4*8 + q)*4 + kk]
 *   = slot 4*k4+kk of the chunk's row q, -1 for padding; slot_of[] holds the CSR slot of every entry (-1 for padding);
 *   vdst[8*c + q] = output row (>= 0), -(partial row) - 1 for a piece of a split row, INT32_MIN for capacity padding;
 *   hub_rows[h] / hub_pptr[h .. h+1] = the split rows and their ranges of partial rows (summed in order by a fix-up).
 * Capacities (host-side bounds, no sync): vdst gg_sell_vrow_capacity() entries, chunk_ptr that / 8 + 1, idx and slot_of
 * 4 * gg_sell_unit_capacity(), hub_rows gg_sell_split_capacity(), hub_pptr one more.  info[8] (device) receives
 * {virtual rows, chunks, int4 units in use, split rows, partial rows}.  gg_sell_permute_f32 re-lays a per-slot array
 * (weights) in unit order: dst[d] = slot_of[d] >= 0 ? src[slot_of[d]] : 0.  Summation order per row: slot order (one
 * group of lanes per virtual row; split rows: pieces in order) — fixed, not the order of the merge-path kernels. */
int64_t gg_sell_vrow_capacity(int64_t num_rows, int64_t num_slots, int seg);
int64_t gg_sell_unit_capacity(int64_t num_rows, int64_t num_slots, int seg);
int64_t gg_sell_split_capacity(int64_t num_slots, int seg);
size_t gg_sell_build_workspace_bytes(int64_t num_rows, int64_t num_slots, int seg);
int gg_sell_build(const int32_t* rowptr, const int32_t* nbr, int64_t num_rows, int64_t num_slots, int seg,
                  uint32_t* chunk_ptr, int32_t* idx, int32_t* slot_of, int32_t* vdst, int32_t* hub_rows,
                  int32_t* hub_pptr, int32_t* info, void* workspace, size_t workspace_bytes, gg_stream_t stream);
int gg_sell_permute_f32(const int32_t* slot_of, int64_t total, const float* src, float* dst, gg_stream_t stream);
/* Hub hint (caching only, results bitwise unchanged): idx_hint[d] = idx[d] with bit 30 set when the source node is one of
 * the ~`hubs` most referenced nodes of the layout (reference counts from `nbr`; the threshold is the smallest count T with
 * #{count >= T} <= hubs).  gg_spmm_sell_f32 with flags bit 3 set and idx = idx_hint keeps hub rows in L2 (evict_last) and
 * streams the others (evict_first).  Workspace: gg_sell_hub_hint_workspace_bytes(num_nodes). */
size_t gg_sell_hub_hint_workspace_bytes(int64_t num_nodes);
int gg_sell_hub_hint(const int32_t* nbr, int64_t num_slots, int64_t num_nodes, const int32_t* idx, int64_t total,
                     int64_t hubs, int32_t* idx_hint, void* workspace, size_t workspace_bytes, gg_stream_t stream);
size_t gg_spmm_sell_workspace_bytes(int64_t partial_rows, int64_t f);
int gg_spmm_sell_f32(const uint32_t* chunk_ptr, int64_t chunks, const int32_t* idx, const float* w_sell,
                     const int32_t* vdst, const int32_t* rowptr, const int32_t* hub_rows, const int32_t* hub_pptr,
                     int64_t hubs, int64_t partial_rows, const float* x, int64_t ldx, float* out, int64_t ldo,
                     float* const* out_peers_host, int world, int64_t rows_per_rank, int64_t num_rows, int64_t f,
                     int reduce, const float* x_self, int64_t ld_self, float self_scale, const float* bias,
                     const float* r1_s, const float* r1_v, const float* r2_s, const float* r2_v, void* workspace,
                     size_t workspace_bytes, int flags, gg_stream_t stream);

/* Max aggregation (csrc/spmm_max.cu; GraphGym cfg.gnn.agg = 'max'):
 *   out[i,c] = max_{s in segment i} w[s] * x[nbr[s],c] (0 for an empty segment) + self_scale * x_self[i,c] + bias[c]
 *   arg[i,c] = the first slot s (strict `>` in slot order) that reaches the maximum; -1 for an empty segment
 *   dx[j,c]  = sum over the CSC slots t of row j with arg[nbr_csc[t],c] == csr_slot(t) of w_csc[t] * g[nbr_csc[t],c]
 *              + self_scale * g[j,c]
 * gg_spmm_sell_max_f32 runs on the CSR's sliced-ELL layout (gg_sell_build; slot_of as built, w_sell re-laid by
 * gg_sell_permute_f32, flags bits 2 / 3 as in gg_spmm_sell_f32); gg_spmm_sell_max_bwd_f32 on the CSC's, with
 * `edge_map` = gg_sell_compose_map(slot_of of the CSC layout, csc -> csr slot map).  Both need f % 4 == 0 and 16-byte
 * aligned rows (GG_ERR_UNSUPPORTED / GG_ERR_INVALID otherwise); widths above 128 run as column tiles of <= 128.
 * Workspace: gg_spmm_sell_max_workspace_bytes(partial rows of the layout, f).  gg_spmm_row_max_f32 /
 * gg_spmm_row_max_bwd_f32: plain CSR / CSC (+ csc2csr), one warp per row, any f and alignment.  All four are bitwise
 * run-to-run deterministic; the sliced-ELL and row forwards give the same bits. */
size_t gg_spmm_sell_max_workspace_bytes(int64_t partial_rows, int64_t f);
int gg_spmm_sell_max_f32(const uint32_t* chunk_ptr, int64_t chunks, const int32_t* idx, const int32_t* slot_of,
                         const float* w_sell, const int32_t* vdst, const int32_t* hub_rows, const int32_t* hub_pptr,
                         int64_t hubs, int64_t partial_rows, const float* x, int64_t ldx, float* out, int64_t ldo,
                         int32_t* arg, int64_t ld_arg, int64_t num_rows, int64_t f, const float* x_self, int64_t ld_self,
                         float self_scale, const float* bias, void* workspace, size_t workspace_bytes, int flags,
                         gg_stream_t stream);
int gg_spmm_sell_max_bwd_f32(const uint32_t* chunk_ptr, int64_t chunks, const int32_t* idx, const int32_t* edge_map,
                             const float* w_sell, const int32_t* vdst, const int32_t* hub_rows, const int32_t* hub_pptr,
                             int64_t hubs, int64_t partial_rows, const float* g, int64_t ldg, const int32_t* arg,
                             int64_t ld_arg, int64_t num_rows, int64_t f, float self_scale, float* dx, int64_t ldd,
                             void* workspace, size_t workspace_bytes, int flags, gg_stream_t stream);
int gg_spmm_row_max_f32(const int32_t* rowptr, const int32_t* nbr, const float* w_slot, const float* x, int64_t ldx,
                        float* out, int64_t ldo, int32_t* arg, int64_t ld_arg, int64_t num_rows, int64_t f,
                        const float* x_self, int64_t ld_self, float self_scale, const float* bias, gg_stream_t stream);
int gg_spmm_row_max_bwd_f32(const int32_t* rowptr, const int32_t* nbr, const int32_t* csc2csr, const float* w_slot,
                            const float* g, int64_t ldg, const int32_t* arg, int64_t ld_arg, int64_t num_rows, int64_t f,
                            float self_scale, float* dx, int64_t ldd, gg_stream_t stream);

/* Edge-feature message passing (csrc/edge_agg.cu; generaledgeconv / generalsampleedgeconv).  The message on edge
 * e = (j -> i), CSR slot s, perm[s] = e, is h_j[j] (+ h_i[i]) + a[e] W_a^T, a the [E, kd] edge features, W_a [f, kd].
 *   gg_edge_row_reduce_f32    out[i,k] = sum over the slots s of row i of a[perm[s],k], in slot order; / indeg(i) with
 *                             `mean` (rows without slots 0)
 *   gg_edge_rows_self_f32     out[i,c] = y[i,c] + r_i h[i,c] + z[i,c] (y, h, z nullable: 0), r_i = indeg(i) or, with
 *                             `mean`, [indeg(i) > 0]; element-wise, out may alias y
 *   gg_max_mask_f32           out[i,c] = arg[i,c] >= 0 ? g[i,c] : 0
 *   gg_edge_max_sell_f32 / gg_edge_max_row_f32
 *                             out[i,c] = max over the slots s of row i of h_j[nbr[s],c] + sum_k a[perm[s],k] W_a[c,k],
 *                             + h_i[i,c] (nullable), 0 for a row without slots; + self_scale x_self[i,c] + bias[c];
 *                             arg[i,c] = the first slot reaching the maximum (strict `>` in slot order, -1 for an empty
 *                             row).  The sliced-ELL entry takes the CSR's gg_sell_build layout (flags bit 2 as in
 *                             gg_spmm_sell_f32), f % 4 == 0, 16-byte aligned rows, workspace
 *                             gg_spmm_sell_max_workspace_bytes(partial rows, f); the row entry takes the plain CSR and any
 *                             f.  Both need kd <= 256 (GG_ERR_UNSUPPORTED) and give the same bits.
 *   gg_edge_max_winner_f32    da[perm[s],k] = sum over the columns c with arg[i,c] == s (s a slot of row i) of
 *                             g[i,c] W_a[c,k], in column order; 0 for an edge that won no column.  Every edge of the
 *                             layout is written once.
 *   gg_edge_max_wgrad_f32     dw[c,k] = sum_i g[i,c] a[perm[arg[i,c]],k] over the rows with arg >= 0; per-block partials
 *                             summed in a fixed order.  Workspace: gg_edge_max_wgrad_workspace_bytes(num_rows, f, kd).
 * All are bitwise run-to-run deterministic (no atomics on data). */
int gg_edge_row_reduce_f32(const int32_t* rowptr, const int32_t* perm, int64_t num_rows, const float* a, int64_t lda,
                           int64_t k, int mean, float* out, int64_t ldo, gg_stream_t stream);
int gg_edge_rows_self_f32(const int32_t* rowptr, int64_t num_rows, int64_t f, int mean, const float* y, int64_t ldy,
                          const float* h, int64_t ldh, const float* z, int64_t ldz, float* out, int64_t ldo,
                          gg_stream_t stream);
int gg_max_mask_f32(const float* g, int64_t ldg, const int32_t* arg, int64_t ld_arg, int64_t num_rows, int64_t f,
                    float* out, int64_t ldo, gg_stream_t stream);
int gg_edge_max_sell_f32(const uint32_t* chunk_ptr, int64_t chunks, const int32_t* idx, const int32_t* slot_of,
                         const int32_t* perm, const int32_t* vdst, const int32_t* hub_rows, const int32_t* hub_pptr,
                         int64_t hubs, int64_t partial_rows, const float* h_j, int64_t ldj, const float* h_i, int64_t ldi,
                         const float* a, int64_t lda, int64_t kd, const float* w_a, int64_t ldw, float* out, int64_t ldo,
                         int32_t* arg, int64_t ld_arg, int64_t num_rows, int64_t f, const float* x_self, int64_t ld_self,
                         float self_scale, const float* bias, void* workspace, size_t workspace_bytes, int flags,
                         gg_stream_t stream);
int gg_edge_max_row_f32(const int32_t* rowptr, const int32_t* nbr, const int32_t* perm, const float* h_j, int64_t ldj,
                        const float* h_i, int64_t ldi, const float* a, int64_t lda, int64_t kd, const float* w_a,
                        int64_t ldw, float* out, int64_t ldo, int32_t* arg, int64_t ld_arg, int64_t num_rows, int64_t f,
                        const float* x_self, int64_t ld_self, float self_scale, const float* bias, gg_stream_t stream);
int gg_edge_max_winner_f32(const int32_t* rowptr, const int32_t* perm, const int32_t* arg, int64_t ld_arg, const float* g,
                           int64_t ldg, const float* w_a, int64_t ldw, int64_t num_rows, int64_t f, int64_t kd, float* da,
                           int64_t ldda, gg_stream_t stream);
size_t gg_edge_max_wgrad_workspace_bytes(int64_t num_rows, int64_t f, int64_t kd);
int gg_edge_max_wgrad_f32(const int32_t* perm, const int32_t* arg, int64_t ld_arg, const float* g, int64_t ldg,
                          const float* a, int64_t lda, int64_t num_rows, int64_t f, int64_t kd, float* dw, int64_t lddw,
                          void* workspace, size_t workspace_bytes, gg_stream_t stream);

/* B-spline weighted mean aggregation (csrc/spline_agg.cu; splineconv, degree 1, kernel size 2, open spline).  Slot s of
 * row i gathers row nbr[s]; its edge perm[s] has pseudo-coordinate u[perm[s]], t = trunc(u), fr = u - floor(u), and the
 * coefficients c[t & 1] = 1 - fr, c[(t & 1) ^ 1] = fr (t & 1: the non-negative t mod 2).  w_s = w_slot[s] (nullable: 1);
 * `mean` divides row i by its slot count (rows without slots: 0 + the epilogue terms).
 *   gg_spline_spread_*_f32    out[i, 0:f] = sum_s w_s c0 x[nbr[s], :], out[i, f:2f] = sum_s w_s c1 x[nbr[s], :]
 *   gg_spline_blend_*_f32     out[i, :] = sum_s w_s (c0 y[nbr[s], 0:f] + c1 y[nbr[s], f:2f]) + res[i, :] + bias
 *                             (res, bias nullable)
 *                             Slot order per row.  The sliced-ELL entries take the layout's gg_sell_build arrays (slot_of
 *                             gives the slot of every entry, w_sell the weights re-laid by gg_sell_permute_f32, flags bit 2
 *                             as in gg_spmm_sell_f32), f % 4 == 0 (GG_ERR_UNSUPPORTED otherwise), 16-byte aligned rows,
 *                             workspace gg_spmm_sell_max_workspace_bytes(partial rows, f); the row entries take the plain
 *                             layout and any f.
 *   gg_spline_du_f32          du[perm[s]] = (dc[(t+1) & 1] - dc[t & 1]) / indeg(i) for every slot s of row i, with
 *                             dc_k = sum_{c < f} a[i, k a_half + c] b[nbr[s], k b_half + c] (a_half / b_half = 0: one
 *                             operand for both k).  One warp per row, fixed reduction order.
 * All are bitwise run-to-run deterministic (no atomics on data). */
int gg_spline_spread_sell_f32(const uint32_t* chunk_ptr, int64_t chunks, const int32_t* idx, const int32_t* slot_of,
                              const float* w_sell, const int32_t* perm, const float* u, const int32_t* vdst,
                              const int32_t* rowptr, const int32_t* hub_rows, const int32_t* hub_pptr, int64_t hubs,
                              int64_t partial_rows, const float* x, int64_t ldx, float* out, int64_t ldo, int64_t num_rows,
                              int64_t f, int mean, void* workspace, size_t workspace_bytes, int flags, gg_stream_t stream);
int gg_spline_blend_sell_f32(const uint32_t* chunk_ptr, int64_t chunks, const int32_t* idx, const int32_t* slot_of,
                             const float* w_sell, const int32_t* perm, const float* u, const int32_t* vdst,
                             const int32_t* rowptr, const int32_t* hub_rows, const int32_t* hub_pptr, int64_t hubs,
                             int64_t partial_rows, const float* y, int64_t ldy, float* out, int64_t ldo, int64_t num_rows,
                             int64_t f, int mean, const float* res, int64_t ld_res, const float* bias, void* workspace,
                             size_t workspace_bytes, int flags, gg_stream_t stream);
int gg_spline_spread_row_f32(const int32_t* rowptr, const int32_t* nbr, const int32_t* perm, const float* w_slot,
                             const float* u, const float* x, int64_t ldx, float* out, int64_t ldo, int64_t num_rows,
                             int64_t f, int mean, gg_stream_t stream);
int gg_spline_blend_row_f32(const int32_t* rowptr, const int32_t* nbr, const int32_t* perm, const float* w_slot,
                            const float* u, const float* y, int64_t ldy, float* out, int64_t ldo, int64_t num_rows,
                            int64_t f, int mean, const float* res, int64_t ld_res, const float* bias, gg_stream_t stream);
int gg_spline_du_f32(const int32_t* rowptr, const int32_t* nbr, const int32_t* perm, const float* u, const float* a,
                     int64_t lda, int64_t a_half, const float* b, int64_t ldb, int64_t b_half, int64_t num_rows, int64_t f,
                     float* du, gg_stream_t stream);

/* Mean / max aggregation of the attention layers (csrc/attn_agg.cu; gaddconv / gmulconv with cfg.gnn.agg = 'mean' /
 * 'max').  heads H splits f into H blocks of c = f / H columns; column col belongs to head col / c.
 *   gg_max_winner_sddmm_f32   dalpha[s*H + k] = sum over the columns col of head k with arg[i,col] == s (s a slot of CSR
 *                             row i) of g[i,col] * h[nbr[s],col]; 0 for a slot that won nothing.  The gradient of the
 *                             attention weights through the max; bitwise run-to-run deterministic (column order).
 *   gg_gat_alpha_heads_f32    alpha[s*H + k] = softmax over row i of leaky_relu(a_tgt[i*H+k] + a_src[nbr[s]*H+k])
 *                             (max-shifted, denominator + 1e-16), as gg_gat_alpha_f32 per head
 *   gg_gat_dz_heads_f32       gg_gat_dz_f32 per head: dz[s*H+k], da_tgt[i*H+k]
 *   gg_gat_src_sum_heads_f32  da_src[j*H+k] = sum over the CSC slots t of row j of dz[slot_map[t]*H + k]
 *   gg_spmm_row_max_heads_f32 gg_spmm_row_max_f32 with weight w[s*H + col/c] (+ bias), one warp per row
 *   gg_spmm_row_max_heads_bwd_f32  its backward on the CSC layout: w indexed by the CSR slot csc2csr[t]
 *   gg_rows_epilogue_f32      out[i,col] = x[i,col] * (1/indeg(i) if rowptr, indeg = rowptr[i+1] - rowptr[i], rows
 *                             without slots unscaled) + s1[i*H+k] v1[col] + s2[i*H+k] v2[col] (if s1) + bias[col];
 *                             element-wise, out may alias x. */
int gg_max_winner_sddmm_f32(const int32_t* rowptr, const int32_t* nbr, const int32_t* arg, int64_t ld_arg, const float* g,
                            int64_t ldg, const float* h, int64_t ldh, int64_t num_rows, int heads, int64_t f, float* dalpha,
                            gg_stream_t stream);
int gg_gat_alpha_heads_f32(const int32_t* rowptr, const int32_t* nbr, const float* a_tgt, const float* a_src,
                           int64_t num_rows, int heads, float slope, float* alpha, gg_stream_t stream);
int gg_gat_dz_heads_f32(const int32_t* rowptr, const int32_t* nbr, const float* a_tgt, const float* a_src,
                        const float* alpha, const float* dalpha, int64_t num_rows, int heads, float slope, float* dz,
                        float* da_tgt, gg_stream_t stream);
int gg_gat_src_sum_heads_f32(const int32_t* rowptr_t, const int32_t* slot_map, const float* dz, int64_t num_rows,
                             int heads, float* da_src, gg_stream_t stream);
int gg_spmm_row_max_heads_f32(const int32_t* rowptr, const int32_t* nbr, const float* w, int heads, const float* x,
                              int64_t ldx, float* out, int64_t ldo, int32_t* arg, int64_t ld_arg, int64_t num_rows, int64_t f,
                              const float* bias, gg_stream_t stream);
int gg_spmm_row_max_heads_bwd_f32(const int32_t* rowptr, const int32_t* nbr, const int32_t* csc2csr, const float* w,
                                  int heads, const float* g, int64_t ldg, const int32_t* arg, int64_t ld_arg, int64_t num_rows,
                                  int64_t f, float* dx, int64_t ldd, gg_stream_t stream);
int gg_rows_epilogue_f32(const float* x, int64_t ldx, int64_t num_rows, int64_t f, const int32_t* rowptr, int heads,
                         const float* s1, const float* v1, const float* s2, const float* v2, const float* bias, float* out,
                         int64_t ldo, gg_stream_t stream);

/* bf16-gather variant (the north star's 1e-2 mode): x is stored in bf16 (`x_bf16`: raw bf16 bits, ldx in
 * elements, rows 16-byte aligned), products and sums are fp32, out / x_self / bias are fp32.  Same plan and the
 * same fixed summation order as gg_spmm_mpg_f32; needs f % 8 == 0 and f <= 256.  gg_cast_f32_bf16 converts a
 * feature matrix with round-to-nearest-even (f % 4 == 0). */
int gg_cast_f32_bf16(const float* src, int64_t ld, int64_t rows, int64_t f, uint16_t* dst, int64_t ld_dst,
                     gg_stream_t stream);
int gg_spmm_mp_bf16(const int32_t* rowptr, const int32_t* nbr, const float* w_slot, const int32_t* item_row,
                    const int32_t* item_slot, int64_t items, const uint16_t* x_bf16, int64_t ldx, float* out,
                    int64_t ldo, int64_t num_rows, int64_t f, int reduce, const float* x_self, int64_t ld_self,
                    float self_scale, const float* bias, void* workspace, size_t workspace_bytes, int flags,
                    gg_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Dense transform with ID-GNN heterogeneous weights (SURVEY §8a row 9):
 *   out[N,F] = act( sum_g diag(scale_g) * A_g[N,K_g] * B_g  + bias ) (.* mask>0)
 * up to GG_GEMM_MAX_SEGMENTS K-segments accumulate into the same output tile, so
 *   X*W + onehot(id)*(X*W_id)   (ref: idconv.py:64-67,152-155,248-251,307-310,372-375)
 * is ONE pass: segment 0 = (X, W, scale null), segment 1 = (X, W_id, scale = multiplicity of the
 * row in `id`, 0 for non-centres; tiles whose rows all have scale 0 skip the segment).
 *   b_trans = 0: B_g is [K_g, F] row-major;  1: B_g is [F, K_g] row-major (used for dX = dH * W^T).
 * ------------------------------------------------------------------------------------------ */
#define GG_GEMM_MAX_SEGMENTS 4
typedef struct gg_gemm_segment {
    const float* a;     /* [n, k] */
    int64_t lda;
    const float* b;     /* [k, f] or [f, k] if b_trans */
    int64_t ldb;
    const float* scale; /* [n] row multipliers, nullable */
    int64_t k;
} gg_gemm_segment;
enum gg_act { GG_ACT_NONE = 0, GG_ACT_RELU = 1, GG_ACT_LRELU = 2 /* post-ops only */ };
int gg_id_gemm_f32(const gg_gemm_segment* segments_host, int num_segments, int b_trans, int64_t n,
                   int64_t f, const float* bias, int act, const float* relu_mask, int64_t ld_mask,
                   float* out, int64_t ldo, gg_stream_t stream);

/* The same transform on the tensor cores: tcgen05.mma kind::tf32 with a 3xTF32 operand split
 * (hi*hi + hi*lo + lo*hi, fp32 accumulation in TMEM), fp32 in / fp32 out, <= 1e-5 relative against the
 * fp32 reference.  Same arguments as gg_id_gemm_f32 plus a workspace for the pre-split B operand images
 * (gg_id_gemm_tc_workspace_bytes).  See csrc/gemm_tc.cu. */
size_t gg_id_gemm_tc_workspace_bytes(const gg_gemm_segment* segments_host, int num_segments, int64_t f);
int gg_id_gemm_tc_f32(const gg_gemm_segment* segments_host, int num_segments, int b_trans, int64_t n,
                      int64_t f, const float* bias, int act, const float* relu_mask, int64_t ld_mask,
                      float* out, int64_t ldo, void* workspace, size_t workspace_bytes, gg_stream_t stream);

/* Weight gradient: out[K,F] = sum_{r<n} A[row(r),:]^T * G[row(r),:], row(r) = row_index ? row_index[r] : r
 * (dW = X^T dH over all N rows; dW_id = X[id]^T dH[id] over the M centre rows, duplicates counted
 * like index_add_, ref: idconv.py:64-67).  Deterministic two-stage split over rows. */
size_t gg_gemm_tn_workspace_bytes(int64_t n, int64_t k, int64_t f);
int gg_gemm_tn_f32(const float* a, int64_t lda, const int64_t* row_index, const float* g, int64_t ldg,
                   int64_t n, int64_t k, int64_t f, float* out, int64_t ldo, void* workspace,
                   size_t workspace_bytes, gg_stream_t stream);

/* Weight gradient on the tensor cores (tcgen05 3xTF32, 512 rows per TMEM accumulation, fp64 reduction of
 * the per-split partial tiles); same arguments as gg_gemm_tn_f32. */
size_t gg_gemm_tn_tc_workspace_bytes(int64_t n, int64_t k, int64_t f);
int gg_gemm_tn_tc_f32(const float* a, int64_t lda, const int64_t* row_index, const float* g, int64_t ldg,
                      int64_t n, int64_t k, int64_t f, float* out, int64_t ldo, void* workspace,
                      size_t workspace_bytes, gg_stream_t stream);

/* Column sums (bias gradient): out[f] = sum_r g[r,f], fixed-order two-stage reduction.
 * workspace: gg_colsum_workspace_bytes. */
size_t gg_colsum_workspace_bytes(int64_t n, int64_t f);
int gg_colsum_f32(const float* g, int64_t ldg, int64_t n, int64_t f, float* out, void* workspace,
                  size_t workspace_bytes, gg_stream_t stream);

/* centre multiplicity: count[r] = number of occurrences of r in id[0..m) (index_add_ semantics:
 * duplicates add twice, idconv.py:67). count must hold n floats. */
int gg_id_count(const int64_t* id, int64_t m, int64_t n, float* count, gg_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * GAT: edge-softmax fused into the aggregation (SURVEY §8a row 8).
 *   ref: GATIDConvLayer.message/update idconv.py:317-342 (same math as pyg.nn.GATConv, layer.py:158);
 *        PyG softmax(alpha, edge_index_i) idconv.py:327; SparseAdj.softmax sparse_adj.py:136-151.
 * h is the transformed feature matrix [n, heads*c]; att is the reference's [1, heads, 2c] parameter
 * (first c = target half a_i, last c = source half a_j).  Needs c % 4 == 0, heads <= 8, heads*c <= 1024.
 *   scores   a_tgt[n,heads], a_src[n,heads]: per-node halves of the logit (z_e = a_tgt[i] + a_src[j])
 *   fwd      alpha[E',heads] = softmax_i(leaky_relu(z)) (max-shifted, denominator + 1e-16), written for
 *            the backward; out[i] = sum_e alpha_e h[j_e] + bias
 *   bwd_edge per target row: dz[E',heads] (gradient of the pre-activation logit), da_tgt[n,heads]
 *   bwd_src  on the CSC layout (slot_map = CSC slot -> CSR slot from gg_layout_slot_map):
 *            dh[j] = sum_e alpha_e g[i_e] + da_src[j] att_src + da_tgt[j] att_tgt; da_src[n,heads]
 *   att_grad datt[heads,2c] = [da_tgt^T h | da_src^T h] per head
 * ------------------------------------------------------------------------------------------ */
int gg_gat_scores_f32(const float* h, int64_t ldh, const float* att, int64_t n, int heads, int c,
                      float* a_tgt, float* a_src, gg_stream_t stream);
int gg_gat_fwd_f32(const int32_t* rowptr, const int32_t* nbr, const float* h, int64_t ldh,
                   const float* a_tgt, const float* a_src, int64_t n, int heads, int c, float slope,
                   const float* bias, float* alpha, float* out, int64_t ldo, gg_stream_t stream);
int gg_gat_bwd_edge_f32(const int32_t* rowptr, const int32_t* nbr, const float* h, int64_t ldh,
                        const float* a_tgt, const float* a_src, const float* alpha, const float* g,
                        int64_t ldg, const float* out, int64_t ldo, const float* bias, int64_t n,
                        int heads, int c, float slope, float* dz, float* da_tgt, gg_stream_t stream);
int gg_gat_bwd_src_f32(const int32_t* rowptr_t, const int32_t* nbr_t, const int32_t* slot_map,
                       const float* alpha, const float* dz, const float* g, int64_t ldg,
                       const float* da_tgt, const float* att, int64_t n, int heads, int c,
                       float* da_src, float* dh, int64_t lddh, gg_stream_t stream);
size_t gg_gat_att_grad_workspace_bytes(int64_t n, int heads, int c);
int gg_gat_att_grad_f32(const float* h, int64_t ldh, const float* da_tgt, const float* da_src,
                        int64_t n, int heads, int c, float* datt, void* workspace,
                        size_t workspace_bytes, gg_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * ID-GNN Fast: cycle features diag(A^p), p = 1..k (SURVEY §8a row 10).
 *   ref: compute_identity graphgym/contrib/transform/identity.py:25-35 (dense n x n powers, fp32).
 * One call handles a block of `src_count` consecutive source nodes [src_begin, src_begin+src_count)
 * inside a node range [row_begin, row_end) that is closed under adjacency (a graph, or a run of graphs
 * of a block-diagonal batch); out[b, p-1] = diag(A^p) at node src_begin + b.
 *   f32: A = the per-slot weights w_slot (A_hat from gg_gcn_norm on the ADD_REMAINING layout), up to
 *        128 sources per call; fp32 propagation, fp64 dot accumulation (parity 1e-5 relative);
 *   i64: A = the unweighted layout (duplicate edges counted), up to 64 sources per call, exact unless
 *        a value exceeds int64: then out = INT64_MAX and *overflow_count is incremented (the caller
 *        zeroes it).  The reference has no integer mode (SURVEY D2).
 * symmetric != 0 uses diag(A^2t) = |A^t e_i|^2, diag(A^2t+1) = <A^t e_i, A^(t+1) e_i> (ceil(k/2) hops);
 * symmetric == 0 propagates k hops and reads the diagonal entry.
 * ------------------------------------------------------------------------------------------ */
size_t gg_cycle_diag_workspace_bytes(int64_t num_rows_in_range);
int gg_cycle_diag_f32(const int32_t* rowptr, const int32_t* nbr, const float* w_slot, int64_t row_begin,
                      int64_t row_end, int k, int symmetric, int64_t src_begin, int src_count, float* out,
                      int64_t ld_out, void* workspace, size_t workspace_bytes, gg_stream_t stream);
/* Whole-graph float variant for large skewed graphs: the propagation step runs on the merge-path aggregation
 * kernel (plan of the same layout from gg_spmm_plan_build) instead of one warp per row. */
size_t gg_cycle_diag_mp_workspace_bytes(int64_t num_rows, int64_t items);
int gg_cycle_diag_mp_f32(const int32_t* rowptr, const int32_t* nbr, const float* w_slot, const int32_t* item_row,
                         const int32_t* item_slot, int64_t items, int64_t num_rows, int k, int symmetric,
                         int64_t src_begin, int src_count, float* out, int64_t ld_out, void* workspace,
                         size_t workspace_bytes, gg_stream_t stream);
/* Same as gg_cycle_diag_mp_f32 with the propagation hops on the sliced-ELL aggregation (gg_sell_build layout of the
 * whole graph; `w_sell`: the normalisation weights re-laid by gg_sell_permute_f32). */
size_t gg_cycle_diag_sell_workspace_bytes(int64_t num_rows, int64_t partial_rows);
int gg_cycle_diag_sell_f32(const int32_t* rowptr, const uint32_t* chunk_ptr, int64_t chunks, const int32_t* idx,
                           const float* w_sell, const int32_t* vdst, const int32_t* hub_rows, const int32_t* hub_pptr,
                           int64_t hubs, int64_t partial_rows, int64_t num_rows, int k, int symmetric, int64_t src_begin,
                           int src_count, float* out, int64_t ld_out, void* workspace, size_t workspace_bytes,
                           gg_stream_t stream);
int gg_cycle_diag_i64(const int32_t* rowptr, const int32_t* nbr, int64_t row_begin, int64_t row_end, int k,
                      int symmetric, int64_t src_begin, int src_count, int64_t* out, int64_t ld_out,
                      int32_t* overflow_count, void* workspace, size_t workspace_bytes, gg_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * ID-GNN Full: batched k-hop ego-net extraction (SURVEY §8a row 11).
 *   ref: ego_nets graphgym/models/transform.py:11-38 (nx.ego_graph per centre + dict relabel).
 * Input: the adjacency of a block-diagonal batch of undirected graphs as a layout grouped by source
 * (both directions of every edge present, the DeepSNAP convention), graph_ptr[G+1] node ranges,
 * graph_of[n] graph id per node, max_graph_nodes (bitmap size; <= ~100K).  radius > 4 => whole graph
 * (transform.py:18-19).  Two phases:
 *   sizes: ego_ptr[n+1] / edge_ptr[n+1] (exclusive scans of the non-centre member count and of the
 *          directed induced-edge count per centre) and out_node_ptr[G+1]; the caller reads
 *          out_node_ptr[G] and edge_ptr[n] to allocate;
 *   fill:  orig_id[total_nodes], edge_index_out[2, total_edges].
 * Numbering (per graph g, centres [lo,hi)): centre c -> out_node_ptr[g] + (c-lo) (so node_id_index of a
 * graph is arange(n_g) + out_node_ptr[g], transform.py:38); the j-th non-centre member of ego c, in
 * ascending original id, -> out_node_ptr[g] + n_g + (ego_ptr[c]-ego_ptr[lo]) + j.  Edges: centres in
 * order, members ascending, adjacency slots in order.
 * ------------------------------------------------------------------------------------------ */
size_t gg_egonet_workspace_bytes(int64_t n, int64_t num_graphs);
int gg_egonet_sizes(const int32_t* rowptr, const int32_t* nbr, int64_t n, int radius,
                    const int32_t* graph_ptr, const int32_t* graph_of, int64_t num_graphs,
                    int max_graph_nodes, uint32_t* ego_ptr, uint32_t* edge_ptr, int64_t* out_node_ptr,
                    void* workspace, size_t workspace_bytes, gg_stream_t stream);
int gg_egonet_fill(const int32_t* rowptr, const int32_t* nbr, int64_t n, int radius,
                   const int32_t* graph_ptr, const int32_t* graph_of, int64_t num_graphs,
                   int max_graph_nodes, const uint32_t* ego_ptr, const uint32_t* edge_ptr,
                   const int64_t* out_node_ptr, int64_t total_edges, int64_t* orig_id,
                   int64_t* edge_index_out, gg_stream_t stream);

/* GAT at scale (heads = 1): the same layer split into light per-slot passes and heavy feature-row passes
 * that run on the merge-path kernels (csrc/gat_mp.cu):
 *   forward   gg_gat_alpha_f32 (alpha per slot)  ->  gg_spmm_mp_f32 with w_slot = alpha (+ bias)
 *   backward  gg_gat_sddmm_mp_f32 (dalpha[s] = <g_i, h_j>, merge-path plan of the CSR layout; `counter` is
 *             one int32 of scratch)  ->  gg_gat_dz_f32 (dz, da_tgt)  ->  gg_gat_csc_gather_f32 (alpha in CSC
 *             order, da_src)  ->  gg_spmm_mp_f32 on the CSC layout with the rank-1 terms
 *             da_src*att_src + da_tgt*att_tgt  ->  gg_gat_att_grad_f32. */
int gg_gat_alpha_f32(const int32_t* rowptr, const int32_t* nbr, const float* a_tgt, const float* a_src,
                     int64_t n, float slope, float* alpha, gg_stream_t stream);
int gg_gat_sddmm_mp_f32(const int32_t* rowptr, const int32_t* nbr, const int32_t* item_row,
                        const int32_t* item_slot, int64_t items, const float* h, int64_t ldh, const float* g,
                        int64_t ldg, int64_t n, int64_t f, float* dalpha, int32_t* counter, gg_stream_t stream);
/* Narrow-row SDDMM (f % 4 == 0, f <= 128) for the feature-sliced exchange: this rank's share
 * dalpha[s] = <g[row(s), 0:f], h[nbr[s], 0:f]> over ITS column slice; the ranks' shares are summed by the
 * caller (all-reduce).  Same plan and counter conventions as gg_gat_sddmm_mp_f32. */
int gg_gat_sddmm_mpg_f32(const int32_t* rowptr, const int32_t* nbr, const int32_t* item_row,
                         const int32_t* item_slot, int64_t items, const float* h, int64_t ldh, const float* g,
                         int64_t ldg, int64_t n, int64_t f, float* dalpha, int32_t* counter, gg_stream_t stream);
int gg_gat_dz_f32(const int32_t* rowptr, const int32_t* nbr, const float* a_tgt, const float* a_src,
                  const float* alpha, const float* dalpha, int64_t n, float slope, float* dz, float* da_tgt,
                  gg_stream_t stream);
int gg_gat_csc_gather_f32(const int32_t* rowptr_t, const int32_t* slot_map, const float* alpha, const float* dz,
                          int64_t n, float* alpha_t, float* da_src, gg_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * On-device batch collation (SURVEY §8f item 2; csrc/collate.cu): the block-diagonal concatenation DeepSNAP's
 * Batch.collate() does on the host every iteration (ref: graphgym/loader.py:245-250, graphgym/train.py:21) and the
 * column-wise feature concat of Preprocess (ref: graphgym/models/feature_augment.py:329-333) as segmented copies, one
 * launch per output array.  The segment tables are DEVICE arrays (the caller uploads them, a few hundred bytes).
 *   gg_collate_index_i64: out[dst_offset + k] = (src ? src[k] : 0) + add, k < count  — edge_index rows and
 *     node_id_index with the graph's node offset added, the `batch` vector (src null, add = graph number), labels.
 *   gg_collate_rows_f32:  out[(dst_row + i) * ldo + col_offset + c] = (float) src[i * ld + c], i < rows, c < f — feature
 *     blocks stacked by graph; call once per feature key with that key's column offset.  src_dtype: GG_DTYPE_*.
 * `scratch_ends_dev`: num_segments int64 of device scratch. */
typedef struct gg_index_segment {
    const int64_t* src; /* nullable */
    int64_t count;
    int64_t dst_offset;
    int64_t add;
    int64_t reserved; /* keeps both segment records at 40 bytes: one table can hold either kind */
} gg_index_segment;
typedef struct gg_rows_segment {
    const void* src;
    int64_t ld;   /* elements between consecutive source rows */
    int64_t rows;
    int64_t f;
    int64_t dst_row;
} gg_rows_segment;
enum gg_dtype { GG_DTYPE_F32 = 0, GG_DTYPE_I64 = 1, GG_DTYPE_U8 = 2 };
int gg_collate_index_i64(const gg_index_segment* segments_dev, int num_segments, int64_t total, int64_t* out,
                         int64_t* scratch_ends_dev, gg_stream_t stream);
int gg_collate_rows_f32(const gg_rows_segment* segments_dev, int num_segments, int64_t total_elements, int src_dtype,
                        float* out, int64_t ldo, int64_t col_offset, int64_t* scratch_ends_dev, gg_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Label / feature binning (SURVEY §8f item 4; csrc/binning.cu) — the numpy preprocessing of
 * graphgym/models/feature_augment.py:139-140,219-231 in float64 on the device:
 *   gg_f64_sort_keys: order-preserving 64-bit keys of x split into two u32 words, index[i] = i.  Ascending stable order =
 *     gg_sort_pairs_u32(key_lo, index) then gg_sort_pairs_u32(gg_gather_u32(key_hi, order), order), 32 bits each.
 *   gg_digitize_f64:  out[i] = #{j : bins[j] <= x[i]} - 1 for ascending bins (= np.digitize(x, bins) - 1). */
int gg_f64_sort_keys(const double* x, int64_t n, uint32_t* key_hi, uint32_t* key_lo, uint32_t* index, gg_stream_t stream);
int gg_gather_u32(const uint32_t* src, const uint32_t* index, int64_t n, uint32_t* dst, gg_stream_t stream);
int gg_digitize_f64(const double* x, int64_t n, const double* bins, int num_bins, int64_t* out, gg_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Fused layer post-ops (SURVEY §8f item 1; csrc/postops.cu) — what GeneralLayer / GNNStackStage apply after the
 * message-passing layer (ref: graphgym/models/layer.py:26-46, graphgym/models/gnn.py:76-81):
 *   a = BatchNorm1d(y)   (mean / invstd null: no BN; gamma / beta null: no affine)
 *   r = act(a)           GG_ACT_NONE | GG_ACT_RELU | GG_ACT_LRELU (slope > 0)
 *   out = l2norm ? r / max(||r||_2, 1e-12) : r          (torch.nn.functional.normalize over dim 1)
 * gg_bn_stats_f32: per-column mean and 1/sqrt(biased var + eps) of y in one pass (deterministic), and, when the pointers
 *   are given, BatchNorm1d's running-statistics update running = (1 - momentum) running + momentum * stat (unbiased var).
 * gg_postops_fwd_f32: one pass; rownorm[n] receives max(||r||, 1e-12) when l2norm (kept for the backward).
 * gg_postops_bwd_f32: dy from go, the SAVED out (activation gates = sign of out), y, mean / invstd, rownorm; train != 0:
 *   batch-statistics BN (dy includes the mean / variance terms); dgamma / dbeta are written whenever mean is given.
 * Workspace: gg_postops_workspace_bytes(n, f) for the statistics and for the backward. */
size_t gg_postops_workspace_bytes(int64_t n, int64_t f);
int gg_bn_stats_f32(const float* y, int64_t ld, int64_t n, int64_t f, float eps, float* mean, float* invstd,
                    float* running_mean, float* running_var, float momentum, void* workspace, size_t workspace_bytes,
                    gg_stream_t stream);
int gg_postops_fwd_f32(const float* y, int64_t ld_y, int64_t n, int64_t f, const float* mean, const float* invstd,
                       const float* gamma, const float* beta, int act, float slope, int l2norm, float* out,
                       int64_t ld_out, float* rownorm, gg_stream_t stream);
int gg_postops_bwd_f32(const float* go, int64_t ld_go, const float* out, int64_t ld_out, const float* y, int64_t ld_y,
                       int64_t n, int64_t f, const float* mean, const float* invstd, const float* gamma, int train,
                       int act, float slope, int l2norm, const float* rownorm, float* dy, int64_t ld_dy, float* dgamma,
                       float* dbeta, void* workspace, size_t workspace_bytes, gg_stream_t stream);

/* The skip epilogue of GNNSkipBlock (ref: graphgym/models/gnn.py GNNSkipBlock / GNNSkipStage) on the same kernels: the
 * last layer's BatchNorm, the skip connection, the stage activation and (last block) the stage's L2 in one pass.
 *   GG_SKIP_SUM     (skipsum, p = 0)     out [n, f]      = l2?(act(BN(y) + res)),  res [n, f]
 *   GG_SKIP_PREFIX  (skipconcat, p >= 1) out [n, p + f]  = l2?([act(res) | act(BN(y))]),  res [n, p]; the L2 over p + f
 * gg_postops_skip_bwd_f32: as gg_postops_bwd_f32 (gates from the SAVED out, go / out rows p + f wide in PREFIX mode), and
 *   dres = dA, the gradient at the activation's input: the f columns (SUM) or the p carried columns (PREFIX);
 *   dgamma / dbeta sum over the f columns only.  Statistics: gg_bn_stats_f32 of y; workspace as gg_postops_bwd_f32. */
enum gg_skip { GG_SKIP_NONE = 0, GG_SKIP_SUM = 1, GG_SKIP_PREFIX = 2 };
int gg_postops_skip_fwd_f32(const float* y, int64_t ld_y, const float* res, int64_t ld_res, int64_t n, int64_t f,
                            int64_t p, int mode, const float* mean, const float* invstd, const float* gamma,
                            const float* beta, int act, float slope, int l2norm, float* out, int64_t ld_out,
                            float* rownorm, gg_stream_t stream);
int gg_postops_skip_bwd_f32(const float* go, int64_t ld_go, const float* out, int64_t ld_out, const float* y,
                            int64_t ld_y, int64_t n, int64_t f, int64_t p, int mode, const float* mean,
                            const float* invstd, const float* gamma, int train, int act, float slope, int l2norm,
                            const float* rownorm, float* dy, int64_t ld_dy, float* dres, int64_t ld_dres, float* dgamma,
                            float* dbeta, void* workspace, size_t workspace_bytes, gg_stream_t stream);

/* Per-row softmax over GIVEN per-slot logits and its backward — the scaled dot-product scorer of the Tfg GAT variant
 * (ref: TfgIDLayer.py:336-345, sparse_adj.py:136-151): alpha[s] = exp(scale z[s] - max_row) / sum_row;
 * dz[s] = scale alpha[s] (dalpha[s] - sum_row alpha dalpha).  The logits come from gg_gat_sddmm_mp_f32 (<Q_i, K_j>). */
int gg_segment_softmax_f32(const int32_t* rowptr, const float* z, int64_t n, float scale, float* alpha,
                           gg_stream_t stream);
int gg_segment_softmax_bwd_f32(const int32_t* rowptr, const float* alpha, const float* dalpha, int64_t n, float scale,
                               float* dz, gg_stream_t stream);

/* GAT (heads = 1) fused into the sliced-ELL aggregation (csrc/gat_sell.cu): alpha never touches memory.
 *   gg_gat_sell_fwd_f32       CSR sliced-ELL layout (gg_sell_build): logits leaky_relu(a_tgt[i] + a_src[j]), online softmax
 *                             fused with out[i] = sum_j alpha_ij h_j (+ bias); rowstat[2 i .. 2 i + 1] = (max, sum of exp);
 *                             out_pos / a_pos (both or neither; training only): the same sums over the slots whose logit
 *                             is positive, consumed by gg_gat_sell_bwd_one_f32
 *   gg_gat_sell_bwd_edge_f32  same layout: dalpha = <g_i, h_j>, alpha recomputed from rowstat, D_i = <g_i, out_i - bias>;
 *                             writes dz[CSR slot] (gradient of the pre-activation logits) and da_tgt[i] = sum_e dz_e
 *   gg_gat_sell_bwd_src_f32   CSC sliced-ELL layout + `edge_map` (gg_sell_compose_map(slot_of_csc, csc->csr slot map)):
 *                             dh[j] = sum_i alpha_ij g_i + da_src[j] att_src + da_tgt[j] att_tgt, da_src[j] = sum_e dz_e;
 *                             `tstat_scratch`: 4 n floats of scratch (per-target record a_tgt, max, 1/(sum + 1e-16))
 * f % 4 == 0, f <= 128; workspace gg_gat_sell_workspace_bytes(partial rows of the layout, f). */
size_t gg_gat_sell_workspace_bytes(int64_t partial_rows, int64_t f);
int gg_sell_compose_map(const int32_t* slot_of, int64_t total, const int32_t* map, int32_t* out, gg_stream_t stream);
int gg_gat_sell_fwd_f32(const uint32_t* chunk_ptr, int64_t chunks, const int32_t* idx, const int32_t* vdst,
                        const int32_t* hub_rows, const int32_t* hub_pptr, int64_t hubs, int64_t partial_rows,
                        const float* h, int64_t ldh, const float* a_tgt, const float* a_src, int64_t n, int64_t f,
                        float slope, const float* bias, float* out, int64_t ldo, float* rowstat, float* out_pos,
                        int64_t ld_pos, float* a_pos, void* workspace, size_t workspace_bytes, gg_stream_t stream);
int gg_gat_sell_bwd_edge_f32(const uint32_t* chunk_ptr, int64_t chunks, const int32_t* idx, const int32_t* slot_of,
                             const int32_t* vdst, const int32_t* hub_rows, const int32_t* hub_pptr, int64_t hubs,
                             int64_t partial_rows, const float* h, int64_t ldh, const float* g, int64_t ldg,
                             const float* fwd_out, int64_t ld_out, const float* bias, const float* a_tgt,
                             const float* a_src, const float* rowstat, int64_t n, int64_t f, float slope, float* dz,
                             float* da_tgt, void* workspace, size_t workspace_bytes, gg_stream_t stream);
int gg_gat_sell_bwd_src_f32(const uint32_t* chunk_ptr, int64_t chunks, const int32_t* idx, const int32_t* edge_map,
                            const int32_t* vdst, const int32_t* hub_rows, const int32_t* hub_pptr, int64_t hubs,
                            int64_t partial_rows, const float* g, int64_t ldg, const float* a_tgt, const float* a_src,
                            const float* rowstat, const float* dz, const float* da_tgt, const float* att_src,
                            const float* att_tgt, int64_t n, int64_t f, float slope, float* dh, int64_t ld_dh,
                            float* da_src, float* tstat_scratch, void* workspace, size_t workspace_bytes,
                            gg_stream_t stream);

/* The whole GAT backward in ONE heavy pass over the CSC sliced-ELL layout (csrc/gat_sell.cu): every slot gathers g_i once,
 * <g_i, h_j> gives dalpha, alpha is recomputed from the target's record, D_i = <g_i, out_i - bias> is precomputed per node;
 * dz never goes to memory: da_src_j is summed in the walk, and da_tgt_i = (1 - slope) (<g_i, out_pos_i> - D_i a_pos_i) comes
 * from the training forward's out_pos / a_pos (the share of the aggregation that arrives through positive logits; pass
 * them to gg_gat_sell_fwd_f32 to have them written).  Writes da_tgt, da_src and
 * dh = sum alpha g_i + da_src att_src + da_tgt att_tgt.  Replaces gg_gat_sell_bwd_edge_f32 + gg_gat_sell_bwd_src_f32 (two
 * passes of gathers).  `tstat_scratch`: 4 n floats. */
int gg_gat_sell_bwd_one_f32(const uint32_t* chunk_ptr, int64_t chunks, const int32_t* idx, const int32_t* vdst,
                            const int32_t* hub_rows, const int32_t* hub_pptr, int64_t hubs, int64_t partial_rows,
                            const float* h, int64_t ldh, const float* g, int64_t ldg, const float* fwd_out, int64_t ld_out,
                            const float* bias, const float* out_pos, int64_t ld_pos, const float* a_pos, const float* a_tgt,
                            const float* a_src, const float* rowstat, const float* att_src, const float* att_tgt, int64_t n,
                            int64_t f, float slope, float* dh, int64_t ld_dh, float* da_tgt, float* da_src,
                            float* tstat_scratch, void* workspace, size_t workspace_bytes, gg_stream_t stream);

/* Row gather / scatter-add / ReLU gradient used by the GIN-ID branch (ref: idconv.py:372-375):
 *   gather:      out[r,:]      = x[id[r],:]
 *   scatter_add: out[id[r],:] += x[r,:]      (atomicAdd: exact order-independence only for unique id,
 *                                             which node_id_index is, transform.py:38)
 *   relu_grad:   out = g .* (y > 0) */
int gg_gather_rows_f32(const float* x, int64_t ldx, const int64_t* id, int64_t m, int64_t f, float* out,
                       int64_t ldo, gg_stream_t stream);
int gg_scatter_add_rows_f32(const float* x, int64_t ldx, const int64_t* id, int64_t m, int64_t f,
                            float* out, int64_t ldo, gg_stream_t stream);
int gg_relu_grad_f32(const float* g, int64_t ldg, const float* y, int64_t ldy, int64_t n, int64_t f,
                     float* out, int64_t ldo, gg_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Peer memory over NVLink / NVSwitch (SURVEY §8e, §8b `gg_halo_*`): the exchange step of the
 * row-partitioned path.  The reference is single-process; one process per GPU here.
 *   gg_peer_alloc   cudaMalloc + zero + export: `handle_host` receives gg_peer_handle_bytes() opaque bytes
 *                   (a CUDA IPC handle) that the host side ships to the other ranks (torch.distributed);
 *   gg_peer_open    map a peer's buffer into this process -> device pointer usable by any kernel here;
 *   gg_peer_close / gg_peer_free  undo the two above;
 *   gg_peer_barrier stream-ordered barrier between the ranks, no host involvement: `flags_host[r]` is rank
 *                   r's flag block (>= GG_PEER_MAX + 1 u32, zero-initialised peer memory; the last word counts
 *                   this rank's barriers on the device, so a launch carries no host state and replays from a
 *                   CUDA graph).  Every rank must issue the same sequence of barriers.  Stores issued on
 *                   `stream` before the barrier are visible
 *                   to kernels the peers launch after theirs.  A peer that never arrives traps the launch
 *                   after ~20 s instead of hanging the GPU;
 *   gg_peer_scatter_cols_f32   forward leg of the feature-sliced exchange: this rank's rows
 *                   src[rows, f] are cut into `world` column slices of f/world and slice c is stored into
 *                   dst_host[c] (rank c's [N, f/world] matrix, peer memory) at rows row_base + i.
 * ------------------------------------------------------------------------------------------ */
#define GG_PEER_MAX 8
int gg_peer_handle_bytes(void);
int gg_peer_alloc(size_t bytes, void** ptr_host, unsigned char* handle_host);
int gg_peer_open(const unsigned char* handle_host, void** ptr_host);
int gg_peer_close(void* ptr);
int gg_peer_free(void* ptr);
int gg_peer_barrier(void* const* flags_host, int world, int rank, gg_stream_t stream);
int gg_peer_scatter_cols_f32(const float* src, int64_t ld, int64_t rows, int64_t f, float* const* dst_host,
                             int world, int rank, int64_t row_base, gg_stream_t stream);
/* Return leg of the feature-sliced exchange as a bulk push (the alternative to the peer-output epilogue of the
 * aggregation kernels): gg_peer_push_rows_f32 sends this rank's finished slice src[n, fs] to the rows' owners — owner o
 * receives rows [o * rows_per_rank, ...) as one contiguous block recv_o[rank][i][0:fs] (recv_host: HOST array of `world`
 * DEVICE pointers to the owners' receive buffers of world * rows_per_rank * fs floats); only the owners in
 * [owner_begin, owner_end) are served by a call, so that the push of one owner group can run on a second stream while the
 * next group's rows are still being aggregated; after a gg_peer_barrier the owner
 * assembles out[i, c * fs + k] = recv[c][i][k] with gg_peer_gather_slices_f32 (local). */
int gg_peer_push_rows_f32(const float* src, int64_t n, int64_t fs, int64_t rows_per_rank, int world, int rank,
                          int owner_begin, int owner_end, float* const* recv_host, gg_stream_t stream);
int gg_peer_gather_slices_f32(const float* recv, int64_t rows_per_rank, int64_t rows, int64_t fs, int world, float* out,
                              int64_t ldo, gg_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Graph-level pooling (SURVEY §8f item 3): global_add / mean / max_pool, ref: graphgym/models/pooling.py:12-33
 * (torch_scatter.scatter over `batch`, after index_select by node_id_index when the dataset transform is 'ego').
 *   gg_segment_bounds_i64  seg_ptr[g] = first position with key >= g for a NON-DECREASING key (DeepSNAP batches are
 *                          block-diagonal); *violations counts out-of-range or out-of-order keys (caller checks);
 *   gg_segment_pool_f32    out[g, :] = reduce over positions p in [seg_ptr[g], seg_ptr[g+1]) of x[row(p), :],
 *                          row(p) = row_index[p] (nullable: p); deterministic (rows in order); max stores the arg-max
 *                          position per (g, column) in `argmax` (nullable otherwise); empty graph -> 0;
 *   gg_segment_pool_bwd_f32 gx[row(p), :] = the gradient of that reduction (gx zero-initialised by the caller).
 * ------------------------------------------------------------------------------------------ */
enum gg_pool_mode { GG_POOL_SUM = 0, GG_POOL_MEAN = 1, GG_POOL_MAX = 2 };
int gg_segment_bounds_i64(const int64_t* key, int64_t m, int64_t num_segments, int32_t* seg_ptr,
                          int32_t* violations, gg_stream_t stream);
int gg_segment_pool_f32(const float* x, int64_t ldx, const int64_t* row_index, const int32_t* seg_ptr,
                        int64_t num_segments, int64_t f, int mode, float* out, int64_t ldo, int32_t* argmax,
                        gg_stream_t stream);
int gg_segment_pool_bwd_f32(const float* g, int64_t ldg, const int64_t* row_index, const int64_t* key,
                            const int32_t* seg_ptr, int64_t m, int64_t f, int mode, const int32_t* argmax, float* gx,
                            int64_t ldgx, gg_stream_t stream);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* GG_B200_H */
