"""ctypes binding of the C-ABI in include/gg_b200.h.

The library is the product: if it is missing or fails to load, every op raises. There is no
CPU / eager-PyTorch fallback anywhere in this package (the CPU restatement lives in ``oracle/``
and is test infrastructure only).
"""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgg_b200.so")
CSRC_DIR = os.path.join(_HERE, "csrc")

c_i64 = ctypes.c_int64
c_int = ctypes.c_int
c_f32 = ctypes.c_float
c_ptr = ctypes.c_void_p
c_size = ctypes.c_size_t

GG_GEMM_MAX_SEGMENTS = 4


class GemmSegment(ctypes.Structure):
    """``gg_gemm_segment`` (include/gg_b200.h)."""
    _fields_ = [("a", c_ptr), ("lda", c_i64), ("b", c_ptr), ("ldb", c_i64), ("scale", c_ptr),
                ("k", c_i64)]


# name -> (restype, argtypes); must list every symbol the header declares (tests check this)
SIGNATURES = {
    "gg_version": (c_int, []),
    "gg_last_error": (ctypes.c_char_p, []),
    "gg_launch_count": (c_i64, []),
    "gg_layout_capacity": (c_i64, [c_i64, c_i64, c_int]),
    "gg_layout_build_workspace_bytes": (c_size, [c_i64, c_i64, c_int]),
    "gg_layout_build": (c_int, [c_ptr, c_i64, c_i64, c_int, c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                c_size, c_ptr]),
    "gg_layout_build_range": (c_int, [c_ptr, c_i64, c_i64, c_int, c_int, c_i64, c_i64, c_i64, c_i64, c_ptr,
                                      c_ptr, c_ptr, c_ptr, c_ptr, c_size, c_ptr]),
    "gg_sort_pairs_workspace_bytes": (c_size, [c_i64]),
    "gg_sort_pairs_u32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_int, c_ptr, c_size, c_ptr]),
    "gg_layout_slot_map": (c_int, [c_ptr, c_ptr, c_i64, c_i64, c_i64, c_ptr, c_ptr, c_ptr]),
    "gg_layout_slot_weights": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_i64, c_i64, c_int, c_f32, c_ptr,
                                       c_ptr, c_ptr]),
    "gg_segment_degree": (c_int, [c_ptr, c_ptr, c_i64, c_ptr, c_ptr]),
    "gg_gcn_norm": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_ptr]),
    "gg_spmm_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_i64, c_int,
                            c_ptr, c_i64, c_f32, c_ptr, c_ptr]),
    "gg_spmm_plan_units": (c_int, [c_i64, c_i64]),
    "gg_spmm_plan_items": (c_i64, [c_i64, c_i64, c_int]),
    "gg_spmm_plan_build": (c_int, [c_ptr, c_i64, c_i64, c_int, c_ptr, c_ptr, c_ptr]),
    "gg_spmm_mp_workspace_bytes": (c_size, [c_i64, c_i64]),
    "gg_spmm_mp_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_i64, c_ptr, c_i64, c_i64,
                               c_i64, c_int, c_ptr, c_i64, c_f32, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                               c_size, c_int, c_ptr]),
    "gg_spmm_group_lanes": (c_int, [c_i64]),
    "gg_spmm_mpg_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_i64, c_ptr, c_i64,
                                c_ptr, c_int, c_i64, c_i64, c_i64, c_int, c_ptr, c_i64, c_f32, c_ptr, c_ptr, c_ptr,
                                c_ptr, c_ptr, c_ptr, c_size, c_int, c_ptr]),
    "gg_sell_vrow_capacity": (c_i64, [c_i64, c_i64, c_int]),
    "gg_sell_unit_capacity": (c_i64, [c_i64, c_i64, c_int]),
    "gg_sell_split_capacity": (c_i64, [c_i64, c_int]),
    "gg_sell_build_workspace_bytes": (c_size, [c_i64, c_i64, c_int]),
    "gg_sell_build": (c_int, [c_ptr, c_ptr, c_i64, c_i64, c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                              c_size, c_ptr]),
    "gg_sell_permute_f32": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_ptr]),
    "gg_sell_hub_hint_workspace_bytes": (c_size, [c_i64]),
    "gg_sell_hub_hint": (c_int, [c_ptr, c_i64, c_i64, c_ptr, c_i64, c_i64, c_ptr, c_ptr, c_size, c_ptr]),
    "gg_spmm_sell_workspace_bytes": (c_size, [c_i64, c_i64]),
    "gg_spmm_sell_f32": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_ptr,
                                 c_i64, c_ptr, c_int, c_i64, c_i64, c_i64, c_int, c_ptr, c_i64, c_f32, c_ptr, c_ptr, c_ptr,
                                 c_ptr, c_ptr, c_ptr, c_size, c_int, c_ptr]),
    "gg_spmm_sell_max_workspace_bytes": (c_size, [c_i64, c_i64]),
    "gg_spmm_sell_max_f32": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_i64,
                                     c_ptr, c_i64, c_ptr, c_i64, c_i64, c_i64, c_ptr, c_i64, c_f32, c_ptr, c_ptr, c_size,
                                     c_int, c_ptr]),
    "gg_spmm_sell_max_bwd_f32": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_ptr,
                                         c_i64, c_ptr, c_i64, c_i64, c_i64, c_f32, c_ptr, c_i64, c_ptr, c_size, c_int,
                                         c_ptr]),
    "gg_spmm_row_max_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_i64, c_ptr,
                                    c_i64, c_f32, c_ptr, c_ptr]),
    "gg_spmm_row_max_bwd_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_i64, c_f32,
                                        c_ptr, c_i64, c_ptr]),
    "gg_edge_row_reduce_f32": (c_int, [c_ptr, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_int, c_ptr, c_i64, c_ptr]),
    "gg_edge_rows_self_f32": (c_int, [c_ptr, c_i64, c_i64, c_int, c_ptr, c_i64, c_ptr, c_i64, c_ptr, c_i64, c_ptr, c_i64,
                                      c_ptr]),
    "gg_max_mask_f32": (c_int, [c_ptr, c_i64, c_ptr, c_i64, c_i64, c_i64, c_ptr, c_i64, c_ptr]),
    "gg_edge_max_sell_f32": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_i64,
                                     c_ptr, c_i64, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_ptr, c_i64, c_ptr, c_i64, c_i64,
                                     c_i64, c_ptr, c_i64, c_f32, c_ptr, c_ptr, c_size, c_int, c_ptr]),
    "gg_edge_max_row_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_ptr, c_i64,
                                    c_ptr, c_i64, c_ptr, c_i64, c_i64, c_i64, c_ptr, c_i64, c_f32, c_ptr, c_ptr]),
    "gg_edge_max_winner_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_i64, c_i64, c_ptr,
                                       c_i64, c_ptr]),
    "gg_edge_max_wgrad_workspace_bytes": (c_size, [c_i64, c_i64, c_i64]),
    "gg_edge_max_wgrad_f32": (c_int, [c_ptr, c_ptr, c_i64, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_i64, c_i64, c_ptr, c_i64,
                                      c_ptr, c_size, c_ptr]),
    "gg_spline_spread_sell_f32": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                          c_i64, c_i64, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_i64, c_int, c_ptr, c_size, c_int,
                                          c_ptr]),
    "gg_spline_blend_sell_f32": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                         c_i64, c_i64, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_i64, c_int, c_ptr, c_i64, c_ptr,
                                         c_ptr, c_size, c_int, c_ptr]),
    "gg_spline_spread_row_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_i64, c_int,
                                         c_ptr]),
    "gg_spline_blend_row_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_i64, c_int,
                                        c_ptr, c_i64, c_ptr, c_ptr]),
    "gg_spline_du_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_i64, c_i64, c_i64, c_ptr,
                                 c_ptr]),
    "gg_max_winner_sddmm_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_int, c_i64, c_ptr,
                                        c_ptr]),
    "gg_gat_alpha_heads_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_int, c_f32, c_ptr, c_ptr]),
    "gg_gat_dz_heads_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_int, c_f32, c_ptr, c_ptr, c_ptr]),
    "gg_gat_src_sum_heads_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_i64, c_int, c_ptr, c_ptr]),
    "gg_spmm_row_max_heads_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_int, c_ptr, c_i64, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_i64,
                                          c_ptr, c_ptr]),
    "gg_spmm_row_max_heads_bwd_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_i64,
                                              c_ptr, c_i64, c_ptr]),
    "gg_rows_epilogue_f32": (c_int, [c_ptr, c_i64, c_i64, c_i64, c_ptr, c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                     c_i64, c_ptr]),
    "gg_cast_f32_bf16": (c_int, [c_ptr, c_i64, c_i64, c_i64, c_ptr, c_i64, c_ptr]),
    "gg_spmm_mp_bf16": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_i64,
                                c_int, c_ptr, c_i64, c_f32, c_ptr, c_ptr, c_size, c_int, c_ptr]),
    "gg_segment_bounds_i64": (c_int, [c_ptr, c_i64, c_i64, c_ptr, c_ptr, c_ptr]),
    "gg_segment_pool_f32": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_i64, c_i64, c_int, c_ptr, c_i64, c_ptr, c_ptr]),
    "gg_segment_pool_bwd_f32": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_int, c_ptr, c_ptr, c_i64,
                                        c_ptr]),
    "gg_peer_handle_bytes": (c_int, []),
    "gg_peer_alloc": (c_int, [c_size, ctypes.POINTER(c_ptr), ctypes.c_char_p]),
    "gg_peer_open": (c_int, [ctypes.c_char_p, ctypes.POINTER(c_ptr)]),
    "gg_peer_close": (c_int, [c_ptr]),
    "gg_peer_free": (c_int, [c_ptr]),
    "gg_peer_barrier": (c_int, [ctypes.POINTER(c_ptr), c_int, c_int, c_ptr]),
    "gg_peer_scatter_cols_f32": (c_int, [c_ptr, c_i64, c_i64, c_i64, ctypes.POINTER(c_ptr), c_int, c_int, c_i64, c_ptr]),
    "gg_peer_push_rows_f32": (c_int, [c_ptr, c_i64, c_i64, c_i64, c_int, c_int, c_int, c_int, ctypes.POINTER(c_ptr), c_ptr]),
    "gg_peer_gather_slices_f32": (c_int, [c_ptr, c_i64, c_i64, c_i64, c_int, c_ptr, c_i64, c_ptr]),
    "gg_id_gemm_f32": (c_int, [ctypes.POINTER(GemmSegment), c_int, c_int, c_i64, c_i64, c_ptr, c_int,
                               c_ptr, c_i64, c_ptr, c_i64, c_ptr]),
    "gg_id_gemm_tc_workspace_bytes": (c_size, [ctypes.POINTER(GemmSegment), c_int, c_i64]),
    "gg_id_gemm_tc_f32": (c_int, [ctypes.POINTER(GemmSegment), c_int, c_int, c_i64, c_i64, c_ptr, c_int,
                                  c_ptr, c_i64, c_ptr, c_i64, c_ptr, c_size, c_ptr]),
    "gg_gemm_tn_workspace_bytes": (c_size, [c_i64, c_i64, c_i64]),
    "gg_gemm_tn_f32": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_i64, c_i64, c_i64, c_i64, c_ptr, c_i64,
                               c_ptr, c_size, c_ptr]),
    "gg_gemm_tn_tc_workspace_bytes": (c_size, [c_i64, c_i64, c_i64]),
    "gg_gemm_tn_tc_f32": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_i64, c_i64, c_i64, c_i64, c_ptr, c_i64,
                                  c_ptr, c_size, c_ptr]),
    "gg_colsum_workspace_bytes": (c_size, [c_i64, c_i64]),
    "gg_colsum_f32": (c_int, [c_ptr, c_i64, c_i64, c_i64, c_ptr, c_ptr, c_size, c_ptr]),
    "gg_id_count": (c_int, [c_ptr, c_i64, c_i64, c_ptr, c_ptr]),
    "gg_mean_weights": (c_int, [c_ptr, c_ptr, c_i64, c_ptr, c_ptr]),
    "gg_gat_scores_f32": (c_int, [c_ptr, c_i64, c_ptr, c_i64, c_int, c_int, c_ptr, c_ptr, c_ptr]),
    "gg_gat_fwd_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_ptr, c_i64, c_int, c_int, c_f32, c_ptr,
                               c_ptr, c_ptr, c_i64, c_ptr]),
    "gg_gat_bwd_edge_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_ptr,
                                    c_i64, c_ptr, c_i64, c_int, c_int, c_f32, c_ptr, c_ptr, c_ptr]),
    "gg_gat_bwd_src_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_ptr, c_i64,
                                   c_int, c_int, c_ptr, c_ptr, c_i64, c_ptr]),
    "gg_gat_att_grad_workspace_bytes": (c_size, [c_i64, c_int, c_int]),
    "gg_gat_att_grad_f32": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_i64, c_int, c_int, c_ptr, c_ptr, c_size,
                                    c_ptr]),
    "gg_cycle_diag_workspace_bytes": (c_size, [c_i64]),
    "gg_cycle_diag_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_int, c_int, c_i64, c_int, c_ptr, c_i64,
                                  c_ptr, c_size, c_ptr]),
    "gg_cycle_diag_mp_workspace_bytes": (c_size, [c_i64, c_i64]),
    "gg_cycle_diag_mp_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_int, c_int, c_i64, c_int, c_ptr,
                                     c_i64, c_ptr, c_size, c_ptr]),
    "gg_cycle_diag_sell_workspace_bytes": (c_size, [c_i64, c_i64]),
    "gg_cycle_diag_sell_f32": (c_int, [c_ptr, c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_i64, c_int,
                                       c_int, c_i64, c_int, c_ptr, c_i64, c_ptr, c_size, c_ptr]),
    "gg_cycle_diag_i64": (c_int, [c_ptr, c_ptr, c_i64, c_i64, c_int, c_int, c_i64, c_int, c_ptr, c_i64, c_ptr,
                                  c_ptr, c_size, c_ptr]),
    "gg_egonet_workspace_bytes": (c_size, [c_i64, c_i64]),
    "gg_egonet_sizes": (c_int, [c_ptr, c_ptr, c_i64, c_int, c_ptr, c_ptr, c_i64, c_int, c_ptr, c_ptr, c_ptr,
                                c_ptr, c_size, c_ptr]),
    "gg_egonet_fill": (c_int, [c_ptr, c_ptr, c_i64, c_int, c_ptr, c_ptr, c_i64, c_int, c_ptr, c_ptr, c_ptr,
                               c_i64, c_ptr, c_ptr, c_ptr]),
    "gg_gat_alpha_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_f32, c_ptr, c_ptr]),
    "gg_gat_sddmm_mp_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_i64,
                                    c_ptr, c_ptr, c_ptr]),
    "gg_gat_sddmm_mpg_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_i64,
                                     c_ptr, c_ptr, c_ptr]),
    "gg_gat_dz_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_f32, c_ptr, c_ptr, c_ptr]),
    "gg_gat_csc_gather_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_ptr, c_ptr]),
    "gg_collate_index_i64": (c_int, [c_ptr, c_int, c_i64, c_ptr, c_ptr, c_ptr]),
    "gg_collate_rows_f32": (c_int, [c_ptr, c_int, c_i64, c_int, c_ptr, c_i64, c_i64, c_ptr, c_ptr]),
    "gg_f64_sort_keys": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_ptr]),
    "gg_gather_u32": (c_int, [c_ptr, c_ptr, c_i64, c_ptr, c_ptr]),
    "gg_digitize_f64": (c_int, [c_ptr, c_i64, c_ptr, c_int, c_ptr, c_ptr]),
    "gg_postops_workspace_bytes": (c_size, [c_i64, c_i64]),
    "gg_bn_stats_f32": (c_int, [c_ptr, c_i64, c_i64, c_i64, c_f32, c_ptr, c_ptr, c_ptr, c_ptr, c_f32, c_ptr, c_size, c_ptr]),
    "gg_postops_fwd_f32": (c_int, [c_ptr, c_i64, c_i64, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_f32, c_int, c_ptr,
                                   c_i64, c_ptr, c_ptr]),
    "gg_postops_bwd_f32": (c_int, [c_ptr, c_i64, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_i64, c_ptr, c_ptr, c_ptr, c_int,
                                   c_int, c_f32, c_int, c_ptr, c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_size, c_ptr]),
    "gg_postops_skip_fwd_f32": (c_int, [c_ptr, c_i64, c_ptr, c_i64, c_i64, c_i64, c_i64, c_int, c_ptr, c_ptr, c_ptr,
                                        c_ptr, c_int, c_f32, c_int, c_ptr, c_i64, c_ptr, c_ptr]),
    "gg_postops_skip_bwd_f32": (c_int, [c_ptr, c_i64, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_i64, c_i64, c_int, c_ptr,
                                        c_ptr, c_ptr, c_int, c_int, c_f32, c_int, c_ptr, c_ptr, c_i64, c_ptr, c_i64,
                                        c_ptr, c_ptr, c_ptr, c_size, c_ptr]),
    "gg_segment_softmax_f32": (c_int, [c_ptr, c_ptr, c_i64, c_f32, c_ptr, c_ptr]),
    "gg_segment_softmax_bwd_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_i64, c_f32, c_ptr, c_ptr]),
    "gg_gat_sell_workspace_bytes": (c_size, [c_i64, c_i64]),
    "gg_sell_compose_map": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_ptr]),
    "gg_gat_sell_fwd_f32": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_ptr, c_ptr,
                                    c_i64, c_i64, c_f32, c_ptr, c_ptr, c_i64, c_ptr, c_ptr, c_i64, c_ptr, c_ptr, c_size,
                                    c_ptr]),
    "gg_gat_sell_bwd_edge_f32": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_i64,
                                         c_ptr, c_i64, c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_f32,
                                         c_ptr, c_ptr, c_ptr, c_size, c_ptr]),
    "gg_gat_sell_bwd_src_f32": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_i64,
                                        c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_f32, c_ptr, c_i64,
                                        c_ptr, c_ptr, c_ptr, c_size, c_ptr]),
    "gg_gat_sell_bwd_one_f32": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_ptr, c_i64, c_ptr,
                                        c_i64, c_ptr, c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_f32,
                                        c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_size, c_ptr]),
    "gg_gather_rows_f32": (c_int, [c_ptr, c_i64, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_ptr]),
    "gg_scatter_add_rows_f32": (c_int, [c_ptr, c_i64, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_ptr]),
    "gg_relu_grad_f32": (c_int, [c_ptr, c_i64, c_ptr, c_i64, c_i64, c_i64, c_ptr, c_i64, c_ptr]),
}

_lib = None


class GGError(RuntimeError):
    """A gg_* entry point returned a negative status."""


def build(verbose=False):
    """Compile graphgym_b200/csrc for sm_100a into graphgym_b200/libgg_b200.so (nvcc, no GPU needed)."""
    cmd = ["make", "-C", CSRC_DIR, "-j8"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout)
        print(res.stderr)
    if res.returncode != 0:
        raise RuntimeError("building libgg_b200.so failed (see output above)")
    return LIB_PATH


def lib():
    """The loaded library; raises loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: the CUDA hot path is not built and there is no fallback. "
                "Run `python -c 'import __graft_entry__ as g; g.build()'` or "
                "`make -C graphgym_b200/csrc`.")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the .so is stale: also loud
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(status, what):
    if status != 0:
        msg = lib().gg_last_error()
        raise GGError(f"{what} failed with status {status}: {msg.decode() if msg else ''}")
