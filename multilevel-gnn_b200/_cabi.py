"""ctypes binding of libmlg_b200.so (include/mlg_b200.h).

This is the only place the product touches native code.  There is NO CPU fallback: if the library
is missing, cannot be loaded, or a tensor is not a contiguous CUDA tensor of the expected dtype, the
call raises.  Every wrapper only enqueues work on ``torch.cuda.current_stream()``.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MLG_B200_LIB") or os.path.join(_HERE, "lib", "libmlg_b200.so")   # override: kernel A/B tuning

_c_i64, _c_int, _c_f32, _c_vp = ctypes.c_int64, ctypes.c_int, ctypes.c_float, ctypes.c_void_p

# name -> (restype, argtypes); mirrors include/mlg_b200.h one to one
_SIGNATURES = {
    "mlg_abi_version": (_c_int, []),
    "mlg_last_error": (ctypes.c_char_p, []),
    "mlg_csr_build_workspace_bytes": (_c_i64, [_c_i64, _c_i64, _c_int]),
    "mlg_csr_build": (_c_int, [_c_vp, _c_i64, _c_i64, _c_int, _c_int, _c_int, _c_vp, _c_vp, _c_vp, _c_vp,
                               _c_i64, _c_vp]),
    "mlg_edge_values": (_c_int, [_c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_f32, _c_vp, _c_vp]),
    "mlg_gen_aggr_fwd": (_c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_int, _c_f32, _c_vp,
                                  _c_f32, _c_vp, _c_vp, _c_f32, _c_int, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp]),
    "mlg_gen_aggr_bwd_partial_rows": (_c_i64, [_c_i64, _c_i64]),
    "mlg_gen_aggr_bwd": (_c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_int, _c_int,
                                  _c_f32, _c_vp, _c_f32, _c_vp, _c_vp, _c_f32, _c_int, _c_vp, _c_vp, _c_vp,
                                  _c_vp, _c_vp, _c_vp, _c_vp]),
    "mlg_gen_aggr_bwd_src_supported": (_c_int, [_c_i64, _c_int, _c_int]),
    "mlg_gen_aggr_bwd_src": (_c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_int, _c_int,
                                  _c_f32, _c_vp, _c_f32, _c_vp, _c_vp, _c_f32, _c_int, _c_vp, _c_vp, _c_vp,
                                  _c_vp, _c_vp, _c_vp, _c_vp]),
    "mlg_gather_sum": (_c_int, [_c_vp, _c_i64, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64,
                                _c_i64, _c_i64, _c_int, _c_int, _c_vp, _c_i64, _c_vp, _c_i64, _c_vp, _c_i64, _c_vp, _c_i64,
                                _c_f32, _c_vp, _c_vp]),
    "mlg_gather_sum_act": (_c_int, [_c_vp, _c_i64, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64,
                                    _c_i64, _c_i64, _c_int, _c_int, _c_vp, _c_i64, _c_vp, _c_i64, _c_vp, _c_i64, _c_vp, _c_i64,
                                    _c_f32, _c_vp, _c_int, _c_f32, _c_vp]),
    "mlg_gather_sum_slices": (_c_i64, [_c_i64, _c_i64, _c_i64]),
    # (xs, e_self, ld_self, e_nbr, ld_nbr, rowptr, idx, val, order, n_rows, C, replicas, bias, slope, out, ld_out, mask_bits, stream)
    "mlg_sage_rank1_fwd": (_c_int, [_c_vp, _c_vp, _c_i64, _c_vp, _c_i64, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64,
                                    _c_vp, _c_f32, _c_vp, _c_i64, _c_vp, _c_vp]),
    # (gz, ld_g, xs, rowptr_t, idx_t, val_t, inv_cnt, order_t, n_rows, C, replicas, g_e12_parts, g_bias_parts, stream)
    "mlg_sage_rank1_bwd": (_c_int, [_c_vp, _c_i64, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64, _c_vp,
                                    _c_vp, _c_vp]),
    "mlg_sage_rank1_bwd_rows_supported": (_c_int, [_c_i64]),
    # (gz, ld_g, y, mask_bits, slope, xs, rowptr, idx, val, order, n_rows, C, replicas, h, g_self, ld_self, g_bias_rows, stream)
    "mlg_sage_rank1_bwd_rows": (_c_int, [_c_vp, _c_i64, _c_vp, _c_vp, _c_f32, _c_vp, _c_int, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64,
                                         _c_vp, _c_vp, _c_i64, _c_vp, _c_vp]),
    "mlg_sage_rank1_bwd_rows_nm": (_c_int, [_c_vp, _c_i64, _c_vp, _c_vp, _c_f32, _c_vp, _c_int, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64,
                                            _c_i64, _c_vp, _c_vp, _c_i64, _c_vp, _c_vp]),
    "mlg_sage_rank1_fwd_rows_nm": (_c_int, [_c_vp, _c_vp, _c_i64, _c_vp, _c_i64, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64,
                                            _c_vp, _c_f32, _c_vp, _c_i64, _c_vp, _c_vp]),
    "mlg_gather_sum_nm_ex": (_c_int, [_c_vp, _c_i64, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_int, _c_vp, _c_i64,
                                      _c_int, _c_f32, _c_vp, _c_i64, _c_vp, _c_i64, _c_int, _c_vp]),
    "mlg_transpose_bn": (_c_int, [_c_vp, _c_i64, _c_i64, _c_vp, _c_vp]),
    "mlg_sage_rank1_fwd_rows_supported": (_c_int, [_c_i64]),
    "mlg_sage_rank1_fwd_rows": (_c_int, [_c_vp, _c_vp, _c_i64, _c_vp, _c_i64, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64,
                                         _c_vp, _c_f32, _c_vp, _c_i64, _c_vp, _c_vp]),
    "mlg_xty_workspace_bytes": (_c_i64, [_c_i64, _c_i64, _c_i64]),
    "mlg_xty_tc_supported": (_c_int, [_c_i64, _c_i64, _c_i64]),
    "mlg_xty_tc_workspace_bytes": (_c_i64, [_c_i64]),
    "mlg_xty_tc": (_c_int, [_c_vp, _c_i64, _c_vp, _c_i64, _c_i64, _c_i64, _c_i64, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_vp]),
    "mlg_skinny_linear_workspace_bytes": (_c_i64, [_c_i64, _c_i64]),
    "mlg_skinny_linear": (_c_int, [_c_vp, _c_i64, _c_vp, _c_i64, _c_vp, _c_i64, _c_i64, _c_i64, _c_int, _c_f32, _c_vp,
                                   _c_i64, _c_vp, _c_i64, _c_vp]),
    "mlg_head_conv_pool_supported": (_c_int, [_c_i64, _c_i64, _c_i64]),
    "mlg_head_conv_pool_bwd_workspace_bytes": (_c_i64, [_c_i64, _c_i64, _c_i64, _c_i64, _c_i64]),
    "mlg_head_conv_pool_fwd": (_c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_f32, _c_i64, _c_i64, _c_i64,
                                        _c_i64, _c_i64, _c_vp, _c_i64, _c_vp]),
    "mlg_head_conv_pool_bwd": (_c_int, [_c_vp, _c_i64, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_f32, _c_i64, _c_i64,
                                        _c_i64, _c_i64, _c_i64, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_vp]),
    "mlg_head_mlp_workspace_bytes": (_c_i64, [_c_i64, _c_i64, _c_i64]),
    "mlg_head_mlp_fwd": (_c_int, [_c_vp, _c_i64, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_f32, _c_vp, _c_vp, _c_i64, _c_i64,
                                  _c_i64, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_vp]),
    "mlg_head_mlp_bwd": (_c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_vp, _c_vp, _c_vp, _c_f32, _c_i64,
                                  _c_i64, _c_i64, _c_vp, _c_i64, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp]),
    "mlg_diffpool_smem_bytes": (_c_i64, [_c_i64, _c_vp]),
    "mlg_diffpool_supported": (_c_int, [_c_i64, _c_vp]),
    "mlg_diffpool_grad_floats": (_c_i64, [_c_i64, _c_vp]),
    "mlg_diffpool_state_floats": (_c_i64, [_c_i64, _c_vp]),
    "mlg_diffpool_ctas": (_c_i64, [_c_i64]),
    "mlg_diffpool_fwd": (_c_int, [_c_vp, _c_vp, _c_vp, _c_i64, _c_vp, _c_i64, _c_vp, _c_vp, _c_vp, _c_vp]),
    "mlg_diffpool_bwd": (_c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_vp, _c_i64, _c_vp, _c_vp, _c_vp, _c_vp,
                                  _c_i64, _c_vp]),
    "mlg_decoder_max_rows": (_c_i64, [_c_i64, _c_i64, _c_int]),
    "mlg_decoder_fwd": (_c_int, [_c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64, _c_i64, _c_i64, _c_i64, _c_vp, _c_vp, _c_vp]),
    "mlg_decoder_bwd": (_c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64, _c_i64, _c_i64, _c_i64, _c_vp,
                                 _c_vp, _c_vp]),
    "mlg_sage_fold_fwd": (_c_int, [_c_vp, _c_vp, _c_i64, _c_i64, _c_i64, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp]),
    "mlg_sage_fold_bwd": (_c_int, [_c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64, _c_vp, _c_vp, _c_vp]),
    "mlg_sage_fold_stacked_fwd": (_c_int, [_c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp,
                                           _c_vp, _c_vp]),
    "mlg_sage_fold_stacked_bwd": (_c_int, [_c_vp, _c_vp, _c_i64, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64, _c_vp, _c_vp, _c_vp]),
    "mlg_pca_indep_loss": (_c_int, [_c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_vp, _c_vp, _c_vp]),
    "mlg_maxpool_cl_fwd": (_c_int, [_c_vp, _c_i64, _c_i64, _c_i64, _c_i64, _c_i64, _c_i64, _c_vp, _c_vp, _c_vp]),
    "mlg_maxpool_cl_bwd": (_c_int, [_c_vp, _c_vp, _c_i64, _c_i64, _c_i64, _c_i64, _c_i64, _c_i64, _c_vp, _c_vp]),
    "mlg_layernorm_supported": (_c_int, [_c_i64]),
    "mlg_layernorm_bwd_workspace_bytes": (_c_i64, [_c_i64, _c_i64]),
    "mlg_layernorm_fwd": (_c_int, [_c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_f32, _c_vp, _c_vp, _c_vp, _c_vp]),
    "mlg_layernorm_bwd": (_c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64,
                                   _c_vp]),
    "mlg_layernorm_relu_fwd": (_c_int, [_c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_f32, _c_vp, _c_vp, _c_vp, _c_vp]),
    "mlg_layernorm_relu_bwd": (_c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_vp, _c_vp, _c_vp, _c_vp,
                                        _c_i64, _c_vp]),
    # (x, edge_scalar, edge_p, edge_q, rowptr, col, eid, n, H, mode, t, t_dev, p, p_dev, y_dev, eps, epilogue, scale, m, aux, h, stream)
    "mlg_gen_aggr_fwd_affine": (_c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_int, _c_f32, _c_vp,
                                         _c_f32, _c_vp, _c_vp, _c_f32, _c_int, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp]),
    # (g, x, edge_scalar, edge_p, edge_q, rowptr, col, eid, n, n_edges, H, mode, learn, t, t_dev, p, p_dev, y_dev, eps, epilogue,
    #  scale, m, aux, g_edge, g_x, partials, g_p, g_q, workspace, workspace_bytes, stream)
    "mlg_gen_aggr_bwd_affine": (_c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64, _c_int,
                                         _c_int, _c_f32, _c_vp, _c_f32, _c_vp, _c_vp, _c_f32, _c_int, _c_vp, _c_vp, _c_vp,
                                         _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_vp]),
    "mlg_gen_aggr_bwd_affine_src": (_c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64, _c_int,
                                         _c_int, _c_f32, _c_vp, _c_f32, _c_vp, _c_vp, _c_f32, _c_int, _c_vp, _c_vp, _c_vp,
                                         _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_vp]),
    "mlg_gen_aggr_bwd_affine_workspace_bytes": (_c_i64, [_c_i64, _c_i64, _c_i64]),
    "mlg_wcolsum_workspace_bytes": (_c_i64, [_c_i64, _c_i64]),
    "mlg_wcolsum": (_c_int, [_c_vp, _c_i64, _c_vp, _c_i64, _c_i64, _c_vp, _c_vp, _c_vp, _c_i64, _c_vp]),
    "mlg_eval_metrics_workspace_bytes": (_c_i64, [_c_i64]),
    "mlg_eval_metrics": (_c_int, [_c_vp, _c_vp, _c_i64, _c_vp, _c_vp, _c_vp, _c_i64, _c_vp]),
    "mlg_xty": (_c_int, [_c_vp, _c_i64, _c_vp, _c_i64, _c_i64, _c_i64, _c_i64, _c_vp, _c_vp, _c_vp, _c_i64, _c_vp]),
    "mlg_bias_act": (_c_int, [_c_vp, _c_vp, _c_i64, _c_i64, _c_f32, _c_vp]),
    "mlg_embed_scale_fwd": (_c_int, [_c_vp, _c_vp, _c_i64, _c_i64, _c_i64, _c_vp, _c_vp]),
    "mlg_embed_scale_bwd": (_c_int, [_c_vp, _c_vp, _c_i64, _c_i64, _c_i64, _c_vp, _c_vp]),
    "mlg_embed_scale_bwd_xs": (_c_int, [_c_vp, _c_vp, _c_i64, _c_i64, _c_i64, _c_vp, _c_vp]),
    "mlg_sage_rank1_bwd_xs_workspace_bytes": (_c_i64, [_c_i64, _c_i64, _c_i64]),
    # (gz, ld_g, gz_nm, y, mask_bits, slope, e_self, ld_self, e_nbr, ld_nbr, rowptr, idx, val, order, rowptr_t, fwd_pos_t,
    #  n_rows, cap, C, replicas, g_xs, workspace, workspace_bytes, stream)
    "mlg_sage_rank1_bwd_xs": (_c_int, [_c_vp, _c_i64, _c_int, _c_vp, _c_vp, _c_f32, _c_vp, _c_i64, _c_vp, _c_i64, _c_vp, _c_vp,
                                       _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64, _c_i64, _c_vp, _c_vp, _c_i64, _c_vp]),
    "mlg_attr_accumulate": (_c_int, [_c_vp, _c_i64, _c_vp, _c_vp, _c_i64, _c_i64, _c_int, _c_vp, _c_vp]),
    "mlg_pool_fwd": (_c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64, _c_i64, _c_i64,
                              _c_i64, _c_int, _c_vp, _c_vp]),
    "mlg_pool_bwd_x": (_c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64, _c_i64,
                                _c_i64, _c_i64, _c_i64, _c_vp, _c_vp]),
    "mlg_pool_bwd_w": (_c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64, _c_i64, _c_i64,
                                _c_i64, _c_int, _c_i64, _c_vp, _c_vp]),
    "mlg_pool_bwd": (_c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64, _c_i64, _c_i64, _c_i64,
                              _c_i64, _c_vp, _c_vp, _c_vp, _c_int, _c_f32, _c_vp, _c_vp]),
    "mlg_pool_bwd_node_major_supported": (_c_int, [_c_i64, _c_i64]),
    "mlg_pool_bwd_layout": (_c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64, _c_i64, _c_i64,
                                     _c_i64, _c_i64, _c_vp, _c_vp, _c_vp, _c_int, _c_f32, _c_vp, _c_int, _c_vp]),
    "mlg_pool_bwd_vm": (_c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64, _c_i64, _c_i64,
                                 _c_i64, _c_i64, _c_vp, _c_vp, _c_vp, _c_int, _c_f32, _c_vp, _c_int, _c_vp, _c_vp]),
    "mlg_gather_sum_nm": (_c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_vp, _c_i64, _c_vp, _c_i64,
                                   _c_vp]),
    "mlg_cast_bf16": (_c_int, [_c_vp, _c_i64, _c_i64, _c_i64, _c_i64, _c_int, _c_vp, _c_i64, _c_vp]),
    "mlg_gemm_bf16": (_c_int, [_c_vp, _c_i64, _c_i64, _c_vp, _c_i64, _c_i64, _c_vp, _c_i64, _c_i64, _c_i64, _c_i64,
                               _c_i64, _c_i64, _c_f32, _c_vp]),
    "mlg_gemm_bf16_workspace_bytes": (_c_i64, []),
    "mlg_gemm_bf16_ws": (_c_int, [_c_vp, _c_i64, _c_i64, _c_vp, _c_i64, _c_i64, _c_vp, _c_i64, _c_i64, _c_i64, _c_i64,
                                  _c_i64, _c_i64, _c_f32, _c_vp, _c_i64, _c_vp]),
    "mlg_split_tf32": (_c_int, [_c_vp, _c_i64, _c_vp, _c_vp, _c_vp]),
    "mlg_gemm_tf32x3_supported": (_c_int, [_c_i64, _c_i64, _c_i64]),
    "mlg_gemm_tf32x3": (_c_int, [_c_vp, _c_i64, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64, _c_i64, _c_int, _c_f32,
                                 _c_vp]),
    "mlg_peer_flag_bytes": (_c_i64, []),
    "mlg_peer_alloc": (_c_vp, [_c_i64]),
    "mlg_peer_free": (_c_int, [_c_vp]),
    "mlg_peer_export": (_c_int, [_c_vp, _c_vp]),
    "mlg_peer_open": (_c_vp, [_c_vp]),
    "mlg_peer_close": (_c_int, [_c_vp]),
    "mlg_peer_adam_step": (_c_int, [_c_vp, _c_vp, _c_vp, _c_int, _c_int, _c_i64, _c_i64, _c_vp, _c_vp, _c_vp, _c_f32, _c_f32,
                                    _c_f32, _c_f32, _c_f32, ctypes.c_double, _c_vp, _c_int, _c_vp]),
    "mlg_peer_emulated_bytes": (_c_i64, [_c_int]),
    "mlg_peer_adam_step_emulated": (_c_int, [_c_vp, _c_vp, _c_vp, _c_int, _c_i64, _c_i64, _c_vp, _c_vp, _c_vp, _c_f32, _c_f32,
                                             _c_f32, _c_f32, _c_f32, ctypes.c_double, _c_vp, _c_vp]),
    "mlg_peer_status": (_c_int, [_c_vp, _c_vp]),
    "mlg_adam_step": (_c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_f32, _c_f32, _c_f32, _c_f32, _c_f32, _c_vp]),
    "mlg_knn_workspace_bytes": (_c_i64, [_c_i64, _c_i64, _c_i64, _c_i64, _c_i64]),
    "mlg_knn_graph": (_c_int, [_c_vp, _c_i64, _c_i64, _c_i64, _c_i64, _c_i64, _c_int, _c_vp, _c_vp, _c_vp, _c_vp,
                               _c_i64, _c_vp]),
}

_lib = None


class NativeLibraryError(RuntimeError):
    pass


def exported_symbols():
    return sorted(_SIGNATURES)


def lib():
    """Loads libmlg_b200.so once; raises NativeLibraryError when it is absent (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeLibraryError(
                "%s not found: build it with `python multilevel-gnn_b200/build.py` "
                "(or __graft_entry__.build()); there is no CPU fallback" % LIB_PATH)
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        if handle.mlg_abi_version() != 1:
            raise NativeLibraryError("libmlg_b200.so ABI version mismatch")
        _lib = handle
    return _lib


def last_error():
    return lib().mlg_last_error().decode()


# kernels launched per C call (own kernels only; CUB's sort passes inside mlg_csr_build are not counted)
_LAUNCHES_PER_CALL = {"mlg_csr_build": 2, "mlg_knn_graph": 2, "mlg_xty": 2, "mlg_xty_tc": 2, "mlg_skinny_linear": 2, "mlg_wcolsum": 2, "mlg_gen_aggr_bwd_affine": 3, "mlg_gen_aggr_bwd_affine_src": 3, "mlg_layernorm_bwd": 2, "mlg_layernorm_relu_bwd": 2, "mlg_pool_bwd": 2, "mlg_pool_bwd_layout": 2, "mlg_adam_step": 2,
                      "mlg_head_conv_pool_bwd": 2, "mlg_head_mlp_fwd": 2, "mlg_diffpool_bwd": 2, "mlg_pca_indep_loss": 2}
LAUNCH_COUNT = 0
TIMER = None        # a KernelTimer while bench.py measures per-kernel device time


def check(rc, who):
    global LAUNCH_COUNT
    if rc != 0:
        raise RuntimeError("%s failed (%d): %s" % (who, rc, last_error()))
    LAUNCH_COUNT += _LAUNCHES_PER_CALL.get(who, 1)


class KernelTimer:
    """CUDA-event spans around tagged kernel launches, on the launching stream (bench.py's roofline leg)."""

    def __init__(self):
        self.spans = []          # (tag, start_event, end_event, algorithmic_bytes)

    def span(self, tag, nbytes):
        return _Span(self, tag, nbytes)

    def summary(self):
        torch.cuda.synchronize()
        out = {}
        for tag, a, b, nbytes in self.spans:
            d = out.setdefault(tag, {"launches": 0, "ms": 0.0, "bytes": 0})
            d["launches"] += 1
            d["ms"] += a.elapsed_time(b)
            d["bytes"] += nbytes
        return out


class _Span:
    def __init__(self, timer, tag, nbytes):
        self.timer, self.tag, self.nbytes = timer, tag, nbytes

    def __enter__(self):
        self.a = torch.cuda.Event(enable_timing=True)
        self.b = torch.cuda.Event(enable_timing=True)
        self.a.record()

    def __exit__(self, *exc):
        self.b.record()
        self.timer.spans.append((self.tag, self.a, self.b, self.nbytes))


class _NoSpan:
    def __enter__(self):
        return None

    def __exit__(self, *exc):
        return False


_NOSPAN = _NoSpan()


def span(tag, nbytes=0):
    """with _cabi.span("gather_sum", bytes): ...  -- no-op unless a KernelTimer is installed."""
    return TIMER.span(tag, nbytes) if TIMER is not None else _NOSPAN


def stream_ptr():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda(*tensors):
    """The product has no CPU path: refuse anything that is not a CUDA tensor."""
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise NativeLibraryError(
                "multilevel-gnn_b200 kernels need CUDA tensors (got %s); there is no CPU fallback" % t.device)


def ptr(t, dtype=None, allow_none=False):
    """Device pointer of a contiguous CUDA tensor (or NULL)."""
    if t is None:
        if allow_none:
            return None
        raise ValueError("required tensor is None")
    if not t.is_cuda:
        raise NativeLibraryError("multilevel-gnn_b200 kernels need CUDA tensors (got %s); no CPU fallback" % t.device)
    if dtype is not None and t.dtype != dtype:
        raise TypeError("expected %s, got %s" % (dtype, t.dtype))
    if not t.is_contiguous():
        raise ValueError("tensor must be contiguous")
    return ctypes.c_void_p(t.data_ptr())


def fptr(t, allow_none=False):
    return ptr(t, torch.float32, allow_none)


def iptr(t, allow_none=False):
    return ptr(t, torch.int32, allow_none)


def lptr(t, allow_none=False):
    return ptr(t, torch.int64, allow_none)
