"""ctypes binding of the C ABI declared in include/s4g_b200.h.

There is NO fallback: if ``libs4g_b200.so`` is missing the import fails loudly, and every entry point
refuses CPU tensors (like the reference's CHECK_CUDA).  The oracle under oracle/ is never used here.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("S4G_LIB_PATH") or os.path.join(_HERE, "libs4g_b200.so")  # override: A/B measurements only

if not os.path.exists(LIB_PATH):
    raise ImportError(
        "s4g_release_b200: %s is missing — build the CUDA library first "
        "(python -c 'import __graft_entry__ as g; g.build()' or python s4g_release_b200/build.py). "
        "There is no CPU fallback." % LIB_PATH)

lib = ctypes.CDLL(LIB_PATH)

_vp = ctypes.c_void_p
_i = ctypes.c_int
_f = ctypes.c_float
_d = ctypes.c_double
_ip = ctypes.POINTER(ctypes.c_int)
_ll = ctypes.c_longlong

_SIGNATURES = {
    "s4g_version": ([], _i),
    "s4g_last_error": ([], ctypes.c_char_p),
    "s4g_launch_count": ([], ctypes.c_ulonglong),
    "s4g_farthest_point_sample_f32": ([_vp, _i, _i, _i, _vp, _vp], _i),
    "s4g_farthest_point_sample_f32_i32": ([_vp, _i, _i, _i, _vp, _vp], _i),
    "s4g_fps_set_bucket_mode": ([_i], _i),
    "s4g_gather_points_f32": ([_vp, _vp, _i, _i, _i, _i, _vp, _vp], _i),
    "s4g_ball_query_f32": ([_vp, _vp, _i, _i, _i, _f, _i, _vp, _vp, _vp], _i),
    "s4g_ball_query_f32_i32": ([_vp, _vp, _i, _i, _i, _f, _i, _vp, _vp, _vp], _i),
    "s4g_ball_query_uses_grid": ([_i, _i, _f], _i),
    "s4g_ball_grid_build_f32": ([_vp, _i, _i, _f, _vp], _vp),
    "s4g_ball_query_with_grid_f32_i32": ([_vp, _vp, _vp, _i, _i, _vp, _vp, _vp], _i),
    "s4g_ball_grid_free": ([_vp, _vp], _i),
    "s4g_group_points_set_staged": ([_i], _i),
    "s4g_group_points_forward_f32": ([_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp], _i),
    "s4g_group_points_backward_f32": ([_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp], _i),
    "s4g_point_search_f32": ([_vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp], _i),
    "s4g_interpolate_forward_f32": ([_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp], _i),
    "s4g_interpolate_backward_f32": ([_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp], _i),
    "s4g_farthest_point_sample_f64_workspace": ([_i, _i], ctypes.c_size_t),
    "s4g_farthest_point_sample_f64": ([_vp, _i, _i, _i, _vp, _vp, ctypes.c_size_t, _vp], _i),
    "s4g_ball_query_f64": ([_vp, _vp, _i, _i, _i, _d, _i, _vp, _vp, _vp], _i),
    "s4g_group_points_forward_f64": ([_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp], _i),
    "s4g_group_points_backward_f64": ([_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp], _i),
    "s4g_point_search_f64": ([_vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp], _i),
    "s4g_interpolate_forward_f64": ([_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp], _i),
    "s4g_interpolate_backward_f64": ([_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp], _i),
    "s4g_three_nn_weights_f32_i32": ([_vp, _vp, _i, _i, _i, _vp, _vp, _vp], _i),
    "s4g_interp_concat_bf16": ([_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp], _i),
    "s4g_interp_concat_act_bf16": ([_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp], _i),
    "s4g_gather_xyz_f32_i32": ([_vp, _vp, _i, _i, _i, _vp, _vp], _i),
    "s4g_rows_segment_max_bf16": ([_vp, _i, _i, _i, _vp, _vp], _i),
    "s4g_broadcast_concat_bf16": ([_vp, _vp, _i, _i, _i, _i, _vp, _vp], _i),
    "s4g_local_eval_rows_bf16": ([_vp, _i, _i, _i, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp], _i),
    "s4g_linear_tf32": ([_vp, ctypes.c_longlong, _vp, ctypes.c_longlong, _vp, _vp, ctypes.c_longlong, ctypes.c_longlong,
                         _i, _i, _i, _i, _vp], _i),
    "s4g_gemm_bf16": ([_vp, _ll, _vp, _ll, _vp, _ll, _ll, _i, _i, _vp], _i),
    "s4g_gemm_bf16_set_weight_stationary": ([_i], _i),
    "s4g_gemm_bf16_set_epilogue_groups": ([_i], _i),
    "s4g_gemm_bf16_set_tile_n": ([_i], _i),
    "s4g_gemm_bf16_plan": ([_ll, _i, _i, _i, _i, _vp], _i),
    "s4g_gemm_bf16_bwd": ([_vp, _ll, _vp, _ll, _vp, _ll, _ll, _i, _i, _vp, _ll, _vp, _vp, _i, ctypes.c_uint, _f, _vp, _vp], _i),
    "s4g_gemm_bf16_stats": ([_vp, _ll, _vp, _ll, _vp, _ll, _ll, _i, _i, _vp, _vp], _i),
    "s4g_train_bn_finalize": ([_vp, _ll, _i, _vp, _vp, _f, _f, _vp, _vp, _vp, _vp], _i),
    "s4g_train_bn_bwd_finalize": ([_vp, _ll, _i, _vp, _vp, _vp, _vp, _vp, _vp], _i),
    "s4g_train_colstats_bf16": ([_vp, _ll, _ll, _i, _vp, _vp], _i),
    "s4g_train_bn_act_bf16": ([_vp, _vp, _vp, _vp, _ll, _i, _i, ctypes.c_uint, _f, _vp], _i),
    "s4g_train_bn_act_maxpool_bf16": ([_vp, _vp, _vp, _vp, _vp, _vp, _ll, _i, _i, _i, _vp], _i),
    "s4g_train_bn_bwd_reduce_bf16": ([_vp, _vp, _i, _vp, _vp, _vp, _ll, _i, _i, ctypes.c_uint, _f, _vp, _vp], _i),
    "s4g_train_bn_bwd_apply_bf16": ([_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _ll, _i, _i, ctypes.c_uint, _f, _vp, _vp], _i),
    "s4g_train_bn_act_segmax_bf16": ([_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _ll, _i, _i, _vp], _i),
    "s4g_train_bn_bwd_reduce_seg_bf16": ([_vp, _vp, _ll, _vp, _vp, _vp, _ll, _i, _i, _vp, _vp], _i),
    "s4g_train_bn_bwd_apply_seg_bf16": ([_vp, _vp, _ll, _vp, _vp, _vp, _vp, _vp, _vp, _ll, _i, _i, _vp, _vp], _i),
    "s4g_train_rows_segment_sum_bf16": ([_vp, _ll, _i, _ll, _i, _vp, _vp], _i),
    "s4g_train_group_rows_bf16":([_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp], _i),
    "s4g_train_group_rows_bwd": ([_vp, _ll, _vp, _i, _i, _i, _i, _i, _vp, _vp], _i),
    "s4g_train_interp_rows_bwd": ([_vp, _ll, _vp, _vp, _i, _i, _i, _i, _vp, _vp], _i),
    "s4g_train_relu_mask_rows_bf16": ([_vp, _vp, _vp, _vp, _ll, _i, _vp, _vp], _i),
    "s4g_train_index_inverse_count": ([_vp, _i, _i, _ll, _vp, _vp], _i),
    "s4g_train_index_inverse_fill": ([_vp, _i, _i, _ll, _vp, _vp, _vp], _i),
    "s4g_train_rows_bwd_gather": ([_vp, _ll, _vp, _vp, _vp, _vp, _i, _ll, _i, _i, _vp, _vp, _vp], _i),
    "s4g_train_f32_to_bf16": ([_vp, _vp, _ll, _vp], _i),
    "s4g_train_head_logits_fwd": ([_vp, _vp, _vp, _vp, _ll, _i, _i, _i, _vp], _i),
    "s4g_train_head_logits_bwd": ([_vp, _vp, _vp, _ll, _i, _i, _i, _vp], _i),
    "s4g_train_head_logits_dw": ([_vp, _vp, _vp, _vp, _ll, _i, _i, _i, _vp], _i),
    "s4g_train_sum_bf16": ([_vp, _vp, _vp, _vp, _vp, _ll, _vp], _i),
    "s4g_chain_create": ([_i, _ip, _ip, _ip, _i, _i, _i, _i, _i, _i], _vp),
    "s4g_chain_create_slots": ([_i, _ip, _ip, _ip, _i, _i, _i, _i, _i, _i, _i], _vp),
    "s4g_chain_create_tuned": ([_i, _ip, _ip, _ip, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i], _vp),
    "s4g_chain_create_tuned_in": ([_i, _ip, _ip, _ip, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i], _vp),
    "s4g_chain_destroy": ([_vp], None),
    "s4g_chain_weight_bytes": ([_vp], ctypes.c_size_t),
    "s4g_chain_cout_pad": ([_vp, _i], _i),
    "s4g_chain_info": ([_vp, _ip, _ip, _ip, _ip, _ip, _ip, _ip], _i),
    "s4g_chain_describe": ([_vp, ctypes.c_char_p, _i], _i),
    "s4g_chain_set_profile": ([_vp, _vp], _i),
    "s4g_chain_pack_weights": ([_vp, _i, _vp, _i, _i, _vp], _i),
    "s4g_chain_set_params": ([_vp, _vp, _vp], _i),
    "s4g_chain_set_xyz_layer": ([_vp, _vp, _i], _i),
    "s4g_chain_run_rows": ([_vp, _vp, _i, ctypes.c_longlong, _vp, _i, _vp], _i),
    "s4g_chain_run_gather": ([_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp], _i),
    "s4g_cloud_transform_select_f32": ([_vp, _i, _i, _vp, _i, _vp, _vp, _vp], _i),
    "s4g_voxel_keys_f32": ([_vp, _i, _vp, _f, _vp, _vp, _vp], _i),
    "s4g_voxel_means_f32": ([_vp, _i, _vp, _vp, _vp, _vp, _i, _vp], _i),
    "s4g_grasp_scores_f32": ([_vp, _i, _i, _i, _vp, _vp], _i),
    "s4g_grasp_select": ([_vp, _vp, _i, _i, _d, _d, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp], _i),
    "s4g_grasp_poses": ([_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp], _i),
    "s4g_grasp_collision_f32": ([_vp, _i, _vp, _i, _vp, _vp, _vp, _vp], _i),
    "s4g_grasp_nms": ([_vp, _vp, _i, _d, _vp, _vp, _vp], _i),
    "s4g_grasp_importance_sample": ([_vp, _i, _vp, _i, _vp, _vp, _vp], _i),
    "s4g_grasp_finish_batch_workspace": ([_i, _i], ctypes.c_size_t),
    "s4g_grasp_finish_batch": ([_vp, _vp, _vp, _i, _i, _vp, _i, _vp, _d, _vp, _i, _vp, ctypes.c_size_t, _vp, _vp, _vp, _vp,
                                _vp], _i),
}

for _name, (_args, _res) in _SIGNATURES.items():
    _fn = getattr(lib, _name)
    _fn.argtypes = _args
    _fn.restype = _res


def exported_symbols():
    return sorted(_SIGNATURES)


launches = 0  # number of C-ABI kernel launches issued by this process (bench.py reports it)


def check(status, what):
    """Non-zero status -> RuntimeError, as the reference's TORCH_CHECK macros raise."""
    global launches
    launches += 1
    if status != 0:
        msg = lib.s4g_last_error().decode("utf-8", "replace")
        raise RuntimeError("%s failed (status %d): %s" % (what, status, msg))


def stream_ptr(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def ptr(t):
    return ctypes.c_void_p(t.data_ptr())
