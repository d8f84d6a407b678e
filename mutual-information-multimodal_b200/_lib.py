"""ctypes binding of libmi_b200.so — one prototype per declaration in include/mi_b200.h."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmi_b200.so")

c_i64, c_int, c_f32, c_sz, c_vp = C.c_int64, C.c_int, C.c_float, C.c_size_t, C.c_void_p

# name -> (restype, argtypes): mirrors include/mi_b200.h (tests check every symbol is exported)
PROTOTYPES = {
    "mi_status_string": (C.c_char_p, [c_int]),
    "mi_last_cuda_error": (C.c_char_p, []),
    "mi_abi_version": (c_int, []),
    "mi_device_check": (c_int, []),
    "mi_launch_count": (c_i64, []),
    "mi_set_profiling": (None, [c_int]),
    "mi_profile_read": (c_int, [c_vp, c_vp]),
    "mi_profile_read_kinds": (c_int, [c_vp, c_vp, c_int]),
    "mi_set_cta_group": (None, [c_int]),
    "mi_set_ref_sample_columns": (None, [c_i64]),
    "mi_set_overlap_reserve_sms": (None, [c_int]),
    "mi_set_mlp_panel_pairs": (None, [c_i64]),
    "mi_set_mlp_mode": (None, [c_int]),
    "mi_get_mlp_mode": (c_int, []),
    "mi_plan_ksplit": (c_int, [c_i64, c_int, c_i64]),
    "mi_plan_mlp_walk": (c_i64, [c_i64, c_i64, c_i64, c_vp, c_i64]),
    "mi_get_cta_group": (c_int, []),
    "mi_gemm_bf16": (c_int, [c_vp, c_i64, c_int, c_vp, c_i64, c_int, c_i64, c_i64, c_i64, c_f32, c_f32, c_vp, c_i64,
                             c_vp, c_i64, c_vp, c_i64, c_int, c_vp]),
    "mi_gemm_bf16_mn_workspace_bytes": (c_sz, [c_i64, c_i64, c_i64, c_int, c_int, c_int, c_int]),
    "mi_gemm_bf16_mn": (c_int, [c_vp, c_i64, c_int, c_int, c_vp, c_i64, c_int, c_int, c_i64, c_i64, c_i64,
                                c_vp, c_i64, c_vp, c_i64, c_int, c_vp, c_sz, c_vp]),
    "mi_transpose_bf16": (c_int, [c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_vp]),
    "mi_cast_f32_to_bf16": (c_int, [c_vp, c_vp, c_i64, c_vp]),
    "mi_score_stats_workspace_bytes": (c_sz, [c_i64, c_i64, c_i64]),
    "mi_score_stats_rc_workspace_bytes": (c_sz, [c_i64, c_i64, c_i64]),
    "mi_score_stats_rc": (c_int, [c_vp, c_i64, c_int, c_vp, c_i64, c_int, c_vp, c_vp, c_i64, c_i64, c_i64, c_i64, c_f32,
                                  c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "mi_score_stats": (c_int, [c_vp, c_i64, c_int, c_vp, c_i64, c_int, c_vp, c_vp, c_i64, c_i64, c_i64, c_i64, c_f32,
                               c_vp, c_vp, c_vp, c_sz, c_vp]),
    "mi_score_grad_workspace_bytes": (c_sz, [c_i64, c_i64, c_i64, c_int]),
    "mi_score_grad": (c_int, [c_vp, c_i64, c_int, c_vp, c_i64, c_int, c_vp, c_vp, c_i64, c_i64, c_i64, c_i64, c_f32,
                              c_vp, c_f32, c_vp, c_f32, c_int, c_int, c_f32, c_f32,
                              c_vp, c_vp, c_i64, c_int, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "mi_score_ref_sample_workspace_bytes": (c_sz, [c_i64, c_i64, c_i64, c_i64]),
    "mi_ref_sample_stride": (c_i64, [c_i64, c_i64, c_i64]),
    "mi_score_ref_sample": (c_int, [c_vp, c_i64, c_int, c_vp, c_i64, c_int, c_vp, c_vp, c_i64, c_i64, c_i64, c_i64, c_f32,
                                    c_int, c_i64, c_i64, c_i64, c_int, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "mi_score_single_pass_workspace_bytes": (c_sz, [c_i64, c_i64, c_i64, c_int]),
    "mi_row_norm_max": (c_int, [c_vp, c_i64, c_int, c_i64, c_i64, c_vp, c_vp, c_vp]),
    "mi_score_single_pass": (c_int, [c_vp, c_i64, c_int, c_vp, c_i64, c_int, c_vp, c_vp, c_i64, c_i64, c_i64, c_i64, c_f32,
                                     c_int, c_int, c_f32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                     c_vp, c_int, c_vp, c_sz, c_vp]),
    "mi_merge_scalars": (c_int, [c_vp, c_int, c_i64, c_int, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mi_single_finalize_q": (c_int, [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_int, c_f32, c_f32, c_vp, c_i64, c_int,
                                     c_vp, c_vp, c_i64, c_int, c_vp]),
    "mi_single_finalize_k": (c_int, [c_vp, c_i64, c_i64, c_vp, c_vp, c_int, c_f32, c_f32, c_vp, c_i64, c_int, c_vp]),
    "mi_critic_workspace_bytes": (c_sz, [c_i64, c_i64, c_int, c_int, c_int, c_int]),
    "mi_critic_loss_fwd_bwd": (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_int, c_int, c_int, c_f32,
                                       c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "mi_critic_loss_fwd_bwd_from_host": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_i64, c_i64, c_int, c_int, c_int, c_f32,
                                                 c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "mi_dist_ctx_create": (c_int, [c_vp, c_vp]),
    "mi_dist_ctx_destroy": (None, [c_vp]),
    "mi_dist_ctx_info": (c_int, [c_vp, c_vp, c_vp]),
    "mi_sharded_critic_workspace_bytes": (c_sz, [c_i64, c_int, c_i64, c_int, c_int, c_int]),
    "mi_sharded_critic_loss_fwd_bwd": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_int, c_int, c_int, c_f32,
                                               c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_int, c_vp]),
    "mi_mlp_critic_workspace_bytes": (c_sz, [c_i64, c_i64, c_i64, c_i64, c_int]),
    "mi_mlp_critic_loss_fwd_bwd": (c_int, [c_vp] * 9 + [c_i64, c_i64, c_i64, c_i64, c_int, c_int] + [c_vp] * 10 + [c_vp, c_sz, c_vp]),
    "mi_mlp_block_workspace_bytes": (c_sz, [c_i64, c_i64, c_i64, c_i64, c_i64, c_int]),
    "mi_mlp_block_state_bytes": (c_sz, [c_i64, c_i64, c_i64, c_i64, c_i64, c_int]),
    "mi_mlp_block_ref_logit": (c_int, [c_vp] * 8 + [c_i64] * 6 + [c_int, c_vp, c_vp, c_sz, c_vp]),
    "mi_mlp_block_fwd": (c_int, [c_vp] * 10 + [c_i64] * 6 + [c_int, c_int, c_vp, c_int, c_vp, c_vp, c_sz, c_vp, c_sz, c_vp]),
    "mi_mlp_block_fwd_rc": (c_int, [c_vp] * 10 + [c_i64] * 6 + [c_int, c_int, c_vp, c_int, c_vp, c_vp, c_vp, c_sz, c_vp, c_sz,
                                                               c_vp]),
    "mi_mlp_block_merge": (c_int, [c_vp, c_int, c_i64, c_int, c_int, c_vp, c_vp, c_vp]),
    "mi_mlp_block_bwd": (c_int, [c_vp] * 10 + [c_i64] * 6 + [c_int, c_int, c_int, c_vp, c_vp, c_vp, c_sz] + [c_vp] * 8
                         + [c_vp, c_sz, c_vp]),
    "mi_mlp_block_bwd_rc": (c_int, [c_vp] * 10 + [c_i64] * 6 + [c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_sz] + [c_vp] * 8
                            + [c_vp, c_sz, c_vp]),
    "mi_mlp_input_grad_workspace_bytes": (c_sz, [c_i64, c_i64, c_i64, c_int]),
    "mi_mlp_input_grad": (c_int, [c_vp, c_vp, c_vp, c_int, c_i64, c_i64, c_i64, c_int, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "mi_gdv_workspace_bytes": (c_sz, [c_i64, c_i64, c_i64, c_int]),
    "mi_gdv": (c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_vp, c_sz, c_vp]),
    "mi_critic_host_scratch_bytes": (c_sz, [c_i64, c_i64, c_int, c_int, c_int, c_int]),
    "mi_critic_loss_fwd_bwd_host": (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_int, c_int, c_int, c_f32,
                                            c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
}

_lib = None


def load():
    """Loads libmi_b200.so (no fallback: raises if it has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc -gencode arch=compute_100a,code=sm_100a). There is no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib
