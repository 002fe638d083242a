"""ctypes binding of the C ABI in include/hzb200.h (hanabizero_b200/csrc/libhzb200.so).

There is no CPU fallback: if the library is missing the import of any product module fails with
a build hint, and every non-zero status from the library raises.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "csrc", "libhzb200.so")

HZ_OK, HZ_ERR_ARG, HZ_ERR_CUDA, HZ_ERR_STATE, HZ_ERR_ILLEGAL = 0, -1, -2, -3, -4


class HzError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__(f"libhzb200 status {status}: {msg}")
        self.status = status


class IllegalMoveError(HzError, ValueError):
    pass


_vp, _i, _f, _i64 = C.c_void_p, C.c_int, C.c_float, C.c_int64

# name -> (restype, argtypes); mirrors include/hzb200.h one to one (tests/test_abi.py checks that
# every function the header declares is listed here and exported by the library)
SIGNATURES = {
    "hz_last_error": (C.c_char_p, []),
    "hz_version": (_i, []),
    "hz_launch_count": (_i64, []),
    "hz_trees_create": (_i, [C.POINTER(_vp), _i, _i, _i, _i]),
    "hz_trees_destroy": (_i, [_vp]),
    "hz_trees_num": (_i, [_vp]),
    "hz_trees_actions": (_i, [_vp]),
    "hz_trees_capacity": (_i, [_vp]),
    "hz_trees_prepare": (_i, [_vp, _vp, _f, _vp, _vp, _vp, _vp]),
    "hz_trees_traverse": (_i, [_vp, _vp, _i, _f, _f, _vp, _f, _vp, _vp, _vp, _vp, _vp, _vp, _i]),
    "hz_trees_backprop": (_i, [_vp, _vp, _i, _f, _vp, _vp, _vp, _i, _vp]),
    "hz_trees_backprop_traverse": (_i, [_vp, _vp, _i, _f, _vp, _vp, _vp, _i, _vp, _f, _i, _f,
                                        _vp, _vp, _vp, _vp, _vp, _vp, _i]),
    "hz_trees_search_step": (_i, [_vp, _vp, _i, _i, _vp]),
    "hz_gemm_plan_create": (_i, [C.POINTER(_vp), _i, _i, _vp, _i]),
    "hz_gemm_plan_destroy": (_i, [_vp]),
    "hz_gemm_plan_steps": (_i, [_vp]),
    "hz_gemm_plan_set_operand": (_i, [_vp, _i, _i, _vp]),
    "hz_gemm_plan_set_sm_target": (_i, [_vp, _i]),
    "hz_gemm_launch_count": (_i64, []),
    "hz_gemm_plan_run": (_i, [_vp, _vp, _i, _i]),
    "hz_rowchain_create": (_i, [C.POINTER(_vp), _i, _vp, _i, _vp, _i64, _vp, _vp]),
    "hz_rowchain_create_small": (_i, [C.POINTER(_vp), _i, _vp, _i, _vp, _i64, _vp, _vp]),
    "hz_rowchain_destroy": (_i, [_vp]),
    "hz_rowchain_set_state": (_i, [_vp, _vp]),
    "hz_rowchain_run": (_i, [_vp, _vp]),
    "hz_rowchain_grid": (_i, [_vp]),
    "hz_rowchain_set_trace": (_i, [_vp, _i]),
    "hz_rowchain_read_trace": (_i, [_vp, _vp, _i64]),
    "hz_trees_set_progress": (_i, [_vp, _i]),
    "hz_trees_set_tie_break": (_i, [_vp, _i, C.c_uint64, _i]),
    "hz_trees_root_stats": (_i, [_vp, _vp, _vp, _vp]),
    "hz_trees_trajectories": (_i, [_vp, _vp, _vp, _i]),
    "hz_trees_export": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "hz_gather_hidden": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i]),
    "hz_support_decode": (_i, [_vp, _vp, _i, _vp, _vp, _i, _i, _i64, _f]),
    "hz_dirichlet_noise": (_i, [_vp, _vp, _i, _i, C.c_double, C.c_uint64, C.c_uint32, C.c_uint32, _vp]),
    "hz_host_dirichlet_noise": (_i, [_vp, _i, _i, C.c_double, C.c_uint64, C.c_uint32, C.c_uint32, _vp]),
    "hz_select_action": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp]),
    "hz_stack_push": (_i, [_vp, _vp, _vp, _i64, _vp, _i, _i, _i]),
    "hz_ring_gather": (_i, [_vp, _vp, _i, _vp, _i64, _i, _i, _i, _i, _i]),
    "hz_ring_refill": (_i, [_vp, _vp, _i, _vp, _i, _i, _i]),
    "hz_traj_begin": (_i, [_vp, _vp, _vp, _i64, _vp, _vp]),
    "hz_traj_append": (_i, [_vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hz_traj_record_u8": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _i64, _vp, _vp]),
    "hz_traj_pack": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hz_visit_policy": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp]),
    "hz_envs_create": (_i, [C.POINTER(_vp), _i, _i, _i, _vp]),
    "hz_envs_destroy": (_i, [_vp]),
    "hz_envs_dims": (_i, [_vp, _vp]),
    "hz_envs_reset": (_i, [_vp, _vp, _vp]),
    "hz_envs_step": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hz_envs_observe": (_i, [_vp, _vp, _vp, _i64, _vp, _i64, _vp]),
    "hz_envs_step_observe": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _i64, _vp, _i64, _vp]),
    "hz_envs_observe_u8": (_i, [_vp, _vp, _vp, _i64, _vp, _i64, _vp]),
    "hz_envs_step_observe_u8": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _i64, _vp, _i64, _vp]),
    "hz_envs_step_observe_u8_terminal": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _i64, _vp, _vp, _i64,
                                              _vp]),
    "hz_envs_step_observe_bits": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _i64, _vp]),
    "hz_envs_host_step": (_i, [_vp, _vp, _vp, _i, _vp, _i64, _vp]),
    "hz_envs_host_wait": (_i, [_vp]),
    "hz_envs_set_random_policy": (_i, [_vp, _vp, _vp, C.c_uint64]),
    "hz_host_random_legal": (_i, [_vp, _i64, _i, _i, _i, C.c_uint64, C.c_uint32, _vp]),
    "hz_envs_check": (_i, [_vp, _vp, _vp]),
    "hz_envs_dump": (_i, [_vp, _vp, _vp]),
    "hz_wave_pack": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "hz_wave_unpack": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _vp]),
    "hz_obs_pack": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "hz_obs_pack_windows": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _vp, _i, _vp, _vp, _vp]),
    "hz_wave_policy": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _vp]),
    "hz_obs_pack_episodes": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _vp, _i, _vp, _vp, _vp]),
}



class SearchIO(C.Structure):
    """struct hz_search_io (include/hzb200.h)."""
    _fields_ = [("value_logits", _vp), ("ld_value", _i64), ("reward_logits", _vp), ("ld_reward", _i64),
                ("policy_logits", _vp), ("ld_policy", _i64), ("next_state", _vp), ("ld_state", _i64),
                ("support", _vp), ("support_width", C.c_int32), ("support_delta", _f), ("elem_bytes", C.c_int32),
                ("sanitize_nan", C.c_int32), ("pool", _vp), ("state_cols", C.c_int32), ("out_batch", _vp),
                ("ld_batch", _i64), ("onehot_cols", C.c_int32), ("out_ix", _vp), ("out_action", _vp),
                ("minmax", _vp), ("value_delta_max", _f), ("discount", _f), ("pb_c_base", C.c_int32),
                ("pb_c_init", _f), ("programmatic_launch", C.c_int32), ("stage_limit", C.c_int32)]


class TrajView(C.Structure):
    """struct hz_traj_view (include/hzb200.h)."""
    _fields_ = [("obs", _vp), ("legal", _vp), ("action", _vp), ("reward", _vp), ("visits", _vp), ("root_value", _vp),
                ("len", _vp), ("bank", _vp), ("finished", _vp), ("overflow", _vp), ("num", C.c_int32),
                ("obs_dim", C.c_int32), ("actions", C.c_int32), ("stack", C.c_int32), ("max_len", C.c_int32), ("banks", C.c_int32)]


class RowChainWeights(C.Structure):
    """struct hz_rowchain_weights (include/hzb200.h)."""
    _fields_ = [("w1", _vp), ("ld_w1", _i64), ("w1a_t", _vp), ("b1", _vp), ("w2", _vp), ("b2", _vp), ("w3", _vp),
                ("b3", _vp), ("wh1", _vp), ("bh1", _vp), ("wb2", _vp), ("bb2", _vp), ("wa2", _vp), ("ba2", _vp),
                ("wb3", _vp), ("bb3", _vp), ("state_cols", C.c_int32), ("head_cols", C.c_int32),
                ("onehot_cols", C.c_int32), ("logit_cols", C.c_int32)]


class GemmStep(C.Structure):
    """struct hz_gemm_step (include/hzb200.h)."""
    _fields_ = [("a", _vp), ("lda", _i64), ("stride_a", _i64), ("w", _vp), ("ldw", _i64), ("stride_w", _i64),
                ("bias", _vp), ("stride_bias", _i64), ("c", _vp), ("ldc", _i64), ("stride_c", _i64),
                ("d", _vp), ("ldd", _i64), ("stride_d", _i64), ("m", C.c_int32), ("n", C.c_int32),
                ("k", C.c_int32), ("batch", C.c_int32), ("relu", C.c_int32)]


class WaveTicket(C.Structure):
    """struct hz_wave_ticket (include/hzb200.h)."""
    _fields_ = [("noise", _vp), ("reward", _vp), ("logits", _vp), ("legal", _vp), ("hidden", _vp),
                ("out_visits", _vp), ("out_values", _vp)]


class PolicyTicket(C.Structure):
    """struct hz_policy_ticket (include/hzb200.h)."""
    _fields_ = [("mask", _vp), ("out", _vp)]


HZ_OBS_F32, HZ_OBS_U8, HZ_OBS_BITS = 0, 1, 2
HZ_LEGAL_I32, HZ_LEGAL_F32, HZ_LEGAL_MASK = 0, 1, 2


class ObsTicket(C.Structure):
    """struct hz_obs_ticket (include/hzb200.h)."""
    _fields_ = [("obs", _vp), ("ld_obs", _i64), ("legal", _vp), ("ld_legal", _i64), ("noise", _vp),
                ("obs_format", C.c_int32), ("legal_format", C.c_int32)]


class EpisodeTicket(C.Structure):
    """struct hz_obs_episode_ticket (include/hzb200.h)."""
    _fields_ = [("frames", _vp), ("ld_frames", _i64), ("legal", _vp), ("samples", _vp), ("noise", _vp), ("mask", _vp)]


class ObsLayout(C.Structure):
    """struct hz_obs_layout (include/hzb200.h)."""
    _fields_ = [("stack", C.c_int32), ("frame_dim", C.c_int32), ("frame_stride", C.c_int32), ("elem_bytes", C.c_int32),
                ("frame_words", C.c_int32), ("bit_offset", C.c_int32)]


_lib = None


def load():
    """dlopen libhzb200.so once and type every entry point."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m hanabizero_b200.build` "
            "(nvcc, sm_100a). hanabizero_b200 has no CPU fallback.")
    import torch  # noqa: F401  (brings libcublasLt.so.12 and the CUDA runtime libraries into the process)
    lib = C.CDLL(LIB_PATH)
    missing = [name for name in SIGNATURES if not hasattr(lib, name)]
    if missing:
        raise ImportError(f"{LIB_PATH} does not export {missing}: stale build, rerun "
                          "`python -m hanabizero_b200.build --force`")
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status):
    if status == HZ_OK:
        return
    msg = load().hz_last_error().decode("utf-8", "replace")
    if status == HZ_ERR_ILLEGAL:
        raise IllegalMoveError(status, msg)
    raise HzError(status, msg)


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def stream_ptr(device=None):
    import torch
    return torch.cuda.current_stream(device).cuda_stream


def launch_count():
    """Kernels of this library launched so far (own CUDA kernels; cuBLASLt GEMMs are counted apart)."""
    return int(load().hz_launch_count())


def gemm_launch_count():
    return int(load().hz_gemm_launch_count())
