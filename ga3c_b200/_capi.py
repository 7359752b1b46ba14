"""ctypes binding of include/ga3c_b200.h.  Loading fails loudly: there is no fallback path."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GA3C_LIB") or os.path.join(_HERE, "_lib", "libga3c_b200.so")     # GA3C_LIB: A/B runs of two builds on one box


# the optimizer and loss fields both network configs end with
_CONFIG_TAIL = [("rmsprop_decay", C.c_float), ("rmsprop_momentum", C.c_float), ("rmsprop_epsilon", C.c_float),
                ("log_epsilon", C.c_float), ("min_policy", C.c_float), ("use_log_softmax", C.c_int32),
                ("use_grad_clip", C.c_int32), ("grad_clip_norm", C.c_float), ("dual_rmsprop", C.c_int32)]


class ga3c_config(C.Structure):
    _fields_ = [("device", C.c_int32), ("num_actions", C.c_int32), ("max_batch", C.c_int32)] + _CONFIG_TAIL + [
        ("image_height", C.c_int32), ("image_width", C.c_int32), ("stacked_frames", C.c_int32)]


class ga3c_mlp_config(C.Structure):
    _fields_ = [("device", C.c_int32), ("kind", C.c_int32), ("state_dim", C.c_int32), ("num_actions", C.c_int32),
                ("max_batch", C.c_int32), ("n_dense", C.c_int32), ("dense_width", C.c_int32 * 8)] + _CONFIG_TAIL


class ga3c_batcher_config(C.Structure):
    _fields_ = [("device", C.c_int32), ("num_agents", C.c_int32), ("state_bytes", C.c_int32), ("x_u8", C.c_int32),
                ("max_batch", C.c_int32), ("num_actions", C.c_int32), ("states", C.c_void_p), ("pending", C.c_void_p),
                ("reply_p", C.c_void_p), ("reply_v", C.c_void_p), ("work_sem", C.c_void_p), ("wake_sems", C.POINTER(C.c_void_p))]


MLP_FORK_VP, MLP_DISCRATE = 0, 1

# name -> (restype, argtypes); the single source the symbol-export test checks against the header
SIGNATURES = {
    "ga3c_last_error": (C.c_char_p, []),
    "ga3c_abi_version": (C.c_int, []),
    "ga3c_create": (C.c_int, [C.POINTER(ga3c_config), C.POINTER(C.c_void_p)]),
    "ga3c_destroy": (C.c_int, [C.c_void_p]),
    "ga3c_reserve": (C.c_int, [C.c_void_p, C.c_int32]),
    "ga3c_param_count": (C.c_int, [C.c_void_p]),
    "ga3c_param_info": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_int64),
                                  C.POINTER(C.c_int32), C.POINTER(C.c_int64)]),
    "ga3c_arena_floats": (C.c_int64, [C.c_void_p]),
    "ga3c_arena_ptrs": (C.c_int, [C.c_void_p] + [C.POINTER(C.c_void_p)] * 4),
    "ga3c_arena_upload": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64]),
    "ga3c_arena_download": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64]),
    "ga3c_global_step": (C.c_int64, [C.c_void_p]),
    "ga3c_set_global_step": (C.c_int, [C.c_void_p, C.c_int64]),
    "ga3c_predict": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ga3c_forward_backward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float,
                                        C.c_void_p, C.c_void_p]),
    "ga3c_fb_head": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float, C.c_void_p, C.c_void_p]),
    "ga3c_fb_tail": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "ga3c_apply_rmsprop": (C.c_int, [C.c_void_p, C.c_float, C.c_void_p]),
    "ga3c_dp_handle_bytes": (C.c_int, []),
    "ga3c_dp_export": (C.c_int, [C.c_void_p, C.c_void_p]),
    "ga3c_dp_attach": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "ga3c_dp_detach": (C.c_int, [C.c_void_p]),
    "ga3c_stage_h2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_void_p]),
    "ga3c_dp_attach_local": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]),
    "ga3c_dp_error": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32)]),
    "ga3c_train_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float, C.c_float,
                                  C.c_void_p, C.c_void_p]),
    "ga3c_arena_ptr": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "ga3c_dual_forward_backward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float,
                                             C.c_void_p, C.c_void_p]),
    "ga3c_dual_forward_backward_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float,
                                                C.c_void_p, C.c_void_p]),
    "ga3c_dual_apply": (C.c_int, [C.c_void_p, C.c_float, C.c_void_p]),
    "ga3c_lock": (C.c_int, [C.c_void_p]),
    "ga3c_unlock": (C.c_int, [C.c_void_p]),
    "ga3c_batcher_create": (C.c_int, [C.c_void_p, C.POINTER(ga3c_batcher_config), C.POINTER(C.c_void_p)]),
    "ga3c_batcher_start": (C.c_int, [C.c_void_p]),
    "ga3c_batcher_stop": (C.c_int, [C.c_void_p]),
    "ga3c_batcher_stats": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int32)]),
    "ga3c_batcher_destroy": (C.c_int, [C.c_void_p]),
    "ga3c_predict_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ga3c_forward_backward_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float,
                                           C.c_void_p, C.c_void_p]),
    "ga3c_fb_head_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float, C.c_void_p, C.c_void_p]),
    "ga3c_fb_tail_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "ga3c_train_step_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float, C.c_float,
                                     C.c_void_p, C.c_void_p]),
    "ga3c_returns": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_double, C.c_int32, C.c_double,
                               C.c_double, C.c_void_p, C.c_void_p]),
    "ga3c_select_actions": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "ga3c_workspace_ptr": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]),
    "ga3c_keep_dn1": (C.c_int, [C.c_void_p, C.c_int32]),
    "ga3c_launch_count": (C.c_int64, [C.c_void_p]),
    "ga3c_kernel_count": (C.c_int, []),
    "ga3c_kernel_name": (C.c_char_p, [C.c_int]),
    "ga3c_timing_enable": (C.c_int, [C.c_void_p, C.c_int32]),
    "ga3c_timing_collect": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.c_int32]),
    "ga3c_evt_begin": (C.c_int, [C.c_void_p]),
    "ga3c_evt_end": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64), C.c_int32, C.POINTER(C.c_int32)]),
    "ga3c_trace_begin": (C.c_int, [C.c_void_p, C.c_void_p]),
    "ga3c_trace_end": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64), C.c_int32]),
    "ga3c_mlp_create": (C.c_int, [C.POINTER(ga3c_mlp_config), C.POINTER(C.c_void_p)]),
    "ga3c_mlp_destroy": (C.c_int, [C.c_void_p]),
    "ga3c_mlp_reserve": (C.c_int, [C.c_void_p, C.c_int32]),
    "ga3c_mlp_param_count": (C.c_int, [C.c_void_p]),
    "ga3c_mlp_param_info": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_int64),
                                      C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(C.c_int32)]),
    "ga3c_mlp_arena_floats": (C.c_int64, [C.c_void_p]),
    "ga3c_mlp_arena_upload": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64]),
    "ga3c_mlp_arena_download": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64]),
    "ga3c_mlp_global_step": (C.c_int64, [C.c_void_p]),
    "ga3c_mlp_set_global_step": (C.c_int, [C.c_void_p, C.c_int64]),
    "ga3c_mlp_predict": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ga3c_mlp_forward_backward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float,
                                            C.c_void_p, C.c_void_p]),
    "ga3c_mlp_apply_rmsprop": (C.c_int, [C.c_void_p, C.c_float, C.c_void_p]),
    "ga3c_mlp_train_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float, C.c_float,
                                      C.c_void_p, C.c_void_p]),
    "ga3c_mlp_launch_count": (C.c_int64, [C.c_void_p]),
    "ga3c_mlp_workspace_ptr": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_int32)]),
    "ga3c_debug_tf32x3_gemm": (C.c_int, [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                         C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "ga3c_histograms": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ga3c_debug_histogram": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ga3c_mlp_histogram_count": (C.c_int, [C.c_void_p]),
    "ga3c_mlp_histograms": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ga3c_mlp_timing_enable": (C.c_int, [C.c_void_p, C.c_int32]),
    "ga3c_mlp_timing_collect": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.c_int32]),
}

RET_DISCOUNTING, RET_INTERMEDIATE, RET_CLIPPING, RET_NSTEP = 1, 2, 4, 8

_lib = None


class Ga3cError(RuntimeError):
    pass


def load():
    """dlopen the C-ABI library (ctypes.CDLL releases the GIL around every call)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise Ga3cError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)        # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().ga3c_last_error()
        raise Ga3cError(f"{what} failed (rc={rc}): {msg.decode() if msg else '?'}")
