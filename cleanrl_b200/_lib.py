"""ctypes binding of libb200rl.so (the C-ABI declared in include/b200rl.h).

The library is the product: there is NO fallback.  If it is missing or a call
fails, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "libb200rl.so"

_p = C.c_void_p
_i64 = C.c_int64
_i = C.c_int
_d = C.c_double
_sz = C.c_size_t

# name -> (restype, argtypes)   -- must list every symbol include/b200rl.h declares
SIGNATURES = {
    "b200rl_version": (_i, []),
    "b200rl_last_error": (C.c_char_p, []),
    "b200rl_compiled_arch": (_i, []),
    "b200rl_launch_count": (C.c_longlong, []),
    "b200rl_profile_enable": (None, [_i]),
    "b200rl_profile_reset": (None, []),
    "b200rl_profile_summary": (_i, [C.c_char_p, _sz]),
    "b200rl_gae_f32": (_i, [_p, _p, _p, _p, _p, _p, _p, _i64, _i64, _d, _d, _i, _p]),
    "b200rl_categorical_sample_f32": (_i, [_p, _i64, _p, _p, _i64, _i64, _i, _p, _p, _p, _p, _p]),
    "b200rl_categorical_eval_f32": (_i, [_p, _i64, _p, _i64, _i, _p, _p, _p]),
    "b200rl_ppo_loss_workspace_bytes": (_sz, [_i64]),
    "b200rl_ppo_loss_f32": (_i, [_p, _i64, _p, _i64, _p, _p, _p, _p, _p, _p, _i64, _i, _d, _d, _d, _i, _i,
                                 _p, _i64, _p, _i64, _p, _p, _sz, _p]),
    "b200rl_gaussian_sample_f32": (_i, [_p, _i64, _p, _p, _p, _i64, _i64, _i, _p, _p, _p, _p, _p]),
    "b200rl_gaussian_eval_f32": (_i, [_p, _i64, _p, _p, _i64, _i, _p, _p, _p]),
    "b200rl_ppo_loss_gaussian_workspace_bytes": (_sz, [_i64]),
    "b200rl_ppo_loss_gaussian_f32": (_i, [_p, _i64, _p, _p, _i64, _p, _p, _p, _p, _p, _p, _i64, _i, _d, _d, _d, _i, _i,
                                          _p, _i64, _p, _p, _i64, _p, _p, _sz, _p]),
    "b200rl_clip_adam_workspace_bytes": (_sz, [_i64]),
    "b200rl_clip_adam_f32": (_i, [_p, _p, _p, _p, _i64, _i64, _d, _d, _d, _d, _d, _i, _p, _p, _sz, _p]),
    "b200rl_adam_step_scalars": (_i, [_i64, _d, _d, _d, _p]),
    "b200rl_clip_adam_dyn_f32": (_i, [_p, _p, _p, _p, _i64, _p, _d, _d, _d, _d, _i, _p, _p, _sz, _p]),
    "b200rl_conv2d_fwd_f32": (_i, [_p, _i, _p, _d, _p, _p, _p, _i64, _i, _i, _i, _i, _i, _i, _i, _i, _p]),
    "b200rl_conv2d_bwd_data_f32": (_i, [_p, _p, _p, _i, _p, _i64, _i, _i, _i, _i, _i, _i, _i, _p]),
    "b200rl_conv2d_bwd_weight_workspace_bytes": (_sz, [_i64, _i, _i, _i, _i, _i, _i, _i]),
    "b200rl_conv2d_bwd_weight_f32": (_i, [_p, _i, _p, _d, _p, _p, _p, _i64, _i, _i, _i, _i, _i, _i, _i, _p, _sz, _p]),
    "b200rl_conv2d_fwd_pad_f32": (_i, [_p, _i, _p, _d, _p, _p, _p, _i64, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p]),
    "b200rl_conv2d_bwd_data_pad_f32": (_i, [_p, _p, _p, _i, _p, _i64, _i, _i, _i, _i, _i, _i, _i, _i, _p]),
    "b200rl_conv2d_bwd_weight_pad_workspace_bytes": (_sz, [_i64, _i, _i, _i, _i, _i, _i, _i, _i]),
    "b200rl_conv2d_bwd_weight_pad_f32": (_i, [_p, _i, _p, _d, _p, _p, _p, _i64, _i, _i, _i, _i, _i, _i, _i, _i, _p, _sz, _p]),
    "b200rl_maxpool3s2_fwd_f32": (_i, [_p, _i64, _i, _i, _p, _p, _p]),
    "b200rl_maxpool3s2_bwd_f32": (_i, [_p, _p, _i64, _i, _i, _p, _p]),
    "b200rl_relu_f32": (_i, [_p, _i64, _p, _p]),
    "b200rl_relu_bwd_f32": (_i, [_p, _p, _p, _i64, _p, _p]),
    "b200rl_add_f32": (_i, [_p, _p, _i64, _p, _p]),
    "b200rl_nhwc_to_nchw_u8": (_i, [_p, _p, _i64, _i, _i, _i, _p, _p]),
    "b200rl_linear_fwd_f32": (_i, [_p, _p, _p, _p, _p, _i64, _i, _i, _i, _p]),
    "b200rl_linear_bwd_data_f32": (_i, [_p, _p, _p, _i, _p, _i64, _i, _i, _p]),
    "b200rl_linear_bwd_weight_workspace_bytes": (_sz, [_i64, _i, _i]),
    "b200rl_linear_bwd_weight_f32": (_i, [_p, _p, _p, _p, _p, _i64, _i, _i, _p, _sz, _p]),
    "b200rl_dqn_td_loss_workspace_bytes": (_sz, [_i64]),
    "b200rl_dqn_td_loss_f32": (_i, [_p, _i64, _p, _i64, _p, _p, _p, _i64, _i, _d, _i, _p, _i64, _p, _p, _sz, _p]),
    "b200rl_argmax_f32": (_i, [_p, _i64, _i64, _i, _p, _p]),
    "b200rl_naturecnn_param_count": (_i64, [_i]),
    "b200rl_naturecnn_bf16_packed_bytes": (_sz, [_i]),
    "b200rl_naturecnn_bf16_acts_bytes": (_sz, [_i64, _i]),
    "b200rl_frames_to_s2d_bf16": (_i, [_p, _p, _i64, _p, _p]),
    "b200rl_naturecnn_bf16_workspace_bytes": (_sz, [_i64, _i]),
    "b200rl_naturecnn_bf16_pack": (_i, [_p, _i, _p, _p]),
    "b200rl_naturecnn_bf16_forward": (_i, [_p, _i, _p, _i64, _i, _p, _p, _p, _p, _p]),
    "b200rl_naturecnn_bf16_rollout_step": (_i, [_p, _p, _p, _i64, _i, _p, _p, _p, _p, _p, _p, _p, _p]),
    "b200rl_naturecnn_bf16_backward": (_i, [_p, _p, _i, _p, _i64, _i, _p, _p, _p, _p, _p, _p, _sz, _p, _p]),
    "b200rl_frames_to_s2d_u8": (_i, [_p, _p, _i64, _p, _p, _p]),
    "b200rl_lstm_mask_state_f32": (_i, [_p, _p, _p, _i64, _i, _p, _p, _p]),
    "b200rl_lstm_cell_fwd_f32": (_i, [_p, _p, _p, _i64, _i, _p, _p, _p, _p]),
    "b200rl_lstm_cell_bwd_f32": (_i, [_p, _p, _p, _p, _p, _p, _p, _i64, _i, _p, _p, _p]),
    "b200rl_naturecnn_grad_tail_offset": (_i64, [_i]),
    "b200rl_frames_delta_s2d_u8": (_i, [_p, _p, _p, _p, _p, _i64, _p, _p, _p]),
    "b200rl_h2d_rows_async": (_i, [_p, _p, _i64, _i64, _i64, _p]),
    "b200rl_stackdelta_create": (_p, [_i64, _i, _i64, _i]),
    "b200rl_stackdelta_destroy": (None, [_p]),
    "b200rl_stackdelta_invalidate": (None, [_p]),
    "b200rl_stackdelta_begin": (_i64, [_p, _p, _i64, _p, _p, _p, _p]),
    "b200rl_stackdelta_wait": (_i64, [_p, _p]),
    "b200rl_mt19937_shuffle_i64": (_i, [_p, _p, _p, _i64]),
    "b200rl_stackdelta_launch": (_i64, [_p, _p, _i64, _p]),
    "b200rl_stackdelta_join": (_i64, [_p, _p, _p]),
}



class PartLaunch(C.Structure):
    """struct B200rlPartLaunch (include/b200rl.h)."""
    _fields_ = [("tracker", _p), ("copy_stream", _p), ("main_stream", _p), ("consumed_event", _p),
                ("n", C.c_int32), ("nchunks", C.c_int32), ("chunk_lo", C.c_int32 * 4), ("chunk_hi", C.c_int32 * 4),
                ("h2d_event", _p * 4), ("graph_exec", _p * 4),
                ("new_d", _p), ("slot_d", _p), ("full_d", _p), ("new_h", _p), ("full_h", _p), ("slot_h", _p),
                ("actions_d", _p), ("actions_h", _p), ("actions_bytes", _i64), ("d2h_event", _p)]


_lib = None


def load():
    """Load the shared library (once) and attach prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m cleanrl_b200.build` "
            "(the CUDA extension is the product; there is no CPU/torch fallback)")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError => header/library out of sync
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().b200rl_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libb200rl {what} failed (status {rc}): {msg}")
