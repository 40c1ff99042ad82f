"""ctypes binding of libmappo_b200.so (the C ABI declared in include/mappo_b200.h).

The library is the product: if it is missing or was not built for this GPU the import of any
engine component raises -- there is no CPU or PyTorch fallback anywhere in this package.
"""
import ctypes as C
import os

MAX_HEADS = 4
MAX_LAYERS = 2
GEMM_FP32, GEMM_TF32 = 0, 1
WORLD_SPREAD, WORLD_REFERENCE = 0, 1          # mappo_rollout_closed_loop_ex
_LIB_PATH = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "lib", "libmappo_b200.so")


class NetDesc(C.Structure):
    _fields_ = [("in_dim", C.c_int32), ("hidden", C.c_int32), ("layer_n", C.c_int32),
                ("use_feature_norm", C.c_int32), ("use_relu", C.c_int32), ("recurrent", C.c_int32),
                ("n_heads", C.c_int32), ("head_dim", C.c_int32 * MAX_HEADS), ("is_critic", C.c_int32)]


class NetLayout(C.Structure):
    _fields_ = [("fn_w", C.c_int32), ("fn_b", C.c_int32),
                ("fc1_w", C.c_int32), ("fc1_b", C.c_int32), ("ln1_w", C.c_int32), ("ln1_b", C.c_int32),
                ("fc2_w", C.c_int32 * MAX_LAYERS), ("fc2_b", C.c_int32 * MAX_LAYERS),
                ("ln2_w", C.c_int32 * MAX_LAYERS), ("ln2_b", C.c_int32 * MAX_LAYERS),
                ("gru_wih", C.c_int32), ("gru_whh", C.c_int32), ("gru_bih", C.c_int32), ("gru_bhh", C.c_int32),
                ("rnn_ln_w", C.c_int32), ("rnn_ln_b", C.c_int32),
                ("head_w", C.c_int32), ("head_b", C.c_int32), ("total", C.c_int32)]


class LossCfg(C.Structure):
    _fields_ = [("clip_param", C.c_float), ("entropy_coef", C.c_float), ("value_loss_coef", C.c_float),
                ("huber_delta", C.c_float),
                ("use_clipped_value_loss", C.c_int32), ("use_huber_loss", C.c_int32),
                ("use_value_active_masks", C.c_int32), ("use_policy_active_masks", C.c_int32),
                ("use_valuenorm", C.c_int32), ("update_actor", C.c_int32), ("gemm_mode", C.c_int32),
                ("happo", C.c_int32), ("inputs_prepared", C.c_int32), ("image_ready", C.c_int32)]


_P = C.c_void_p


class Batch(C.Structure):
    _fields_ = [(n, _P) for n in ("obs", "share_obs", "actions", "old_logp", "value_preds", "returns", "advantages",
                                  "masks", "active_masks", "avail", "h0_actor", "h0_critic", "rows", "seq_first", "factor")] + \
               [("n_rows", C.c_int32), ("seq_len", C.c_int32), ("n_seq", C.c_int32)]


_i32, _u64, _f32, _i64 = C.c_int32, C.c_uint64, C.c_float, C.c_int64
_SIGS = {
    "mappo_abi_version": (_i32, []),
    "mappo_last_error": (C.c_char_p, []),
    "mappo_device_check": (_i32, [C.POINTER(_i32)] * 3),
    "mappo_net_layout": (_i32, [C.POINTER(NetDesc), C.POINTER(NetLayout)]),
    "mappo_policy_step": (_i32, [C.POINTER(NetDesc), _P, C.POINTER(NetDesc), _P] + [_P] * 7 +
                          [_u64, _P, _i32, _i32] + [_P] * 6 + [_P, _P] + [_P]),
    "mappo_rollout_persistent": (_i32, [C.POINTER(NetDesc), _P, _P, C.POINTER(NetDesc), _P, _P] + [_P] * 11 + [_P] * 6 +
                                 [_P, _u64, _P, _i32, _i32, _P]),
    "mappo_rollout_image_floats": (_i32, [C.POINTER(NetDesc)]),
    "mappo_big_net": (_i32, [C.POINTER(NetDesc)]),
    "mappo_debug_big_timing": (_i32, [_i32, _P, _P]),
    "mappo_debug_gru_timing": (_i32, [_i32, _P, _P]),
    "mappo_debug_gru_cycles": (_i32, [_P]),
    "mappo_debug_big_lin": (_i32, [_P, _i32, _P, _i32, _P, _P, _P, _P, _i32, _i32, _i32, _i32, _P]),
    "mappo_debug_big_grad": (_i32, [_P, _i32, _i32, _i32, _P, _i32, _i32, _i32, _P, _P, _i32, _P]),
    "mappo_debug_big_grad_splits": (_i32, [_i32, _i32, _i32, _i32]),
    "mappo_rollout_workspace_floats": (_i64, [C.POINTER(NetDesc), _i32]),
    "mappo_pack_rollout_weights_ex": (_i32, [C.POINTER(NetDesc), _P, _P, _i32, _P]),
    "mappo_policy_step_ex": (_i32, [C.POINTER(NetDesc), _P, C.POINTER(NetDesc), _P] + [_P] * 7 +
                             [_u64, _P, _i32, _i32] + [_P] * 6 + [_P, _P] + [_i32, _P]),
    "mappo_pack_rollout_weights": (_i32, [C.POINTER(NetDesc), _P, _P, _P]),
    "mappo_counter_add": (_i32, [_P, _u64, _P]),
    "mappo_p2p_allreduce_f32": (_i32, [_P, _P, _i32, _i32, _i64, _i32, _P, _P, _P, _P, _P]),
    "mappo_p2p_allreduce_f64": (_i32, [_P, _P, _i32, _i32, _i64, _i32, _P, _P, _P]),
    "mappo_env_insert": (_i32, [_P] * 6 + [_i32] * 5 + [_P] * 8 + [_P, _u64] + [_P]),
    "mappo_compute_returns": (_i32, [_P] * 6 + [_i32, _i32, _f32, _f32, _i32, _i32] + [_P] * 3 + [_P]),
    "mappo_advantages": (_i32, [_P, _P, _P, _P, _i32, _P, _P, _P]),
    "mappo_evaluate_actions": (_i32, [C.POINTER(NetDesc), _P, C.POINTER(Batch), C.POINTER(LossCfg), _P, _P, _P, _P, _P]),
    "mappo_minibatch_stats": (_i32, [_P, _P, _P, _i32, _P, _P]),
    "mappo_debug_launch_count": (_i64, []),
    "mappo_rollout_closed_loop": (_i32, [C.POINTER(NetDesc), _P, C.POINTER(NetDesc), _P] + [_P] * 7 + [_P] * 4 +
                                  [_P, _u64, _P, _P, _u64, _P, _i32, _i32, _i32, _i32, _i32, _P]),
    "mappo_rollout_closed_loop_ex": (_i32, [C.POINTER(NetDesc), _P, C.POINTER(NetDesc), _P] + [_P] * 9 + [_i32] + [_P] * 6 +
                                     [_P, _u64, _P, _P, _u64, _P, _i32, _i32, _i32, _i32, _i32, _P]),
    "mappo_mpe_spread_step": (_i32, [_P, _P, _P, _P, _P, _P, _u64, _P, _i32, _i32, _i32, _i32, _P, _P, _P, _P, _P]),
    "mappo_mpe_reference_step": (_i32, [_P, _P, _P, _P, _P, _P, _P, _P, _u64, _P, _i32, _i32, _P, _P, _P, _P, _P]),
    "mappo_minibatch_stats_batch": (_i32, [_P, _P, _P, _i64, _i32, _i32, _P, _P]),
    "mappo_randperm_batch": (_i32, [_i32, _i32, _u64, _P, _P, _P]),
    "mappo_valuenorm_update": (_i32, [_P, _P, _P]),
    "mappo_gather_rows": (_i32, [_P, _P, _i32, _i32, _P, _P]),
    "mappo_chunk_rows": (_i32, [_P, _i32, _i32, _i32, _i32, _P, _P, _P]),
    "mappo_randperm": (_i32, [_i32, _u64, _P, _P, _P]),
    "mappo_debug_big_plan": (_i32, [C.POINTER(NetDesc), _i32, _P]),
    "mappo_update_tail": (_i32, [C.POINTER(NetDesc), _P, _P, _i32, _P, _P, _P, _P, _i32, _P, _P, _f32, _f32, _i32, _P, _P, _P, _i32, _P, _P, _i32, _i32, _i64, _P, _P]),
    "mappo_update_workspace_floats": (_i64, [C.POINTER(NetDesc), _i32, _i32]),
    "mappo_update_grad_slots": (_i32, [C.POINTER(NetDesc), _i32, _i32]),
    "mappo_tf32_supported": (_i32, [C.POINTER(NetDesc)]),
    "mappo_debug_tc_timing": (_i32, [C.POINTER(_i64)]),
    "mappo_debug_pol_timing": (_i32, [C.POINTER(_i64), _i32]),
    "mappo_update_fwd_bwd": (_i32, [C.POINTER(NetDesc), _P, C.POINTER(Batch), C.POINTER(LossCfg), _P, _P, _P, _P,
                                    _i32, _P, _P, _P]),
    "mappo_update_slot_floats": (_i32, [C.POINTER(NetDesc), _i32]),
    "mappo_update_finish": (_i32, [C.POINTER(NetDesc), _P, _P, _i32, _i32, _P, _P, C.POINTER(_i32), _P, _P]),
    "mappo_grad_reduce": (_i32, [_P, _i32, _i32, _P, _P, C.POINTER(_i32), _P]),
    "mappo_grad_sumsq": (_i32, [_P, _i32, _P, C.POINTER(_i32), _P]),
    "mappo_clip_adam": (_i32, [_P, _P, _P, _P, _i32, _P, _i32, _P, _P, _f32, _f32, _i32, _P, _P, _P]),
}
EXPORTS = tuple(_SIGS)

_lib = None


def lib_path():
    return _LIB_PATH


def load():
    """dlopen the library and attach signatures; raises with a build hint when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise RuntimeError(
            f"{_LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C on-policy_b200/csrc`). The MAPPO engine has no CPU fallback.")
    lib = C.CDLL(_LIB_PATH)
    for name, (res, args) in _SIGS.items():
        fn = getattr(lib, name)          # AttributeError here = header / library out of sync
        fn.restype = res
        fn.argtypes = args
    if lib.mappo_abi_version() != 5:
        raise RuntimeError("libmappo_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise RuntimeError(f"libmappo_b200: status {rc}: {load().mappo_last_error().decode()}")


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL). Tensors must be contiguous CUDA tensors."""
    if t is None:
        return None
    if not t.is_cuda or not t.is_contiguous():
        raise RuntimeError("libmappo_b200 takes contiguous CUDA tensors")
    return t.data_ptr()
