"""ctypes binding of libxb200.so (include/xb200.h).

The reference's own native-boundary idiom is a ctypes-loaded C library
(xuance/environment/magent2/c_lib.py:10-23); this is the same idea for the PPO hot path.  There is NO CPU or
PyTorch fallback: if the library is missing or fails to load, importing any product path raises.
"""
import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
# XB200_LIB: an alternative build of the same library (e.g. the instrumented one of tools/profile/dense_timeline.py)
LIB_PATH = os.environ.get("XB200_LIB") or os.path.join(_PKG, "libxb200.so")

_i64, _i32, _f32, _f64, _u64, _vp = C.c_int64, C.c_int, C.c_float, C.c_double, C.c_uint64, C.c_void_p

# name -> argtypes, exactly the prototypes of include/xb200.h (pointers and the stream are void*)
SIGNATURES = {
    "xb_version": [],
    "xb_env_reset": [_i32, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _vp],
    "xb_env_step": [_i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _vp],
    "xb_rollout_step": [_i32, _vp, _vp, _vp, _u64, _vp, _u64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                        _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f32, _vp, _vp, _vp,
                        _vp, _vp, _i32, _f32, _vp, _vp, _vp, _f64, _i32, _vp, _vp, _vp, _i64, _vp],
    "xb_eval_step": [_i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _i64, _vp, _vp, _vp, _i64, _vp, _vp,
                     _i32, _vp, _vp, _i64, _vp],
    "xb_sincos_f64": [_vp, _vp, _vp, _i64, _vp],
    "xb_store": [_vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f32, _i32, _i64, _vp],
    "xb_gae": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _f64, _f64, _i32, _i32, _vp],
    "xb_gather_obs": [_vp, _i64, _i64, _i64, _vp, _i32, _vp, _vp, _vp, _vp],
    "xb_gather_batch": [_vp, _i64, _i64, _i64, _vp, _i32, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                        _vp, _vp],
    "xb_normalize_adv": [_vp, _vp, _i64, _i64, _vp],
    "xb_ppo_loss_categorical": [_vp, _i64, _i64, _i64, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _f32, _f32,
                                _f32, _f32, _f32, _i64, _vp, _vp, _vp, _vp],
    "xb_ppo_loss_gaussian": [_vp, _i64, _i64, _i64, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _f32, _f32,
                             _f32, _f32, _f32, _i64, _vp, _vp, _vp, _vp, _vp],
    "xb_dist_loss_categorical": [_i64, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _f32, _f32, _f32, _vp, _f32, _f32, _f32, _f32,
                                 _vp, _vp, _vp, _vp, _vp],
    "xb_dist_loss_gaussian": [_i64, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _f32, _f32, _f32, _vp, _f32, _f32,
                              _f32, _f32, _vp, _vp, _vp, _vp, _vp, _vp],
    "xb_kl_coef_adapt": [_vp, _vp, _f32, _i64, _vp],
    "xb_pack_records": [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp],
    "xb_gather_records": [_vp, _i64, _i64, _i64, _vp, _i32, _vp, _vp, _vp, _vp],
    "xb_gather_trunk_fwd": [_vp, _i64, _i64, _i64, _vp, _i32, _vp, _vp, _f32, _i32, _vp, _vp, _vp, _vp, _vp, _vp],
    "xb_sample_categorical": [_vp, _i32, _u64, _vp, _u64, _vp, _vp, _i64, _vp],
    "xb_sample_gaussian": [_vp, _vp, _i32, _u64, _vp, _u64, _vp, _vp, _i64, _vp],
    "xb_counter_add": [_vp, _u64, _vp],
    "xb_host_permutation": [_vp, _i64, _u64],
    "xb_host_permutation32": [_vp, _i64, _u64],
    "xb_random_permutation": [_vp, _i64, _u64, _vp, _u64, _vp],
    "xb_moments4": [_vp, _i32, _vp, _vp, _i64, _vp],
    "xb_rms_normalize": [_vp, _i32, _vp, _vp, _vp, _f32, _vp, _i64, _i64, _vp],
    "xb_returns_track": [_vp, _vp, _vp, _vp, _f64, _i32, _vp, _vp, _i64, _vp],
    "xb_rms_merge_scalar": [_vp, _vp, _vp, _vp],
    "xb_rms_apply": [_vp, _i32, _i32, _vp, _vp, _i64, _f32, _vp, _i64, _vp],
    "xb_rms_update_rows": [_vp, _i32, _i32, _i64, _vp, _vp, _vp, _vp, _vp],
    "xb_rms_merge_sums": [_vp, _i32, _vp, _vp, _i32, _vp, _vp, _vp],
    "xb_head_fwd": [_vp, _vp, _vp, _vp, _i64, _i32, _i32, _vp],
    "xb_head_bwd_act": [_vp, _vp, _vp, _f32, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _i32, _vp],
    "xb_bias_act_fwd": [_vp, _vp, _f32, _i64, _i32, _vp],
    "xb_act_bias_bwd": [_vp, _vp, _f32, _vp, _vp, _vp, _i64, _i32, _vp],
    "xb_dense_split_weights": [_vp, _i32, _i32, _vp, _vp, _vp, _vp, _i32, _i32, _vp],
    "xb_dense_split_weights2": [_vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp],
    "xb_dense_fwd": [_vp, _i64, _i32, _vp, _vp, _i32, _vp, _f32, _vp, _vp, _vp, _i32, _vp, _i32, _vp],
    "xb_dense_fwd2": [_vp, _i64, _i32, _i32, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32,
                      _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp],
    "xb_dense_fwd2_loss": [_vp, _i64, _i32, _i32, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                           _i32, _vp, _i32, _vp, _vp, _i64, _f32, _f32, _f32, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                           _vp, _vp, _vp],
    "xb_mlp_fwd_from_obs": [_vp, _i32, _i32, _vp, _vp, _i64, _i32, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp,
                            _vp, _vp, _vp, _i32, _vp, _vp, _vp, _i64, _f32, _i32, _vp],
    "xb_mlp_fwd_from_obs_train": [_vp, _i32, _i32, _vp, _vp, _i64, _i32, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp,
                                  _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _i64, _f32, _f32, _f32, _f32, _vp, _vp, _vp, _vp,
                                  _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "xb_dense_dgrad": [_vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _i32, _i32, _i64, _vp, _vp, _i32, _vp, _f32, _vp, _i32, _vp,
                       _vp, _vp],
    "xb_dense_wgrad_workspace_floats": [_i32],
    "xb_dense_wgrad": [_vp, _vp, _vp, _i32, _vp, _vp, _vp, _i32, _vp, _i64, _i32, _i32, _f32, _vp, _vp, _vp, _vp, _vp, _vp,
                       _vp, _vp, _vp, _vp],
    "xb_mlp_trunk_fwd": [_vp, _i32, _i32, _vp, _vp, _f32, _vp, _i64, _i32, _vp, _vp],
    "xb_mlp_trunk_wgrad_workspace_floats": [_i32, _i32],
    "xb_mlp_trunk_wgrad_parts": [],
    "xb_mlp_backward_tail": [_vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp,
                             _vp, _vp, _vp, _i32, _vp],
    "xb_mlp_backward_tail_norm": [_vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32,
                                  _vp, _vp, _vp, _vp, _i32, _vp, _vp, _f32, _f32, _i64, _f32, _f32, _f32, _f32, _vp, _vp, _vp],
    "xb_mlp_backward_tail_bin": [_vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32,
                                 _vp, _vp, _vp, _vp, _i32, _vp, _vp, _f32, _f32, _i64, _f32, _f32, _f32, _f32, _vp, _vp,
                                 _vp, _vp, _vp, _vp, _vp, _vp, _f32, _vp],
    "xb_dense_wgrad_bin": [_vp, _i32, _vp, _i32, _vp, _i32, _vp, _i64, _i32, _i32, _vp, _vp],
    "xb_head3_fold": [_vp, _vp, _vp, _vp, _i32, _vp],
    "xb_head3_unfold_grads": [_vp, _vp, _i32, _vp],
    "xb_mlp_trunk_wgrad": [_vp, _vp, _i32, _i32, _vp, _vp, _vp, _i64, _i32, _vp],
    "xb_peer_stats_max": [],
    "xb_peer_alloc": [_vp, _i64],
    "xb_peer_free": [_vp],
    "xb_peer_export": [_vp, _vp],
    "xb_peer_import": [_vp, _vp],
    "xb_peer_close": [_vp],
    "xb_peer_allreduce_grad_norm": [_vp, _i32, _i32, _i64, _vp, _vp, _vp, _vp, _f32, _f32, _i64, _f32, _f32, _f32, _f32, _f32, _vp,
                                    _vp, _vp, _vp],
    "xb_adam_apply": [_vp, _vp, _vp, _vp, _i64, _f32, _f32, _f32, _f32, _vp, _vp],
    "xb_adam_apply_split": [_vp, _vp, _vp, _vp, _i64, _f32, _f32, _f32, _f32, _vp, _i64, _vp, _vp, _i64, _vp, _vp, _i32, _i32,
                            _vp, _vp, _vp],
    "xb_peer_allreduce_mean": [_vp, _i32, _i32, _i64, _vp, _vp, _vp, _vp],
    "xb_peer_allreduce_f64": [_vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp],
    "xb_peer_allreduce_merge": [_vp, _i32, _i32, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp],
    "xb_adv_stats_minibatches": [_vp, _i64, _i64, _i64, _i64, _vp, _i64, _vp, _vp],
    "xb_clip_adam_step": [_vp, _vp, _vp, _vp, _i64, _vp, _f32, _f32, _i64, _f32, _f32, _f32, _f32, _f32, _vp, _vp, _vp, _vp],
}

_lib = None


class XB200Error(RuntimeError):
    pass


def load():
    """Loads libxb200.so; raises (never falls back) if it is absent or unloadable."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise XB200Error(
            "libxb200.so not found at %s. Build it with `python -m xuanpolicy_b200.csrc.build` "
            "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here means header and library are out of sync
        fn.argtypes = argtypes
        fn.restype = C.c_int
    for name in ("xb_peer_block_bytes", "xb_peer_stats_offset", "xb_peer_grad_offset"):
        fn = getattr(lib, name)
        fn.argtypes = [C.c_int64] if name == "xb_peer_block_bytes" else []
        fn.restype = C.c_int64
    lib.xb_error_string.argtypes = [C.c_int]
    lib.xb_error_string.restype = C.c_char_p
    if lib.xb_version() != 100:
        raise XB200Error("libxb200.so version %d does not match the binding (100)" % lib.xb_version())
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().xb_error_string(rc).decode()
        raise XB200Error("%s failed with code %d: %s" % (what or "xb200 call", rc, msg))


def call(name, *args):
    check(getattr(load(), name)(*args), name)
