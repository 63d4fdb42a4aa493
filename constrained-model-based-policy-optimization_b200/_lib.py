"""ctypes binding of libcmbpo_b200.so (the C ABI declared in include/cmbpo_b200.h).

There is deliberately no fallback: if the shared library is missing, or no B200 is
visible, every entry point raises.  The library is built in-tree by `build.sh` /
`__graft_entry__.build()`.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# CMBPO_B200_LIB: developer override to A/B two builds of the same ABI on one GPU box
LIB_PATH = os.environ.get("CMBPO_B200_LIB") or os.path.join(_HERE, "libcmbpo_b200.so")

# enums of include/cmbpo_b200.h
NET_DYN, NET_V, NET_VC, NET_ACTOR = 0, 1, 2, 3
ACT_IDS = {None: 0, "swish": 1, "tanh": 2, "ReLU": 3, "sigmoid": 4}
PREC_FP32, PREC_BF16, PREC_FP16 = 0, 1, 2
PRECISIONS = {"fp32": PREC_FP32, "bf16": PREC_BF16, "fp16": PREC_FP16}
TERM_NO_DONE, TERM_ANTSAFE = 0, 1
COST_ZERO, COST_HCS, COST_ANTSAFE = 0, 1, 2
END_ALIVE, END_UNCERTAIN, END_HORIZON, END_TERMINAL, END_CAPPED, END_STOPPED = range(6)
SCAN_STRICT, SCAN_WARP = 0, 1

c_f32p = C.c_void_p   # device pointers travel as integers


class EnvCfg(C.Structure):
    _fields_ = [("term_id", C.c_int), ("cost_id", C.c_int), ("predicts_cost", C.c_int),
                ("deterministic", C.c_int), ("predicts_delta", C.c_int)]


class RolloutBufs(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "start_obs", "act_eps", "elite_pos", "state_eps",
        "obs", "act", "nextobs", "mu",
        "rew", "val", "cost", "cval", "logp", "dyn_error", "dkl",
        "term", "length", "end_reason", "last_val", "last_cval",
        "cum_dkl", "path_return", "path_cost", "final_obs", "step_stats")]


class RolloutCfg(C.Structure):
    _fields_ = [("B", C.c_int64), ("path_id_base", C.c_int64), ("T", C.c_int),
                ("max_steps", C.c_int), ("uncertainty_mode", C.c_int), ("dkl_lim", C.c_double),
                ("seed", C.c_uint64), ("precision", C.c_int), ("env", EnvCfg),
                ("flags", C.c_int), ("compact_every", C.c_int)]


ROLLOUT_NO_COMPACT, ROLLOUT_FUSE, ROLLOUT_NO_STORE = 1, 2, 4
LOSS_MSPE, LOSS_MSE = 0, 1


class TrainCfg(C.Structure):
    _fields_ = [("loss", C.c_int), ("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float),
                ("eps", C.c_float), ("weight_decay", C.c_float * 8), ("math", C.c_int)]


# name -> (restype, argtypes); every symbol include/cmbpo_b200.h declares
_vp, _i, _i64, _d, _f, _u64 = C.c_void_p, C.c_int, C.c_int64, C.c_double, C.c_float, C.c_uint64
SIGNATURES = {
    "cmbpo_abi_version": (_i, []),
    "cmbpo_last_error": (C.c_char_p, []),
    "cmbpo_ctx_create": (_i, [_i, C.POINTER(_vp)]),
    "cmbpo_ctx_destroy": (_i, [_vp]),
    "cmbpo_ctx_set_stream": (_i, [_vp, _vp]),
    "cmbpo_ctx_synchronize": (_i, [_vp]),
    "cmbpo_ctx_launch_count": (_i64, [_vp]),
    "cmbpo_ctx_profile": (_i, [_vp, _i]),
    "cmbpo_ctx_profile_read": (_i, [_vp, _i, C.POINTER(_d), C.POINTER(_i64), _i]),
    "cmbpo_net_set_weights": (_i, [_vp, _i, _i, _i, C.POINTER(_i), C.POINTER(_vp), C.POINTER(_vp),
                                   C.POINTER(_i), _vp, _vp, _vp, _vp, _i, C.POINTER(_i), _i, _i]),
    "cmbpo_actor_set_log_std": (_i, [_vp, _vp, _i, _i]),
    "cmbpo_ens_predict": (_i, [_vp, _i, _vp, _i64, _i, _vp, _vp, _i]),
    "cmbpo_ens_predict_mean": (_i, [_vp, _i, _vp, _i64, _vp, _vp, _i]),
    "cmbpo_policy_act": (_i, [_vp, _vp, _i64, _vp, _vp, _u64, _i, _vp, _vp, _vp, _vp, _vp, _i]),
    "cmbpo_fakeenv_step": (_i, [_vp, C.POINTER(EnvCfg), _vp, _vp, _i64, _vp, _vp, _vp, _u64, _i,
                                _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i]),
    "cmbpo_rollout": (_i, [_vp, C.POINTER(RolloutCfg), C.POINTER(RolloutBufs)]),
    "cmbpo_rollout_histogram": (_i, [_vp, _vp, _vp, _i64, _i, C.POINTER(_i64)]),
    "cmbpo_rollout_truncate": (_i, [_vp, C.POINTER(RolloutBufs), _i64, _i, _i, _i64, _i]),
    "cmbpo_archive_index": (_i, [_vp, _vp, _i64, _i, _vp, _vp, C.POINTER(C.c_int64)]),
    "cmbpo_archive_sample_epochs": (_i, [_vp, _vp, _vp, _vp, _i, _i64, _u64, _u64, _vp]),
    "cmbpo_archive_sample_boltz": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i64, _u64, _u64, _vp]),
    "cmbpo_gather_rows": (_i, [_vp, _vp, _i, _vp, _i64, _vp]),
    "cmbpo_policy_kl_epochs": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i64, _i, C.POINTER(C.c_double)]),
    "cmbpo_rollout_diagnostics": (_i, [_vp, C.POINTER(RolloutBufs), _i64, _vp, _vp, C.POINTER(C.c_double)]),
    "cmbpo_gae_paths": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _i, _i64, _i64, _vp, _vp, _vp,
                             _d, _d, _d, _d, _vp, _vp, _vp, _vp, _i]),
    "cmbpo_gae_flat": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _vp, _i64, _vp, _vp,
                            _d, _d, _d, _d, _vp, _vp, _vp, _vp, _i]),
    "cmbpo_adv_stats_pass1": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _i, _i64, _i64, _vp, _vp]),
    "cmbpo_adv_stats_pass2": (_i, [_vp, _vp, _i64, _i, _i64, _i64, _vp, _f, _vp]),
    "cmbpo_adv_normalise": (_i, [_vp, _vp, _vp, _i64, _i, _i64, _i64, _vp, _f, _f, _f]),
    "cmbpo_adv_stats_pass2_dev": (_i, [_vp, _vp, _i64, _i, _i64, _i64, _vp, _vp, _vp]),
    "cmbpo_adv_normalise_dev": (_i, [_vp, _vp, _vp, _i64, _i, _i64, _i64, _vp, _vp]),
    "cmbpo_ens_train_begin": (_i, [_vp, _i]),
    "cmbpo_ens_train_step": (_i, [_vp, _i, _vp, _vp, _i64, C.POINTER(TrainCfg), _vp]),
    "cmbpo_ens_train_loss": (_i, [_vp, _i, _vp, _vp, _i64, _vp]),
    "cmbpo_ens_train_grads": (_i, [_vp, _i, _i, _vp, _vp]),
    "cmbpo_ens_train_end": (_i, [_vp, _i, _vp, _i]),
    "cmbpo_net_get_weights": (_i, [_vp, _i, _i, _vp, _vp]),
    "cmbpo_net_set_scalers": (_i, [_vp, _i, _vp, _vp, _vp, _vp]),
    "cmbpo_path_offsets": (_i, [_vp, _vp, _i64, _vp]),
    "cmbpo_compact_field": (_i, [_vp, _vp, _i64, _i, _i, _vp, _vp, _vp]),
    "cmbpo_scatter_rows": (_i, [_vp, _vp, _i64, _i, _i, _vp, _vp, _i64]),
}

_lib = None
ABI_VERSION = 2


class CmbpoError(RuntimeError):
    pass


def load():
    """Load the shared library (once) and attach the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CmbpoError(
            "libcmbpo_b200.so is not built (%s): run ./build.sh or __graft_entry__.build(); "
            "there is no CPU fallback" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    if lib.cmbpo_abi_version() != ABI_VERSION:
        raise CmbpoError("ABI version mismatch")
    _lib = lib
    return lib


def check(status):
    if status != 0:
        raise CmbpoError(load().cmbpo_last_error().decode("utf-8", "replace"))
