"""ctypes binding of include/icrl_b200.h (libicrl_b200.so, sm_100a CUDA kernels).

There is deliberately no fallback: if the shared library is missing or a call fails, the caller gets
an exception.  The library is built in-tree by `python -m icrl_b200.build` (see __graft_entry__.build()).
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libicrl_b200.so")

ABI_VERSION = 2
MAX_SELECT, MAX_HIDDEN, CN_MAX_WIDTH = 512, 3, 64
PPO_STATS_PER_STEP = 8

c_float_p = C.POINTER(C.c_float)
c_void = C.c_void_p


class CnDesc(C.Structure):
    _fields_ = [
        ("obs_dim", C.c_int32), ("acs_dim", C.c_int32), ("is_discrete", C.c_int32), ("n_select", C.c_int32),
        ("select", C.c_int32 * MAX_SELECT), ("n_hidden", C.c_int32), ("hidden", C.c_int32 * MAX_HIDDEN),
        ("has_norm", C.c_int32), ("has_clip_obs", C.c_int32), ("has_clip_acs", C.c_int32), ("clip_obs", C.c_double),
        ("params", c_void), ("obs_mean", c_void), ("obs_rstd", c_void), ("acs_low", c_void), ("acs_high", c_void),
    ]


class CnTrainCfg(C.Structure):
    _fields_ = [
        ("iterations", C.c_int32), ("importance_sampling", C.c_int32), ("per_step_is", C.c_int32),
        ("train_gail_lambda", C.c_int32), ("eps", C.c_float), ("regularizer_coeff", C.c_float),
        ("target_kl_old_new", C.c_float), ("target_kl_new_old", C.c_float), ("lr", C.c_double),
        ("adam_beta1", C.c_double), ("adam_beta2", C.c_double), ("adam_eps", C.c_double),
        ("batch_size", C.c_int32), ("perm", c_void),
    ]


class CnDist(C.Structure):
    _fields_ = [("rank", C.c_int32), ("world", C.c_int32), ("recv", c_void * 8), ("buffer_bytes", C.c_int64),
                ("seq_base", C.c_uint32), ("n_nominal_global", C.c_int64), ("n_expert_global", C.c_int64),
                ("n_episodes_global", C.c_int32), ("episode_base", C.c_int32)]


class CnTrainMetrics(C.Structure):
    _fields_ = [(n, C.c_float) for n in (
        "cn_loss", "expert_loss", "unweighted_nominal_loss", "nominal_loss", "regularizer_loss", "is_mean", "is_max",
        "is_min", "nominal_preds_max", "nominal_preds_min", "nominal_preds_mean", "expert_preds_max",
        "expert_preds_min", "expert_preds_mean", "kl_old_new", "kl_new_old")] + [
        ("early_stop_itr", C.c_int32), ("steps_taken", C.c_int32)]


class PpoCfg(C.Structure):
    _fields_ = [
        ("obs_dim", C.c_int32), ("act_dim", C.c_int32), ("is_discrete", C.c_int32), ("hidden", C.c_int32 * 2),
        ("T", C.c_int32), ("E", C.c_int32), ("batch_size", C.c_int32), ("n_epochs", C.c_int32),
        ("has_target_kl", C.c_int32), ("has_clip_vf_reward", C.c_int32), ("has_clip_vf_cost", C.c_int32),
        ("clip_range", C.c_float), ("clip_range_reward_vf", C.c_float), ("clip_range_cost_vf", C.c_float),
        ("ent_coef", C.c_float), ("reward_vf_coef", C.c_float), ("cost_vf_coef", C.c_float),
        ("max_grad_norm", C.c_float), ("target_kl", C.c_float), ("nu", C.c_float),
        ("lr", C.c_double), ("adam_beta1", C.c_double), ("adam_beta2", C.c_double), ("adam_eps", C.c_double),
        ("max_steps", C.c_int32), ("trunk_hidden", (C.c_int32 * 2) * 3),
    ]


class PpoData(C.Structure):
    _fields_ = [(n, c_void) for n in (
        "observations", "actions", "old_log_prob", "old_reward_values", "reward_advantages", "reward_returns",
        "old_cost_values", "cost_advantages", "cost_returns", "perm", "nu_device")]


class PpoDist(C.Structure):
    _fields_ = [("rank", C.c_int32), ("world", C.c_int32), ("recv", c_void * 8), ("flags", c_void * 8),
                ("flag_base", C.c_uint32), ("advsums", c_void)]


PPO_RECV_BYTES = 32 * 1024 * 1024
PPO_FLAG_BYTES = 2 * 8 * 4 * 4

# name -> (restype, argtypes); every symbol include/icrl_b200.h declares (checked by tests/test_abi.py)
SIGNATURES = {
    "icrl_abi_version": (C.c_int, []),
    "icrl_last_error": (C.c_char_p, []),
    "icrl_launch_count": (C.c_int64, []),
    "icrl_device_info": (C.c_int, [C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "icrl_measure_peaks": (C.c_int, [C.POINTER(C.c_double), c_void]),
    "icrl_cn_param_count": (C.c_int64, [C.POINTER(CnDesc)]),
    "icrl_cn_forward": (C.c_int, [C.POINTER(CnDesc), c_void, C.c_int32, c_void, C.c_int64, c_void, C.c_int32, c_void]),
    "icrl_cn_forward_host": (C.c_int, [C.POINTER(CnDesc), c_void, C.c_int32, c_void, C.c_int64, c_void, C.c_int32,
                                       c_void]),
    "icrl_cn_train": (C.c_int, [C.POINTER(CnDesc), C.POINTER(CnTrainCfg), c_void, C.c_int32, c_void, C.c_int64, c_void,
                                C.c_int32, c_void, C.c_int32, c_void, C.c_int64, c_void, c_void, C.POINTER(C.c_int64),
                                C.POINTER(CnTrainMetrics), c_void]),
    "icrl_cn_dist_bytes": (C.c_int64, [C.POINTER(CnDesc), C.c_int32]),
    "icrl_cn_train_dist": (C.c_int, [C.POINTER(CnDesc), C.POINTER(CnTrainCfg), c_void, C.c_int32, c_void, C.c_int64, c_void,
                                     C.c_int32, c_void, C.c_int32, c_void, C.c_int64, c_void, c_void, C.POINTER(C.c_int64),
                                     C.POINTER(CnTrainMetrics), C.POINTER(CnDist), c_void]),
    "icrl_dual_gae": (C.c_int, [c_void] * 8 + [C.c_int32, C.c_int32] + [C.c_double] * 4 + [c_void] * 5),
    "icrl_dual_gae_host": (C.c_int, [c_void] * 8 + [C.c_int32, C.c_int32] + [C.c_double] * 4 + [c_void] * 5),
    "icrl_ppo_param_count": (C.c_int64, [C.POINTER(PpoCfg)]),
    "icrl_ppo_train": (C.c_int, [C.POINTER(PpoCfg), C.POINTER(PpoData), c_void, c_void, c_void, C.c_int64, c_void,
                                 c_void, c_void]),
    "icrl_ppo_train_dist": (C.c_int, [C.POINTER(PpoCfg), C.POINTER(PpoData), c_void, c_void, c_void, C.c_int64, c_void,
                                      c_void, C.POINTER(PpoDist), c_void]),
    "icrl_ppo_local_advsums": (C.c_int, [C.POINTER(PpoCfg), C.POINTER(PpoData), c_void, c_void]),
    "icrl_comm_alloc": (C.c_int, [C.c_int64, C.POINTER(c_void), C.c_char_p]),
    "icrl_comm_open": (C.c_int, [C.c_char_p, C.POINTER(c_void)]),
    "icrl_comm_close": (C.c_int, [c_void]),
    "icrl_comm_free": (C.c_int, [c_void]),
    "icrl_policy_forward": (C.c_int, [C.POINTER(PpoCfg), c_void, c_void, C.c_int64, c_void, c_void, c_void, c_void]),
    "icrl_dual_update": (C.c_int, [c_void, c_void, C.c_int64, C.c_double, C.c_double, C.c_int64, C.c_double, c_void]),
    "icrl_cost_normalize": (C.c_int, [c_void, c_void, c_void, C.c_int32, C.c_int32, C.c_double, C.c_double, C.c_double,
                                      C.c_int32, C.c_int32, c_void, c_void, c_void]),
}


class IcrlError(RuntimeError):
    pass


_lib = None


def lib():
    """Load (once) and return the ctypes handle.  Raises if the CUDA library has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise IcrlError(f"{LIB_PATH} not found: build it with `python -m icrl_b200.build` "
                            "(there is no CPU fallback for the learner hot path)")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        if handle.icrl_abi_version() != ABI_VERSION:
            raise IcrlError("ABI version mismatch between icrl_b200/_lib.py and libicrl_b200.so")
        _lib = handle
    return _lib


def check(rc):
    if rc != 0:
        msg = lib().icrl_last_error().decode(errors="replace")
        raise IcrlError(f"icrl_b200 call failed (code {rc}): {msg}")


def ptr(t):
    """Raw device/host address of a torch tensor or numpy array (None -> NULL)."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return C.c_void_p(t.data_ptr())
    return C.c_void_p(t.__array_interface__["data"][0])      # (ndarray.ctypes builds a helper object per access: ~2 us)


def current_stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
