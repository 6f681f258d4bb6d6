"""ctypes binding of libpearlb200.so (include/pearl_b200.h).

The product path has NO CPU fallback: if the shared library is missing or the
process has no B200, `load()` / `init()` raise.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpearlb200.so")

PRL_BUF_DISCRETE = 0x1
PRL_BUF_CONTINUOUS = 0x2
PRL_BUF_DYNAMIC_ACTIONS = 0x4
PRL_EINVAL = -1


class BufDesc(C.Structure):
    _fields_ = [("capacity", C.c_int64), ("obs_dim", C.c_int32), ("act_dim", C.c_int32),
                ("n_actions", C.c_int32), ("flags", C.c_int32)]


class BufLayout(C.Structure):
    _fields_ = [("record_words", C.c_int32), ("off_state", C.c_int32), ("off_next_state", C.c_int32),
                ("off_action", C.c_int32), ("off_reward", C.c_int32), ("off_flags", C.c_int32),
                ("off_avail", C.c_int32), ("act_words", C.c_int32), ("storage_bytes", C.c_int64)]


class PerCfg(C.Structure):
    _fields_ = [("capacity", C.c_int64), ("alpha", C.c_double), ("beta", C.c_double), ("eps", C.c_double),
                ("seed", C.c_uint64)]


class SacCfg(C.Structure):
    _fields_ = [("obs_dim", C.c_int32), ("act_dim", C.c_int32), ("actor_h1", C.c_int32), ("actor_h2", C.c_int32),
                ("critic_h1", C.c_int32), ("critic_h2", C.c_int32), ("autotune", C.c_int32), ("max_batch", C.c_int32),
                ("max_rounds", C.c_int32), ("actor_lr", C.c_double), ("critic_lr", C.c_double), ("beta1", C.c_double),
                ("beta2", C.c_double), ("eps", C.c_double), ("weight_decay", C.c_double), ("gamma", C.c_double),
                ("tau", C.c_double)]


class DsacCfg(C.Structure):
    _fields_ = [("obs_dim", C.c_int32), ("n_actions", C.c_int32), ("actor_h1", C.c_int32), ("actor_h2", C.c_int32),
                ("critic_h1", C.c_int32), ("critic_h2", C.c_int32), ("autotune", C.c_int32), ("max_batch", C.c_int32),
                ("max_rounds", C.c_int32), ("actor_lr", C.c_double), ("critic_lr", C.c_double), ("entropy_lr", C.c_double),
                ("beta1", C.c_double), ("beta2", C.c_double), ("eps", C.c_double), ("weight_decay", C.c_double),
                ("gamma", C.c_double), ("tau", C.c_double), ("target_entropy", C.c_double), ("entropy_eps", C.c_double)]


class Td3Cfg(C.Structure):
    _fields_ = [("obs_dim", C.c_int32), ("act_dim", C.c_int32), ("actor_h1", C.c_int32), ("actor_h2", C.c_int32),
                ("critic_h1", C.c_int32), ("critic_h2", C.c_int32), ("actor_update_freq", C.c_int32), ("max_batch", C.c_int32),
                ("max_rounds", C.c_int32), ("actor_lr", C.c_double), ("critic_lr", C.c_double), ("beta1", C.c_double),
                ("beta2", C.c_double), ("eps", C.c_double), ("weight_decay", C.c_double), ("gamma", C.c_double),
                ("actor_tau", C.c_double), ("critic_tau", C.c_double), ("noise_clip", C.c_double)]


class PpoCfg(C.Structure):
    _fields_ = [("obs_dim", C.c_int32), ("n_actions", C.c_int32), ("actor_h1", C.c_int32), ("actor_h2", C.c_int32),
                ("critic_h1", C.c_int32), ("critic_h2", C.c_int32), ("max_batch", C.c_int32), ("max_rounds", C.c_int32),
                ("max_rollout", C.c_int64), ("actor_lr", C.c_double), ("critic_lr", C.c_double), ("beta1", C.c_double),
                ("beta2", C.c_double), ("eps", C.c_double), ("weight_decay", C.c_double), ("gamma", C.c_double),
                ("lam", C.c_double), ("epsilon", C.c_double), ("entropy_bonus", C.c_double)]


class DqnCfg(C.Structure):
    _fields_ = [("obs_dim", C.c_int32), ("n_actions", C.c_int32), ("hidden1", C.c_int32),
                ("hidden2", C.c_int32), ("double_dqn", C.c_int32), ("target_update_freq", C.c_int32),
                ("max_batch", C.c_int32), ("max_rounds", C.c_int32), ("rows_per_cta", C.c_int32),
                ("lr", C.c_double), ("beta1", C.c_double), ("beta2", C.c_double), ("eps", C.c_double),
                ("weight_decay", C.c_double), ("gamma", C.c_double), ("tau", C.c_double)]


_P = C.c_void_p
_SIGNATURES = {
    "prl_abi_version": (C.c_int, []),
    "prl_init": (C.c_int, [C.c_int]),
    "prl_last_error": (C.c_char_p, []),
    "prl_sm_count": (C.c_int, []),
    "prl_buf_layout_of": (C.c_int, [C.POINTER(BufDesc), C.POINTER(BufLayout)]),
    "prl_buf_create": (C.c_int, [C.POINTER(_P), C.POINTER(BufDesc), _P, _P]),
    "prl_buf_destroy": (C.c_int, [_P]),
    "prl_buf_len": (C.c_int64, [_P]),
    "prl_buf_capacity": (C.c_int64, [_P]),
    "prl_buf_head": (C.c_int64, [_P]),
    "prl_buf_clear": (C.c_int, [_P]),
    "prl_buf_set_occupancy": (C.c_int, [_P, C.c_int64, C.c_int64]),
    "prl_buf_set_shard": (C.c_int, [_P, C.c_int, C.c_int, C.c_int64]),
    "prl_buf_global_len": (C.c_int64, [_P]),
    "prl_buf_push_host": (C.c_int, [_P, C.c_int64, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "prl_buf_push_host_multi": (C.c_int, [_P, C.c_int, C.c_int64, _P, _P, _P, _P, _P, _P, _P]),
    "prl_buf_push_device": (C.c_int, [_P, C.c_int64, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "prl_rng_set_state": (C.c_int, [_P, _P, _P]),
    "prl_rng_get_state": (C.c_int, [_P, _P, _P]),
    "prl_rng_seed": (C.c_int, [_P, _P, C.c_int, _P]),
    "prl_buf_sample_indices": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, _P]),
    "prl_buf_gather": (C.c_int, [_P, _P, C.c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "prl_dqn_param_count": (C.c_int64, [C.POINTER(DqnCfg)]),
    "prl_dqn_workspace_bytes": (C.c_int64, [C.POINTER(DqnCfg)]),
    "prl_dqn_create": (C.c_int, [C.POINTER(_P), C.POINTER(DqnCfg), _P, _P, _P, _P, _P, C.c_int64, _P]),
    "prl_dqn_destroy": (C.c_int, [_P]),
    "prl_dqn_adam_step": (C.c_int64, [_P]),
    "prl_dqn_set_adam_step": (C.c_int, [_P, C.c_int64]),
    "prl_dqn_set_lr": (C.c_int, [_P, C.c_double]),
    "prl_dqn_learn": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int64, _P, _P, _P, _P, _P]),
    "prl_dqn_learn_batch": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, _P, _P, _P, C.c_int, _P, _P, _P, _P]),
    "prl_dqn_q_values": (C.c_int, [_P, C.c_int, _P, C.c_int, _P, _P]),
    "prl_comm_create": (C.c_int, [C.POINTER(_P), C.c_int, C.c_int, C.c_int64]),
    "prl_comm_local_handles": (C.c_int, [_P, _P]),
    "prl_comm_open_peers": (C.c_int, [_P, _P]),
    "prl_comm_destroy": (C.c_int, [_P]),
    "prl_dqn_set_comm": (C.c_int, [_P, _P]),
    "prl_dqn_tc_supported": (C.c_int, [_P, C.c_int]),
    "prl_dqn_learn_multi": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P]),
    "prl_per_tree_floats": (C.c_int64, [C.c_int64]),
    "prl_per_create": (C.c_int, [C.POINTER(_P), C.POINTER(PerCfg), _P, _P, _P, _P]),
    "prl_per_destroy": (C.c_int, [_P]),
    "prl_per_set_beta": (C.c_int, [_P, C.c_double]),
    "prl_per_draws": (C.c_int64, [_P]),
    "prl_per_push": (C.c_int, [_P, C.c_int64, C.c_int64, _P]),
    "prl_per_sample": (C.c_int, [_P, C.c_int, _P, _P, _P]),
    "prl_per_set_priorities": (C.c_int, [_P, _P, _P, C.c_int, _P, _P]),
    "prl_dqn_learn_per": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int64, _P, _P, _P, _P, _P, _P]),
    "prl_ppo_gae": (C.c_int, [C.c_int, _P, C.c_float, _P, _P, _P, C.c_double, C.c_double, _P, _P, _P, _P]),
    "prl_sac_actor_param_count": (C.c_int64, [C.POINTER(SacCfg)]),
    "prl_sac_critic_param_count": (C.c_int64, [C.POINTER(SacCfg)]),
    "prl_sac_workspace_bytes": (C.c_int64, [C.POINTER(SacCfg)]),
    "prl_sac_create": (C.c_int, [C.POINTER(_P), C.POINTER(SacCfg)] + [_P] * 13 + [C.c_int64, _P]),
    "prl_sac_destroy": (C.c_int, [_P]),
    "prl_sac_adam_step": (C.c_int64, [_P]),
    "prl_sac_set_graph": (C.c_int, [_P, C.c_int]),
    "prl_sac_last_launches": (C.c_int64, [_P]),
    "prl_sac_learn": (C.c_int, [_P, _P, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P]),
    "prl_dsac_actor_param_count": (C.c_int64, [C.POINTER(DsacCfg)]),
    "prl_dsac_critic_param_count": (C.c_int64, [C.POINTER(DsacCfg)]),
    "prl_dsac_workspace_bytes": (C.c_int64, [C.POINTER(DsacCfg)]),
    "prl_dsac_create": (C.c_int, [C.POINTER(_P), C.POINTER(DsacCfg)] + [_P] * 11 + [C.c_int64, _P]),
    "prl_dsac_destroy": (C.c_int, [_P]),
    "prl_dsac_adam_step": (C.c_int64, [_P]),
    "prl_dsac_set_lr": (C.c_int, [_P, C.c_double, C.c_double]),
    "prl_dsac_learn": (C.c_int, [_P, _P, C.c_int, C.c_int, _P, _P, _P, _P, _P]),
    "prl_dsac_set_graph": (C.c_int, [_P, C.c_int]),
    "prl_dsac_last_launches": (C.c_int64, [_P]),
    "prl_td3_actor_param_count": (C.c_int64, [C.POINTER(Td3Cfg)]),
    "prl_td3_critic_param_count": (C.c_int64, [C.POINTER(Td3Cfg)]),
    "prl_td3_workspace_bytes": (C.c_int64, [C.POINTER(Td3Cfg)]),
    "prl_td3_create": (C.c_int, [C.POINTER(_P), C.POINTER(Td3Cfg)] + [_P] * 12 + [C.c_int64, C.c_int64, _P]),
    "prl_td3_destroy": (C.c_int, [_P]),
    "prl_td3_actor_adam_step": (C.c_int64, [_P]),
    "prl_td3_critic_adam_step": (C.c_int64, [_P]),
    "prl_td3_learn": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int64, _P, _P, _P, _P, _P]),
    "prl_td3_set_graph": (C.c_int, [_P, C.c_int]),
    "prl_td3_last_launches": (C.c_int64, [_P]),
    "prl_ppo_actor_param_count": (C.c_int64, [C.POINTER(PpoCfg)]),
    "prl_ppo_critic_param_count": (C.c_int64, [C.POINTER(PpoCfg)]),
    "prl_ppo_workspace_bytes": (C.c_int64, [C.POINTER(PpoCfg)]),
    "prl_ppo_create": (C.c_int, [C.POINTER(_P), C.POINTER(PpoCfg)] + [_P] * 8 + [C.c_int64, _P]),
    "prl_ppo_destroy": (C.c_int, [_P]),
    "prl_ppo_adam_step": (C.c_int64, [_P]),
    "prl_ppo_set_graph": (C.c_int, [_P, C.c_int]),
    "prl_ppo_last_launches": (C.c_int64, [_P]),
    "prl_ppo_preprocess": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P]),
    "prl_ppo_gae_redo": (C.c_int, [_P, _P, C.c_float, C.c_float, _P, _P, _P]),
    "prl_ppo_learn": (C.c_int, [_P, _P, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P, _P]),
    "prl_dqn_set_timing": (C.c_int, [_P, C.c_int]),
    "prl_dqn_set_profile": (C.c_int, [_P, _P]),
    "prl_dqn_last_kernel_ms": (C.c_int, [_P, C.POINTER(C.c_float)]),
    "prl_test_umma_gemm": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, _P]),
    "prl_test_umma_gemm_ts": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, _P]),
    "prl_test_umma_gemm2": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "prl_set_contraction_engine": (C.c_int, [C.c_int]),
    "prl_get_contraction_engine": (C.c_int, []),
    "prl_test_contraction": (C.c_int, [C.c_int] * 5 + [_P, _P, _P, C.c_int, _P, _P, C.c_int, C.c_int, _P, _P, C.c_int, _P]),
    "prl_test_contraction_stamps": (C.c_int, [_P]),
    "prl_dqn_last_launch_info": (C.c_int, [_P, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                           C.POINTER(C.c_int32)]),
}
EXPORTS = tuple(_SIGNATURES)

_lib = None
_inited = set()


def load() -> C.CDLL:
    """dlopen the library (no CUDA call).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m pearl_b200.build` "
                "(pearl_b200 has no CPU or PyTorch fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        if lib.prl_abi_version() != 1:
            raise RuntimeError("libpearlb200.so ABI version mismatch")
        _lib = lib
    return _lib


def last_error() -> str:
    return (load().prl_last_error() or b"").decode(errors="replace")


def check(rc: int) -> None:
    """Map a PRL_* return code to the exception type the reference would raise."""
    if rc == 0:
        return
    msg = last_error()
    if rc == PRL_EINVAL:
        raise ValueError(msg)
    raise RuntimeError(f"libpearlb200: {msg} (code {rc})")


def init(device_index: int) -> C.CDLL:
    lib = load()
    if device_index not in _inited:
        check(lib.prl_init(device_index))
        _inited.add(device_index)
    return lib


def ptr(t) -> C.c_void_p:
    """Raw device/host pointer of a torch tensor (or None)."""
    if t is None:
        return C.c_void_p(0)
    return C.c_void_p(t.data_ptr())
