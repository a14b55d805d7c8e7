"""ctypes binding of include/cstr_b200.h.  There is NO fallback: if the CUDA library is missing or a
call fails, a ``CstrLibraryError`` is raised (the product never routes through a CPU path)."""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_uint32, c_uint64, c_void_p
from typing import Optional

from . import _build

ABI_VERSION = 17
MATH_STRICT, MATH_FAST = 0, 1
INIT_RANDOM, INIT_STATIC = 0, 1
REC_FLOATS = 16
ACTOR_TANH, ACTOR_GAUSSIAN = 0, 1


class CstrLibraryError(RuntimeError):
    pass


class EnvParams(Structure):
    """struct cstr_env_params"""

    _fields_ = [
        ("seed", c_uint64),
        ("env_offset", c_int64),
        ("target_c2", c_double),
        ("max_steps", c_int32),
        ("init_mode", c_int32),
    ]


class ActorF32(Structure):
    """struct cstr_actor_f32"""

    _fields_ = [
        ("W1", c_void_p), ("b1", c_void_p),
        ("W2", c_void_p), ("b2", c_void_p),
        ("W3", c_void_p), ("b3", c_void_p),
        ("H1", c_int32), ("H2", c_int32),
        ("kind", c_int32), ("reserved", c_int32),
    ]


class EpisodeStatsStruct(Structure):
    """struct cstr_episode_stats"""

    _fields_ = [("ep_return", c_void_p), ("finished", c_void_p), ("count", c_void_p), ("capacity", c_uint32), ("reserved", c_uint32)]


class NormParams(Structure):
    """struct cstr_norm_params"""

    _fields_ = [("stats", c_void_p), ("epsilon", c_double), ("clip_obs", c_double), ("clip_reward", c_double),
                ("norm_obs", c_int32), ("norm_reward", c_int32)]


class RolloutNorm(Structure):
    """struct cstr_rollout_norm"""

    _fields_ = [("stats", c_void_p), ("returns", c_void_p), ("workspace", c_void_p), ("gamma", c_double), ("epsilon", c_double),
                ("clip_obs", c_double), ("training", c_int32), ("norm_obs", c_int32)]


class Td3Config(Structure):
    """struct cstr_td3_config"""

    _fields_ = [("h1", c_int32), ("h2", c_int32), ("batch", c_int32), ("policy_delay", c_int32), ("gamma", c_float), ("tau", c_float),
                ("lr", c_float), ("beta1", c_float), ("beta2", c_float), ("eps", c_float), ("target_policy_noise", c_float),
                ("target_noise_clip", c_float), ("seed", c_uint64), ("gemm_mode", c_int32), ("n_critics", c_int32)]


class Td3State(Structure):
    """struct cstr_td3_state"""

    _fields_ = [("params", c_void_p), ("targets", c_void_p), ("grads", c_void_p), ("adam_m", c_void_p), ("adam_v", c_void_p),
                ("workspace", c_void_p), ("workspace_bytes", c_int64), ("losses", c_void_p), ("counters", c_void_p), ("peer", c_void_p)]


PEER_MAX_WORLD = 8


class PeerComm(Structure):
    """struct cstr_peer_comm"""

    _fields_ = [("world", c_int32), ("rank", c_int32), ("grads", c_void_p * PEER_MAX_WORLD), ("flags", c_void_p * PEER_MAX_WORLD)]


class SacConfig(Structure):
    """struct cstr_sac_config"""

    _fields_ = [("h1", c_int32), ("h2", c_int32), ("batch", c_int32), ("target_update_interval", c_int32), ("gamma", c_float), ("tau", c_float),
                ("lr", c_float), ("beta1", c_float), ("beta2", c_float), ("eps", c_float), ("target_entropy", c_float), ("reserved0", c_float),
                ("seed", c_uint64), ("gemm_mode", c_int32), ("local_step", c_int32)]


class BcqConfig(Structure):
    """struct cstr_bcq_config"""

    _fields_ = [("latent", c_int32), ("vae_hidden", c_int32), ("pert_hidden", c_int32), ("h1", c_int32), ("h2", c_int32), ("batch", c_int32),
                ("actor_delay", c_int32), ("n_candidates", c_int32), ("gamma", c_float), ("tau", c_float), ("lr", c_float), ("beta1", c_float),
                ("beta2", c_float), ("eps", c_float), ("max_perturbation", c_float), ("reserved0", c_float), ("seed", c_uint64),
                ("gemm_mode", c_int32), ("reserved1", c_int32)]


class MaConfig(Structure):
    """struct cstr_ma_config"""

    _fields_ = [("centralised", c_int32), ("h1", c_int32), ("h2", c_int32), ("batch", c_int32), ("policy_delay", c_int32), ("n_critics", c_int32),
                ("gamma", c_float), ("tau", c_float), ("beta1", c_float), ("beta2", c_float), ("eps", c_float), ("target_policy_noise", c_float),
                ("target_noise_clip", c_float), ("reserved0", c_float), ("actor_lr", c_float * 2), ("critic_lr", c_float * 2), ("seed", c_uint64),
                ("gemm_mode", c_int32), ("reserved1", c_int32)]


TD3_CRITIC_GRAD, TD3_CRITIC_APPLY, TD3_ACTOR_GRAD, TD3_ACTOR_APPLY, TD3_ALL = 1, 2, 4, 8, 15

P = c_void_p
_SIGNATURES = {
    # name: (restype, argtypes)  — mirrors include/cstr_b200.h one to one
    "cstr_b200_abi_version": (c_int, []),
    "cstr_last_error": (c_char_p, []),
    "cstr_device_info": (c_int, [POINTER(c_int), POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "cstr_reset": (c_int, [POINTER(EnvParams), c_int64, P, P, c_int, P, P, P, P]),
    "cstr_vec_step_f32": (c_int, [POINTER(EnvParams), c_int64, c_int, c_int, P, P, P, P, P, P, P, P, P, P, P, P, P]),
    "cstr_vec_step_f64": (c_int, [POINTER(EnvParams), c_int64, c_int, P, P, P, P, P, P, P, P, P, P, P, P, P]),
    "cstr_tape_f32": (c_int, [POINTER(EnvParams), c_int64, c_int64, c_int, P, c_uint32, P, P, P, P, P, P, P, P, P]),
    "cstr_tape_f64": (c_int, [POINTER(EnvParams), c_int64, c_int64, P, c_uint32, P, P, P, P, P, P, P, P, P]),
    "cstr_tape_f32_host": (c_int, [POINTER(EnvParams), c_int64, c_int64, c_int, P, P, P, P, P, P, P]),
    "cstr_replay_add": (c_int, [c_int64, c_int64, P, P, P, P, P, P, P, P]),
    "cstr_replay_sample": (c_int, [c_int64, c_int64, P, P, P, P, P, P, P, P, POINTER(NormParams), P]),
    "cstr_replay_sample_philox": (c_int, [c_uint64, c_uint64, c_int64, c_int64, c_int64, P, P, P, P, P, P, P, P, POINTER(NormParams), P]),
    "cstr_replay_sample_philox_dev": (c_int, [c_uint64, P, c_int64, c_int64, c_int64, P, P, P, P, P, P, P, P, POINTER(NormParams), P]),
    "cstr_norm_update": (c_int, [c_int64, P, P, P, P, c_double, P, P, P]),
    "cstr_norm_apply": (c_int, [c_int64, P, P, P, c_double, c_double, c_double, P, P, P]),
    "cstr_td3_param_count": (c_int64, [c_int32, c_int32]),
    "cstr_td3_layout": (c_int, [c_int32, c_int32, POINTER(c_int64)]),
    "cstr_td3_workspace_bytes": (c_int64, [POINTER(Td3Config)]),
    "cstr_td3_update": (c_int, [POINTER(Td3Config), POINTER(Td3State), P, P, P, P, P, P, c_int64, c_int64, c_int64, c_int32, P]),
    "cstr_sac_param_count": (c_int64, [c_int32, c_int32]),
    "cstr_sac_layout": (c_int, [c_int32, c_int32, POINTER(c_int64)]),
    "cstr_sac_workspace_bytes": (c_int64, [POINTER(SacConfig)]),
    "cstr_sac_update": (c_int, [POINTER(SacConfig), POINTER(Td3State), P, P, P, P, P, P, P, c_int64, c_int64, c_int32, P]),
    "cstr_bcq_param_count": (c_int64, [POINTER(BcqConfig)]),
    "cstr_bcq_layout": (c_int, [POINTER(BcqConfig), POINTER(c_int64)]),
    "cstr_bcq_workspace_bytes": (c_int64, [POINTER(BcqConfig)]),
    "cstr_bcq_update": (c_int, [POINTER(BcqConfig), POINTER(Td3State), P, P, P, P, P, P, P, P, c_int64, c_int64, c_int64, P]),
    "cstr_ma_param_count": (c_int64, [POINTER(MaConfig)]),
    "cstr_ma_layout": (c_int, [POINTER(MaConfig), POINTER(c_int64)]),
    "cstr_ma_workspace_bytes": (c_int64, [POINTER(MaConfig)]),
    "cstr_ma_update": (c_int, [POINTER(MaConfig), POINTER(Td3State), P, P, P, P, P, P, c_int64, c_int64, c_int64, P]),
    "cstr_peer_flag_bytes": (c_int64, []),
    "cstr_peer_alloc": (c_int, [c_int64, POINTER(c_void_p), P]),
    "cstr_peer_open": (c_int, [P, POINTER(c_void_p)]),
    "cstr_peer_close": (c_int, [P]),
    "cstr_peer_free": (c_int, [P]),
    "cstr_peer_error": (c_int, [POINTER(PeerComm), POINTER(c_uint32), P]),
    "cstr_rollout_fused": (c_int, [POINTER(EnvParams), c_int64, c_int64, c_int, c_int, POINTER(ActorF32), P, c_float, P, c_int,
                                   c_uint32, P, P, P, P, c_int64, c_int64, P, P, POINTER(EpisodeStatsStruct), P]),
    "cstr_rollout_norm_workspace_bytes": (c_int64, [c_int64, c_int]),
    "cstr_rollout_fused_norm": (c_int, [POINTER(EnvParams), c_int64, c_int64, c_int, c_int, POINTER(ActorF32), P, c_float, P, c_int,
                                        c_uint32, P, P, P, P, c_int64, c_int64, P, P, POINTER(EpisodeStatsStruct), POINTER(RolloutNorm), P]),
    "cstr_rollout_fused_multi": (c_int, [POINTER(EnvParams), c_int64, c_int64, c_int, P, c_int, c_uint32, P, P, P, P, c_int64, c_int64, P, P,
                                         POINTER(EpisodeStatsStruct), P]),
    "cstr_actor_pack_bf16": (c_int64, [POINTER(ActorF32), P, P]),
    "cstr_probe_pipe": (c_int, [c_int, c_int64, c_int, c_int, P, P]),
    "cstr_selftest": (c_int, [c_int, P, P]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib: Optional[ctypes.CDLL] = None


def library_path() -> str:
    return _build.LIB_PATH


def load(build_if_missing: bool = True) -> ctypes.CDLL:
    """dlopen libcstr_b200.so (building it in-tree first if it is missing or stale and nvcc exists)."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB_PATH
    if build_if_missing and _build.is_stale():
        try:
            _build.build()
        except Exception as exc:  # a missing library is fatal; a present-but-older one is used, loudly (the ABI check below still applies)
            if not os.path.exists(path):
                raise CstrLibraryError(f"libcstr_b200.so is missing and could not be built: {exc}") from exc
            import warnings

            warnings.warn(f"libcstr_b200.so is older than its sources and the rebuild failed ({exc}); loading the stale library",
                          RuntimeWarning, stacklevel=2)
    if not os.path.exists(path):
        raise CstrLibraryError(f"{path} not found — run `python __graft_entry__.py build` (no CPU fallback exists)")
    try:
        lib = ctypes.CDLL(path)
    except OSError as exc:
        raise CstrLibraryError(f"could not load {path}: {exc}") from exc
    for name, (restype, argtypes) in _SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as exc:
            raise CstrLibraryError(f"{path} does not export {name} (stale build?)") from exc
        fn.restype = restype
        fn.argtypes = argtypes
    got = lib.cstr_b200_abi_version()
    if got != ABI_VERSION:
        raise CstrLibraryError(f"ABI version mismatch: library {got}, binding {ABI_VERSION} — rebuild")
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().cstr_last_error()
        raise CstrLibraryError(f"{what} failed (code {rc}): {msg.decode() if msg else '?'}")


def require_cuda():
    """Import torch and insist on a CUDA device — the product has no CPU path."""
    import torch

    if not torch.cuda.is_available():
        raise CstrLibraryError("no CUDA device: the CSTR kernels are sm_100a-only and have no CPU fallback")
    return torch


def ptr(t) -> Optional[int]:
    """data_ptr of a torch tensor (None passes NULL)."""
    return None if t is None else t.data_ptr()


def stream_handle(torch_stream=None) -> int:
    import torch

    s = torch_stream if torch_stream is not None else torch.cuda.current_stream()
    return s.cuda_stream
