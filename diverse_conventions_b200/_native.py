"""ctypes binding of the C ABI (include/ocb.h) — the only way Python reaches the kernels.

There is deliberately no fallback: if ``libocb.so`` is missing or a call fails, an
exception is raised.
"""
from __future__ import annotations

import ctypes
import os
import re
from typing import List

from . import build as _build
from .layouts import ocb_config

OCB_OK = 0
ACT_I32, ACT_I64, ACT_F32, ACT_U8 = 0, 1, 2, 3

_lib = None

_vp = ctypes.c_void_p
_i = ctypes.c_int
_u32 = ctypes.c_uint32
_u64 = ctypes.c_uint64
_sz = ctypes.c_size_t
_pp = ctypes.POINTER(ctypes.c_void_p)

# name -> (restype, argtypes); must list every function declared in include/ocb.h
PROTOTYPES = {
    "ocb_abi_version": (_i, []),
    "ocb_last_error": (ctypes.c_char_p, []),
    "ocb_device_count": (_i, []),
    "ocb_create": (_i, [ctypes.POINTER(ocb_config), _i, _u32, _u64, _pp]),
    "ocb_destroy": (_i, [_vp]),
    "ocb_num_worlds": (_i, [_vp]),
    "ocb_num_players": (_i, [_vp]),
    "ocb_obs_channels": (_i, [_vp]),
    "ocb_obs_bytes_per_agent": (_i, [_vp]),
    "ocb_state_ints_per_world": (_i, [_vp]),
    "ocb_set_tuning": (_i, [_vp, _i, _i]),
    "ocb_get_tuning": (_i, [_vp, ctypes.POINTER(_i), ctypes.POINTER(_i), ctypes.POINTER(_i)]),
    "ocb_reset": (_i, [_vp, _vp, _vp]),
    "ocb_observe": (_i, [_vp, _vp, _vp]),
    "ocb_step": (_i, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "ocb_step_ex": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "ocb_rollout_actions": (_i, [_vp, _i, _vp, _i, _vp, _vp, _vp, _vp]),
    "ocb_rollout_random": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "ocb_step_host": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "ocb_step_host_async": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "ocb_step_host_wait": (_i, [_vp]),
    "ocb_get_state": (_i, [_vp, _vp, _sz]),
    "ocb_set_state": (_i, [_vp, _vp, _sz]),
    "ocb_read_episode_stats": (_i, [_vp, _vp, _vp, _vp]),
    "ocb_clear_episode_stats": (_i, [_vp, _vp]),
    "ocb_step_count": (_u64, [_vp]),
    "ocb_set_world_offset": (_i, [_vp, _u32]),
    "ocb_policy_create": (_i, [ctypes.POINTER(ocb_config), _i, _i, _i, _pp]),
    "ocb_policy_destroy": (_i, [_vp]),
    "ocb_policy_set_weights": (_i, [_vp, _i, _i] + [_vp] * 8),
    "ocb_policy_act": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _i, _u64, _u64, _vp]),
    "ocb_policy_act_ex": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _i, _u64, _u64, _vp, _vp]),
    "ocb_policy_value": (_i, [_vp, _vp, _i, _vp, _vp, _vp]),
    "ocb_policy_forward": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _u64, _u64, _vp, _vp]),
    "ocb_policy_set_sampling_rows": (_i, [_vp, _u32, _u32, _u32]),
    "ocb_policy_info": (_i, [_vp, ctypes.POINTER(_i), ctypes.POINTER(_i), ctypes.POINTER(_i)]),
    "ocb_policy_reserve": (_i, [_vp, _i]),
    "ocb_policy_debug_profile": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _i]),
    "ocb_step_counter_device": (_vp, [_vp]),
    "ocb_rollout_policy": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _u64, _vp]),
    "ocb_rollout_policy_fused": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _u64, _vp]),
    "ocb_rollout_crossplay_fused": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _u64, _vp]),
    "ocb_rollout_population_fused": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _u64, _vp]),
    "ocb_rollout_fused_debug_trace": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _u64, _vp, _i, _i]),
    "ocb_rollout_mixed_scratch_bytes": (_sz, [_vp]),
    "ocb_rollout_mixed": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _u64, _u64, _vp, _sz, _vp]),
    "ocb_rollout_mixed_fused": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _u64, _u64, _vp]),
    "ocb_compute_returns": (_i, [_i, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ocb_compute_returns_dev": (_i, [_i, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ocb_normalize_advantages": (_i, [_i, _vp, _sz, _vp, _vp]),
    "ocb_policy_evaluate": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ocb_minibatch_gather": (_i, [_i, _vp, _i, _i, _vp, _vp, _i, _i, _pp, _pp, _i, _pp, _pp, _vp]),
    "ocb_ppo_loss": (_i, [_i, _vp, _i] + [_vp] * 15),
    "bb_create": (_i, [_i, _u32, _u64, _pp]),
    "bb_destroy": (_i, [_vp]),
    "bb_num_worlds": (_i, [_vp]),
    "bb_reset": (_i, [_vp, _vp, _vp]),
    "bb_observe": (_i, [_vp, _vp, _vp]),
    "bb_step": (_i, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "bb_rollout_random": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "bb_get_state": (_i, [_vp, _vp, _sz]),
    "bb_set_state": (_i, [_vp, _vp, _sz]),
}


class NativeError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__("libocb error %d: %s" % (code, message))
        self.code = code


def header_path() -> str:
    return os.path.join(os.path.dirname(_build.HERE), "include", "ocb.h")


def declared_symbols() -> List[str]:
    """Function names declared in include/ocb.h (parsed, so the header stays the source of truth)."""
    with open(header_path()) as f:
        text = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    names = re.findall(r"\b((?:ocb|bb)_[a-z0-9_]+)\s*\(", text)
    return sorted(set(names))


def lib(build_if_missing: bool = True):
    """Load (building first if the sources are newer) and return the ctypes library."""
    global _lib
    if _lib is None:
        path = _build.LIB_PATH
        if build_if_missing and _build.is_stale() and _build.find_nvcc() is not None:
            _build.build_native()
        if not os.path.exists(path):
            raise ImportError(
                "%s is missing: build it with `python -m diverse_conventions_b200.build` "
                "(there is no CPU fallback)" % path)
        L = ctypes.CDLL(path)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(L, name)  # AttributeError if the .so lacks a declared symbol
            fn.restype, fn.argtypes = res, args
        if L.ocb_abi_version() != 1:
            raise ImportError("libocb.so ABI version mismatch")
        _lib = L
    return _lib


OCB_ERR_UNSUPPORTED = -6


def check(code: int) -> int:
    if code < 0:
        raise NativeError(code, lib().ocb_last_error().decode("utf-8", "replace"))
    return code
