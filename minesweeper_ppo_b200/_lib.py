"""ctypes binding of libmsw_b200.so (include/msw_b200.h).

There is no CPU fallback: if the CUDA library is missing or fails to load, importing
callers get a RuntimeError telling them to build it.
"""
from __future__ import annotations

import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libmsw_b200.so")

MSW_VERSION = 1
OBS_CHANNELS = 10
MAX_CELLS = 1024


class EnvDesc(C.Structure):          # msw_env_desc
    _fields_ = [
        ("H", C.c_int32), ("W", C.c_int32), ("mine_count", C.c_int32), ("safe_nbhd", C.c_int32),
        ("reward_step", C.c_float), ("reward_loss", C.c_float), ("reward_win", C.c_float),
        ("reserved", C.c_int32), ("seed", C.c_uint64), ("env_id_base", C.c_int64),
    ]


class State(C.Structure):            # msw_state
    _fields_ = [("mines", C.c_void_p), ("revealed", C.c_void_p), ("flags", C.c_void_p), ("meta", C.c_void_p)]


class EncodeOut(C.Structure):        # msw_encode_out
    _fields_ = [("obs", C.c_void_p), ("mask", C.c_void_p), ("mine_labels", C.c_void_p), ("mine_valid", C.c_void_p)]


class StepIO(C.Structure):           # msw_step_io
    _fields_ = [
        ("actions32", C.c_void_p), ("actions64", C.c_void_p), ("inject_bits", C.c_void_p),
        ("inject_sel", C.c_void_p), ("reward", C.c_void_p), ("done", C.c_void_p), ("outcome", C.c_void_p),
        ("new_reveals", C.c_void_p), ("step", C.c_void_p), ("revealed_count", C.c_void_p), ("enc", EncodeOut),
        ("rand_mode", C.c_int32), ("rand_step", C.c_uint32), ("rand_seed", C.c_uint64), ("actions_out32", C.c_void_p),
    ]


class HostOut(C.Structure):          # msw_host_out
    _fields_ = [
        ("obs", C.c_void_p), ("mask", C.c_void_p), ("reward", C.c_void_p), ("done", C.c_void_p),
        ("outcome", C.c_void_p), ("new_reveals", C.c_void_p), ("step", C.c_void_p), ("revealed_count", C.c_void_p),
        ("stage", C.c_void_p), ("threads", C.c_int32), ("shadow_valid", C.c_int32), ("shadow", C.c_void_p),
    ]


# every symbol include/msw_b200.h declares: name -> (restype, argtypes)
_P = C.POINTER
SIGNATURES = {
    "msw_version": (C.c_int, []),
    "msw_last_error": (C.c_char_p, []),
    "msw_words_per_board": (C.c_int, [C.c_int32, C.c_int32]),
    "msw_reset": (C.c_int, [_P(EnvDesc), _P(State), C.c_int64, _P(EncodeOut), C.c_void_p]),
    "msw_step": (C.c_int, [_P(EnvDesc), _P(State), _P(StepIO), C.c_int64, C.c_void_p]),
    "msw_encode": (C.c_int, [_P(EnvDesc), _P(State), C.c_int64, _P(EncodeOut), C.c_void_p]),
    "msw_unpack_state": (C.c_int, [_P(EnvDesc), _P(State), C.c_int64] + [C.c_void_p] * 5),
    "msw_random_actions": (C.c_int, [_P(EnvDesc), _P(State), C.c_int64, C.c_uint64, C.c_uint32, C.c_int32,
                                     C.c_void_p, C.c_void_p, C.c_void_p]),
    "msw_gae": (C.c_int, [C.c_void_p] * 6 + [C.c_int64, C.c_int64, C.c_float, C.c_float, C.c_int32, C.c_void_p]),
    "msw_step_host": (C.c_int, [_P(EnvDesc), _P(State), _P(StepIO), C.c_void_p, _P(HostOut), C.c_int64, C.c_void_p]),
    "msw_expand_obs_host": (C.c_int, [_P(EnvDesc), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                      C.c_int32]),
    "msw_shadow_words": (C.c_int, [C.c_int32, C.c_int32]),
    "msw_expand_obs_host_delta": (C.c_int, [_P(EnvDesc), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_int32, C.c_int32]),
    "msw_masked_sample": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_int32, C.c_uint64,
                                    C.c_uint64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "msw_gn_act": (C.c_int, [C.c_void_p] * 7 + [C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_int32,
                             C.c_float, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                             C.c_void_p, C.c_int64, C.c_void_p]),
    "msw_pack_obs16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p]),
    "msw_cell_heads": (C.c_int, [C.c_void_p] * 7 + [C.c_int64, C.c_int32, C.c_void_p]),
    "msw_conv3x3": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                              C.c_void_p]),
    "msw_conv3x3_gn": (C.c_int, [C.c_void_p] * 9 + [C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_float,
                                 C.c_float, C.c_uint64, C.c_uint64, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]),
    "msw_cnn_forward": (C.c_int, [C.c_void_p] * 18 + [C.c_int64] + [C.c_int32] * 8 + [C.c_float, C.c_float, C.c_void_p]),
    "msw_gn_act_bwd": (C.c_int, [C.c_void_p] * 13 + [C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_void_p]),
    "msw_late_start": (C.c_int, [_P(EnvDesc), _P(State), C.c_int64, C.c_void_p, C.c_uint64, C.c_float, C.c_int32,
                                 C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "msw_gather_encode": (C.c_int, [_P(EnvDesc)] + [C.c_void_p] * 4 + [C.c_int64, C.c_void_p, C.c_int64,
                                    _P(EncodeOut), C.c_void_p]),
    "msw_forced_subset": (C.c_int, [_P(EnvDesc), _P(State), C.c_int64, C.c_void_p, C.c_void_p]),
    "msw_avoidability": (C.c_int, [_P(EnvDesc), _P(State), C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_uint32, C.c_void_p]),
    "msw_masked_argmax": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]),
    "msw_eval_pre_step": (C.c_int, [_P(EnvDesc), _P(State), C.c_int64, C.c_int64] + [C.c_void_p] * 11
                          + [C.c_int64, C.c_void_p]),
    "msw_eval_post_step": (C.c_int, [C.c_int64] + [C.c_void_p] * 6 + [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
}

# int64 counter slots of msw_eval_pre_step / msw_eval_post_step (enum in include/msw_b200.h)
EVAL_COUNTERS = (
    "invalid", "forced_steps", "forced_correct", "guess_attempts", "guess_success", "reveal_total",
    "forced_guess_total", "forced_guess_success", "safe_option_total", "safe_option_hits", "safe_option_misses",
    "safe_cells", "comp_size_sum", "comp_count", "chosen_size_sum", "chosen_count",
    "wins", "total_steps", "new_reveals", "forced_guess_episodes", "error_key",
)

_lib = None


def load() -> C.CDLL:
    """Load the CUDA library, failing loudly (no fallback of any kind)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: the B200 CUDA library has not been built. "
            "Run `python -m minesweeper_ppo_b200.build` (needs nvcc); there is no CPU fallback.")
    try:
        lib = C.CDLL(LIB_PATH)
    except OSError as e:
        raise RuntimeError(f"failed to load {LIB_PATH}: {e}; there is no CPU fallback") from e
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise RuntimeError(f"{LIB_PATH} does not export {name}; rebuild with "
                               "`python -m minesweeper_ppo_b200.build --force`") from e
        fn.restype, fn.argtypes = res, args
    v = lib.msw_version()
    if v != MSW_VERSION:
        raise RuntimeError(f"libmsw_b200.so version {v} != binding version {MSW_VERSION}; rebuild")
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().msw_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed (code {rc}): {msg}")
