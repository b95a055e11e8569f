"""ctypes bindings of libngp.so (include/ngp.h).  There is no CPU fallback: if the CUDA library
cannot be loaded, importing anything that computes raises."""
from __future__ import annotations

import ctypes
import os

from . import build as _build

NGP_MAX_LAYERS = 8
ACT_NONE, ACT_UP, ACT_DOWN = 0, 1, 2
STATE_START_1P, STATE_START_2P = 0, 1
SCHEDULE_REFERENCE, SCHEDULE_ROUND_ROBIN = 0, 1
CORE_INTERPRETER, CORE_TRANSLATED = 0, 1
# left-player codes of ngp_play_matches that are not genome rows (include/ngp.h NGP_OPP_*)
OPP_HARDCODED, OPP_SCORE_HARDCODED, OPP_ROBOT = -1, -2, -3
# a seat of a match session whose decisions the caller supplies (include/ngp.h NGP_PLAYER_EXTERNAL)
PLAYER_EXTERNAL = -4
# bits of a match session's per-match flags (include/ngp.h NGP_SESSION_*)
SESSION_NEED, SESSION_DONE, SESSION_EMULATOR_ERROR = 1, 2, 4
# sizeof(ngp_frame_record) (include/ngp.h): one recorded frame of ngp_record_matches
NGP_FRAME_RECORD_BYTES = 32
# sizeof(ngp_game_state) (include/ngp.h): one save state of a game
NGP_GAME_STATE_BYTES = 512
# button map codes (include/ngp.h NGP_BTN_*): fire of paddle p = BTN_FIRE_P0 + p; paddle p up / down = BTN_UP_P0 + 2p / + 2p + 1
BTN_NONE, BTN_FIRE_P0, BTN_UP_P0, BTN_SELECT, BTN_RESET = 0, 1, 5, 13, 14

EXPORTS = [
    "ngp_default_config", "ngp_last_error", "ngp_version", "ngp_create", "ngp_destroy", "ngp_gene_size",
    "ngp_env_reset", "ngp_env_step", "ngp_env_step_core", "ngp_env_digest", "ngp_find_stuff", "ngp_mlp_forward", "ngp_evaluate",
    "ngp_evaluate_host", "ngp_ga_step", "ngp_init_population", "ngp_launch_count", "ngp_profile_enable", "ngp_profile_read",
    "ngp_config_size", "ngp_set_option", "ngp_select", "ngp_mate", "ngp_mutate", "ngp_hof_update", "ngp_exchange_bytes",
    "ngp_pack_elites", "ngp_unpack_elites", "ngp_mlp_prepare", "ngp_mlp_forward_prepared",
    "ngp_play_matches", "ngp_record_matches", "ngp_env_get_state", "ngp_env_set_state", "ngp_play_matches_states",
    "ngp_play_matches_stepwise", "ngp_session_begin", "ngp_session_step", "ngp_session_status", "ngp_session_end",
]


class NgpConfig(ctypes.Structure):
    _fields_ = [
        ("n_layers", ctypes.c_int32), ("nodes", ctypes.c_int32 * NGP_MAX_LAYERS), ("bias", ctypes.c_int32),
        ("games_to_play", ctypes.c_int32), ("win_score", ctypes.c_int32), ("timeout_thresh", ctypes.c_int32),
        ("schedule", ctypes.c_int32), ("max_frames", ctypes.c_int32), ("time_scaler", ctypes.c_float),
        ("scaled_paddle_height", ctypes.c_float), ("ball_colour", ctypes.c_uint8 * 3), ("left_colour", ctypes.c_uint8 * 3),
        ("right_colour", ctypes.c_uint8 * 3), ("pad_", ctypes.c_uint8 * 3),
        ("cxpb", ctypes.c_float), ("cx_alpha", ctypes.c_float), ("mutpb", ctypes.c_float), ("mut_mu", ctypes.c_float),
        ("mut_sigma", ctypes.c_float), ("mut_indpb", ctypes.c_float), ("tournament_size", ctypes.c_int32), ("core", ctypes.c_int32),
        ("button_map", ctypes.c_uint8 * 16),
    ]


class NgpNoise(ctypes.Structure):
    _fields_ = [("sel_draws", ctypes.c_void_p), ("cx_do", ctypes.c_void_p), ("cx_u", ctypes.c_void_p),
                ("mut_do", ctypes.c_void_p), ("mut_u", ctypes.c_void_p), ("mut_z", ctypes.c_void_p)]


class NgpError(RuntimeError):
    pass


_lib = None


def lib_path() -> str:
    return _build.LIB_PATH


def load(build_if_missing: bool = True):
    """Load libngp.so (building it in-tree with nvcc when absent)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_build.LIB_PATH):
        if not build_if_missing:
            raise NgpError(f"{_build.LIB_PATH} is missing and there is no CPU fallback; run __graft_entry__.build()")
        _build.build()
    # NGP_LIBRARY: another build of the same sources (kernel experiments: tools/ variants); the default is the in-tree library
    L = ctypes.CDLL(os.environ.get("NGP_LIBRARY") or _build.LIB_PATH)
    vp, i32, u64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_uint64
    L.ngp_config_size.restype = i32
    if L.ngp_config_size() != ctypes.sizeof(NgpConfig):
        raise NgpError(f"ngp_config layout mismatch: library {L.ngp_config_size()} bytes, binding {ctypes.sizeof(NgpConfig)}")
    L.ngp_default_config.argtypes = [ctypes.POINTER(NgpConfig), i32]; L.ngp_default_config.restype = None
    L.ngp_last_error.restype = ctypes.c_char_p
    L.ngp_version.restype = ctypes.c_char_p
    L.ngp_create.argtypes = [ctypes.POINTER(NgpConfig), ctypes.c_char_p, i32, ctypes.POINTER(vp)]
    L.ngp_destroy.argtypes = [vp]
    L.ngp_gene_size.argtypes = [vp]; L.ngp_gene_size.restype = i32
    L.ngp_env_reset.argtypes = [vp, i32, i32, vp]
    L.ngp_env_step.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    L.ngp_env_step_core.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp, vp]
    L.ngp_env_digest.argtypes = [vp, vp, vp]
    L.ngp_find_stuff.argtypes = [vp, vp, i32, vp, vp, vp]
    L.ngp_mlp_forward.argtypes = [vp, vp, vp, i32, i32, vp, vp, vp]
    L.ngp_mlp_prepare.argtypes = [vp, vp, i32, vp]
    L.ngp_mlp_forward_prepared.argtypes = [vp, vp, vp, i32, i32, vp, vp, vp]
    L.ngp_evaluate.argtypes = [vp, vp, i32, vp, vp, i32, vp, u64, u64, vp, vp, vp, ctypes.POINTER(u64), vp]
    L.ngp_play_matches.argtypes = [vp, vp, i32, vp, vp, vp, i32, u64, u64, vp, vp, vp, ctypes.POINTER(u64), vp]
    L.ngp_record_matches.argtypes = [vp, vp, i32, vp, vp, vp, vp, i32, u64, u64, i32, vp, vp, vp, vp, ctypes.POINTER(u64), vp]
    L.ngp_env_get_state.argtypes = [vp, vp, vp]
    L.ngp_env_set_state.argtypes = [vp, vp, i32, vp]
    L.ngp_play_matches_states.argtypes = [vp, vp, i32, vp, vp, vp, vp, i32, vp, i32, vp, i32, vp, vp, i32, vp, u64, u64, vp, vp, vp,
                                          ctypes.POINTER(u64), vp]
    L.ngp_play_matches_stepwise.argtypes = L.ngp_play_matches_states.argtypes
    L.ngp_session_begin.argtypes = [vp, vp, i32, vp, vp, vp, vp, i32, vp, i32, vp, i32, i32, vp, u64, u64, vp, vp, vp, vp, vp, vp,
                                    ctypes.POINTER(vp)]
    L.ngp_session_step.argtypes = [vp, vp, vp, vp, vp, vp]
    L.ngp_session_status.argtypes = [vp, ctypes.POINTER(i32), ctypes.POINTER(u64), vp]
    L.ngp_session_end.argtypes = [vp]
    L.ngp_evaluate_host.argtypes = [vp, vp, i32, vp, vp, i32, u64, u64, vp, ctypes.POINTER(u64)]
    L.ngp_ga_step.argtypes = [vp, vp, vp, i32, u64, u64, ctypes.POINTER(NgpNoise), vp, vp, vp, vp, vp]
    L.ngp_init_population.argtypes = [vp, vp, i32, u64, vp]
    L.ngp_launch_count.argtypes = [vp]; L.ngp_launch_count.restype = u64
    L.ngp_profile_enable.argtypes = [vp, i32]
    L.ngp_profile_read.argtypes = [vp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(i32)]
    L.ngp_set_option.argtypes = [vp, ctypes.c_char_p, ctypes.c_int64]
    L.ngp_select.argtypes = [vp, vp, i32, i32, vp, u64, u64, vp, vp]
    L.ngp_mate.argtypes = [vp, vp, vp, vp, i32, u64, u64, vp]
    L.ngp_mutate.argtypes = [vp, vp, vp, vp, i32, u64, u64, vp]
    L.ngp_hof_update.argtypes = [vp, vp, vp, ctypes.POINTER(i32), i32, vp, vp, i32, vp]
    L.ngp_exchange_bytes.argtypes = [vp, i32, i32]; L.ngp_exchange_bytes.restype = ctypes.c_int64
    L.ngp_pack_elites.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp, vp]
    L.ngp_unpack_elites.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, vp]
    _lib = L
    return L


def check(rc: int, what: str):
    if rc != 0:
        raise NgpError(f"{what} failed ({rc}): {load().ngp_last_error().decode()}")
