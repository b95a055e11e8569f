"""Builds and binds tests/host_sim, the CPU build of the CUDA core's device source (host_sim/host_sim.cpp), for the host_sim
test modules: one g++ command line, one declaration of every hs_* entry point, one library per set of build flags."""
import ctypes
import functools
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST_SIM = os.path.join(ROOT, "tests", "host_sim")

vp, i32, u64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint64
# name -> (restype, argtypes)
SIGNATURES = {
    "hs_create": (vp, [ctypes.c_char_p]),
    "hs_create_colours": (vp, [ctypes.c_char_p, vp, vp, vp]),
    "hs_destroy": (None, [vp]),
    "hs_env_reset": (None, [vp, i32]),
    "hs_env_power_on": (None, [vp]),
    "hs_env_run_frame": (i32, [vp, i32, i32, i32, i32, i32] + [vp] * 6),
    "hs_env_step_fast": (i32, [vp, i32] + [vp] * 4),
    "hs_env_step": (i32, [vp, i32] + [vp] * 7),
    "hs_evaluate": (None, [vp, i32, vp, i32, i32, i32, i32, i32, vp, i32, vp, vp, i32, vp, u64, u64, vp, vp]),
    "hs_validate_state": (i32, [vp, u64]),
    "hs_play_list": (ctypes.c_long, [vp, i32, vp, i32, i32, i32, vp, i32, vp, vp, vp, vp, i32, vp, i32, vp, i32, vp, vp, i32, vp, u64,
                                     u64, u64, vp, vp, vp, vp]),
    "hs_hot_latch_selftest": (i32, [u64, i32]),
}
STATS_SIGNATURE = (ctypes.POINTER(ctypes.c_ulonglong * 16), [])       # hs_stats: -DA26_STATS builds only


@functools.lru_cache(maxsize=None)
def library(variant: str = "", flags: tuple = ()) -> ctypes.CDLL:
    """tests/host_sim/libhost_sim[_<variant>].so built with `flags` (host_sim_stats.cpp added for -DA26_STATS), loaded and
    declared; built once per process."""
    lib = os.path.join(HOST_SIM, f"libhost_sim_{variant}.so" if variant else "libhost_sim.so")
    srcs = [os.path.join(HOST_SIM, "host_sim.cpp")] + ([os.path.join(HOST_SIM, "host_sim_stats.cpp")] if "-DA26_STATS" in flags else [])
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-Wno-unknown-pragmas", *flags, "-o", lib, *srcs])
    L = ctypes.CDLL(lib)
    signatures = dict(SIGNATURES, **({"hs_stats": STATS_SIGNATURE} if "-DA26_STATS" in flags else {}))
    for name, (restype, argtypes) in signatures.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = restype, argtypes
    return L
