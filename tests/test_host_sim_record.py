"""CPU-side check of the recording form of the fused rollout (ngp_record_matches): tests/host_sim/host_sim_record.cpp runs
csrc/rollout.cuh's episode_frame<.., REC = true> and record_frame over the irregular match list of test_host_sim_matches,
and every recorded frame must equal the oracle's perform_episode trace: both decisions, both scores, the three valid bits,
the timeout counter and the frame count.  With a key list, match m must equal the oracle run with env_id = key[m]."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import oracle
from test_host_sim_matches import MATCHES, OPP_ROBOT, OPP_SCORE_HARDCODED

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "host_sim", "host_sim_record.cpp")
LIB = os.path.join(ROOT, "tests", "host_sim", "libhost_sim_record.so")
vp = ctypes.c_void_p
MAX_RECORD = 12000
# include/ngp.h ngp_frame_record
FRAME_RECORD = np.dtype([("loc", "<f4", (3, 2)), ("valid", "u1"), ("score", "u1", (2,)), ("act", "u1"), ("timeout", "<i4")])
assert FRAME_RECORD.itemsize == 32


@pytest.fixture(scope="module")
def hs():
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", LIB, SRC])
    L = ctypes.CDLL(LIB)
    L.hs_create.restype = vp
    L.hs_record_matches.argtypes = [vp, ctypes.c_int, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, vp, ctypes.c_int,
                                    ctypes.c_uint64, ctypes.c_uint64, ctypes.c_int, vp, vp, vp, vp]
    return L, vp(L.hs_create(oracle.load_rom()))


def P(a):
    return None if a is None else a.ctypes.data_as(vp)


def oracle_trace(shape, genomes, right, left, mult, seed, generation, env_id):
    env = oracle.Atari()
    env.reset_to_state(oracle.STATE_START_1P if left == OPP_ROBOT else oracle.STATE_START_2P)
    opp = ("mlp", genomes[left]) if left >= 0 else ("score", None) if left == OPP_SCORE_HARDCODED else ("hardcoded", None)
    return env.episode(shape, opp, ("mlp", genomes[right]), mult=mult, seed=seed, env_id=env_id, generation=generation,
                       trace_cap=MAX_RECORD)


def check_against_oracle(rec, rew, frm, sc, genomes, right, left, mult, keys, seed, generation, sentinel=-12345):
    """rec: FRAME_RECORD[M, T]; entries past a game must still hold `sentinel` in timeout (None = not checked).  Returns the
    number of random fall-back frames (ball found, a paddle not)."""
    shape = oracle.Shape.make([6, 2, 2])
    fallback = 0
    for m in range(len(right)):
        res, tr = oracle_trace(shape, genomes, int(right[m]), int(left[m]), float(mult[m]), seed, generation, int(keys[m]))
        assert (rew[m], frm[m], sc[m, 0], sc[m, 1]) == (res.reward, res.frames, res.score1, res.score2), m
        T = int(frm[m])
        assert 0 < T <= MAX_RECORD and len(tr) == T, m
        r = rec[m, :T]
        assert np.array_equal(r["act"] & 3, tr[:, 128]) and np.array_equal(r["act"] >> 2, tr[:, 129]), m
        assert np.array_equal(r["score"][:, 0], tr[:, 130]) and np.array_equal(r["score"][:, 1], tr[:, 131]), m
        valid = tr[:, 132].astype(np.int32) | tr[:, 133].astype(np.int32) << 1 | tr[:, 134].astype(np.int32) << 2
        assert np.array_equal(r["valid"], valid), m
        assert np.array_equal(r["timeout"], tr[:, 136:140].copy().view("<u4")[:, 0].astype(np.int32)), m
        # centroids: 0 exactly where nothing was found
        for t in range(3):
            missing = (r["valid"] >> t & 1) == 0
            assert np.all(r["loc"][missing, t] == 0.0), (m, t)
        fallback += int(np.sum((valid & 1) == 1) - np.sum(valid == 7))
        if sentinel is not None:
            assert np.all(rec[m, T:]["timeout"] == sentinel), m                 # untouched past the game
    return fallback


@pytest.mark.parametrize("core", [0, 1])
@pytest.mark.parametrize("with_key", [False, True])
def test_record_matches_oracle_trace(hs, core, with_key):
    L, sim = hs
    rng = np.random.RandomState(3)
    nodes = np.array([6, 2, 2], np.int32)
    genomes = (rng.standard_normal((5, 20)) * 2).astype(np.float32)
    right = np.array([m[0] for m in MATCHES], np.int32)
    left = np.array([m[1] for m in MATCHES], np.int32)
    mult = np.array([m[2] for m in MATCHES], np.float64)
    n = len(MATCHES)
    keys = (np.array([7, 0, 123456, 3, 3, 99, 1, 2**31 - 1, 40, 11, 5, 8], np.int32) if with_key else np.arange(n, dtype=np.int32))
    rec = np.zeros((n, MAX_RECORD), FRAME_RECORD)
    rec["timeout"] = -12345
    rew = np.zeros(n); frm = np.zeros(n, np.int32); sc = np.zeros((n, 2), np.int32)
    seed, generation = 21, 3
    L.hs_record_matches(sim, core, P(nodes), 3, 1, 0, P(genomes), P(right), P(left), P(mult), P(keys) if with_key else None, n, seed,
                        generation, MAX_RECORD, P(rec), P(rew), P(frm), P(sc))
    check_against_oracle(rec, rew, frm, sc, genomes, right, left, mult, keys, seed, generation)


@pytest.mark.parametrize("core", [0, 1])
def test_key_drives_the_random_fall_back(hs, core):
    """With a left-paddle colour that matches nothing every frame with the ball in view takes get_actions' random fall-back
    (self-play between visible paddles showed none), so the key decides the game.  Match m played with key[m] must equal
    the keyless game at list position key[m] bit for bit, and its decisions must be the oracle's Philox draws for key[m]."""
    L, _ = hs
    L.hs_create_colours.restype = vp
    L.hs_create_colours.argtypes = [ctypes.c_char_p, vp, vp, vp]
    colour = lambda c: np.array(c, np.uint8)                                                    # noqa: E731
    ball, blind, right_c = colour([236, 236, 236]), colour([1, 2, 3]), colour([92, 186, 92])
    sim = vp(L.hs_create_colours(oracle.load_rom(), P(ball), P(blind), P(right_c)))
    nodes = np.array([6, 2, 2], np.int32)
    genomes = (np.random.RandomState(4).standard_normal((4, 20)) * 2).astype(np.float32)
    T, seed, generation = 300, 21, 3

    def run(right, left, keys):
        n = len(right)
        rec = np.zeros((n, T), FRAME_RECORD)
        rew = np.zeros(n); frm = np.zeros(n, np.int32); sc = np.zeros((n, 2), np.int32)
        L.hs_record_matches(sim, core, P(nodes), 3, 1, T, P(genomes), P(right), P(left), P(np.ones(n)), P(keys), n, seed, generation,
                            T, P(rec), P(rew), P(frm), P(sc))
        return rec, rew, frm, sc

    right = np.array([0, 1, 2, 3, 0], np.int32)
    left = np.array([1, 2, 3, 0, 2], np.int32)
    keys = np.array([6, 2, 0, 9, 4], np.int32)
    rec, rew, frm, sc = run(right, left, keys)
    # the keyless list with match m at position keys[m] (other positions: any pairing)
    r2, l2 = np.zeros(10, np.int32), np.ones(10, np.int32)
    r2[keys], l2[keys] = right, left
    rec2, rew2, frm2, sc2 = run(r2, l2, None)
    for m, k in enumerate(keys):
        assert (rew[m], frm[m]) == (rew2[k], frm2[k]) and np.array_equal(sc[m], sc2[k]), m
        assert rec[m].tobytes() == rec2[k].tobytes(), m
    # the same list without keys plays other games
    rec3, _, _, _ = run(right, left, None)
    assert rec3.tobytes() != rec.tobytes()
    bit = oracle.lib().eo_philox_bit
    for m, k in enumerate(keys):
        r = rec[m, :frm[m]]
        fb = np.nonzero((r["valid"] & 1) == 1)[0]
        assert np.all(r["valid"] >> 1 & 1 == 0) and len(fb) > 0, m          # left paddle never found; the ball is
        for t in fb:
            want = [oracle.ACT_DOWN if bit(seed, generation, int(k), int(t), p) else oracle.ACT_UP for p in (0, 1)]
            assert int(r["act"][t]) & 3 == want[0], (m, t)                   # left: no paddle found, so no bounds clamp
            # right: through the bounds clamp (the recorded row is the centroid rounded to float; rows within rounding of a
            # bound are skipped)
            row = float(r["loc"][t, 2, 0])
            if all(oracle.lib().eo_clamp(int(r["valid"][t] >> 2 & 1), row + d, want[1]) == oracle.lib().eo_clamp(
                    int(r["valid"][t] >> 2 & 1), row, want[1]) for d in (-1e-4, 1e-4)):
                assert int(r["act"][t]) >> 2 == oracle.lib().eo_clamp(int(r["valid"][t] >> 2 & 1), row, want[1]), (m, t)
