"""CPU-side check of the match-list form of the fused rollout (ngp_play_matches): tests/host_sim runs
csrc/rollout.cuh's plan_env with an explicit list, and every match must equal the oracle's perform_episode with the same
opponent, start state, multiplier and random key (environment index = match index): reward, frame count and both scores.
The list holds pairings neither built-in schedule can express."""
import ctypes

import numpy as np
import pytest

import oracle
from host_sim_lib import library

vp = ctypes.c_void_p

OPP_HARDCODED, OPP_SCORE_HARDCODED, OPP_ROBOT = -1, -2, -3        # include/ngp.h NGP_OPP_*

# (right row, left row or NGP_OPP_* code, multiplier); row 4 only ever plays on the left
MATCHES = [
    (0, 0, 1.0),                      # a genome against itself
    (1, 2, 1.0),
    (2, OPP_HARDCODED, 1.0),
    (3, OPP_SCORE_HARDCODED, 1.0),
    (0, OPP_ROBOT, 1.0),
    (1, 4, 1.0),                      # left-only genome
    (3, 1, 0.37),                     # hall-of-fame multiplier on a genome opponent
    (2, OPP_SCORE_HARDCODED, 2.5),    # ... and on a scripted one
    (1, 2, 1.0),                      # match 1 again, at another match index = random key
    (3, 4, 1.0),
    (2, OPP_ROBOT, 0.5),
    (0, OPP_HARDCODED, 1.0),
]


@pytest.fixture(scope="module")
def hs():
    L = library()
    return L, vp(L.hs_create(oracle.load_rom()))


def P(a):
    return a.ctypes.data_as(vp)


def oracle_match(shape, genomes, right, left, mult, seed, generation, m):
    """perform_episode of match m through the oracle (main.py:69-112), opponent and start state as main.evaluate picks them."""
    env = oracle.Atari()
    env.reset_to_state(oracle.STATE_START_1P if left == OPP_ROBOT else oracle.STATE_START_2P)
    opp = ("mlp", genomes[left]) if left >= 0 else ("score", None) if left == OPP_SCORE_HARDCODED else ("hardcoded", None)
    res, _ = env.episode(shape, opp, ("mlp", genomes[right]), mult=mult, seed=seed, env_id=m, generation=generation)
    return res


@pytest.mark.parametrize("core", [0, 1])
def test_match_list_matches_oracle(hs, core):
    L, sim = hs
    rng = np.random.RandomState(3)
    nodes = np.array([6, 2, 2], np.int32)
    genomes = (rng.standard_normal((5, 20)) * 2).astype(np.float32)
    right = np.array([m[0] for m in MATCHES], np.int32)
    left = np.array([m[1] for m in MATCHES], np.int32)
    mult = np.array([m[2] for m in MATCHES], np.float64)
    n = len(MATCHES)
    rew = np.zeros(n); frm = np.zeros(n, np.int32); sc = np.zeros((n, 2), np.int32)
    seed, generation = 21, 3
    L.hs_play_list(sim, core, P(nodes), 3, 1, 0, P(genomes), len(genomes), P(right), P(left), P(mult), None, n, None, 0, None, 0, None,
                   None, 0, None, 0, seed, generation, P(rew), P(frm), P(sc), None)
    shape = oracle.Shape.make([6, 2, 2])
    for m in range(n):
        res = oracle_match(shape, genomes, int(right[m]), int(left[m]), float(mult[m]), seed, generation, m)
        assert (rew[m], frm[m], sc[m, 0], sc[m, 1]) == (res.reward, res.frames, res.score1, res.score2), m
    assert len(set(zip(rew.tolist(), frm.tolist()))) >= n // 2          # the list is not one game played twelve times
