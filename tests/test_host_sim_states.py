"""CPU-side check of save states (ngp_play_matches_states): tests/host_sim/host_sim_states.cpp runs csrc/rollout.cuh's frame
code and csrc/game_state.cuh's pack / unpack / validate exactly as the recording twins of rollout_kernel call them, on both
6507 cores.  A resumed capture must replay the rest of the uninterrupted game bit for bit; captures must not depend on the core;
a fresh start from a capture must equal the oracle stepped to that frame and then playing a new episode; and no corrupted,
foreign or mismatched state may get past the list check."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import oracle
from test_host_sim_matches import MATCHES, OPP_ROBOT, OPP_SCORE_HARDCODED
from test_host_sim_record import FRAME_RECORD

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "host_sim", "host_sim_states.cpp")
LIB = os.path.join(ROOT, "tests", "host_sim", "libhost_sim_states.so")
vp = ctypes.c_void_p
STATE_BYTES = 512                     # include/ngp.h NGP_GAME_STATE_BYTES
MAX_RECORD = 12000
SENTINEL = -12345
SEED, GENERATION = 21, 3
NODES = np.array([6, 2, 2], np.int32)


def fnv1a64(data: bytes) -> int:
    h = 14695981039346656037
    for b in data:
        h = ((h ^ b) * 1099511628211) & (2**64 - 1)
    return h


def seal(state: np.ndarray) -> np.ndarray:
    """The checksum of DESIGN.md's state format, computed here independently: FNV-1a over the little-endian words 0..125."""
    s = state.copy()
    h = 14695981039346656037
    for w in s[:504].view("<u4").tolist():
        h = ((h ^ w) * 1099511628211) & (2**64 - 1)
    s[504:512] = np.frombuffer(np.uint64(h).tobytes(), np.uint8)
    return s


@pytest.fixture(scope="module")
def hs():
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", LIB, SRC])
    L = ctypes.CDLL(LIB)
    L.hs_create.restype = vp
    L.hs_validate_state.argtypes = [vp, ctypes.c_uint64]
    L.hs_play_states.restype = ctypes.c_long
    L.hs_play_states.argtypes = [vp, ctypes.c_int, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, ctypes.c_int, vp, vp, vp, vp,
                                 ctypes.c_int, vp, ctypes.c_int, vp, ctypes.c_int, vp, vp, ctypes.c_int, vp, ctypes.c_uint64,
                                 ctypes.c_uint64, ctypes.c_uint64, vp, vp, vp, vp]
    rom = oracle.load_rom()
    return L, vp(L.hs_create(rom)), fnv1a64(rom)


def P(a):
    return None if a is None else a.ctypes.data_as(vp)


def play(hs, core, genomes, right, left, mult, key=None, states=None, start=None, fresh=0, capture_at=None, record=True,
         cart=None, capture=None):
    """One hs_play_states call.  Returns (faults, dict of results); the record's timeout field starts at SENTINEL and the
    capture buffer at 0xAB (or `capture`)."""
    L, sim, cart0 = hs
    n = len(right)
    out = {"rewards": np.full(n, -1.0), "frames": np.full(n, -1, np.int32), "scores": np.full((n, 2), -1, np.int32),
           "total": ctypes.c_uint64(0)}
    rec = None
    if record:
        rec = np.zeros((n, MAX_RECORD), FRAME_RECORD)
        rec["timeout"] = SENTINEL
    cap = None
    if capture_at is not None:
        cap = np.full((n, STATE_BYTES), 0xAB, np.uint8) if capture is None else capture
    n_states = 0 if states is None else len(states)
    faults = L.hs_play_states(sim, core, P(NODES), 3, 1, 0, P(genomes), len(genomes), P(right), P(left), P(mult), P(key), n,
                              P(states), n_states, P(start), fresh, P(capture_at), P(cap), MAX_RECORD, P(rec),
                              cart0 if cart is None else cart, SEED, GENERATION, P(out["rewards"]), P(out["frames"]),
                              P(out["scores"]), ctypes.byref(out["total"]))
    out["record"], out["capture"], out["total"] = rec, cap, out["total"].value
    return faults, out


def _lists():
    genomes = (np.random.RandomState(3).standard_normal((5, 20)) * 2).astype(np.float32)
    right = np.array([m[0] for m in MATCHES], np.int32)
    left = np.array([m[1] for m in MATCHES], np.int32)
    mult = np.array([m[2] for m in MATCHES], np.float64)
    return genomes, right, left, mult


def _capture_plan(frames):
    """(match, t) pairs: t = 0, 1, a frame in the middle and frames - 1 of every match, plus t = frames (never written)"""
    plan = []
    for m, T in enumerate(frames.tolist()):
        plan += [(m, 0), (m, 1), (m, T // 2), (m, T - 1), (m, T)]
    return plan


def _capture(hs, core, genomes, right, left, mult):
    full = play(hs, core, genomes, right, left, mult)[1]
    plan = _capture_plan(full["frames"])
    idx = np.array([m for m, _ in plan], np.int32)
    t = np.array([t for _, t in plan], np.int32)
    faults, cap = play(hs, core, genomes, right[idx], left[idx], mult[idx], key=idx, capture_at=t, record=False)
    assert faults == 0
    return full, plan, idx, t, cap


@pytest.mark.parametrize("core", [0, 1])
def test_resume_equals_the_uninterrupted_game(hs, core):
    genomes, right, left, mult = _lists()
    full, plan, idx, t, cap = _capture(hs, core, genomes, right, left, mult)
    written = t < full["frames"][idx]
    untouched = np.all(cap["capture"] == 0xAB, axis=1)
    assert np.array_equal(untouched, ~written)                  # a capture at t >= frames is not written
    # resume every written capture with the same genomes, key, seed and generation
    sel = np.nonzero(written)[0].astype(np.int32)
    states = np.ascontiguousarray(cap["capture"][sel])
    faults, res = play(hs, core, genomes, right[idx[sel]], left[idx[sel]], mult[idx[sel]], key=idx[sel], states=states,
                       start=np.arange(len(sel), dtype=np.int32))
    assert faults == 0
    assert res["total"] == int(np.sum(full["frames"][idx[sel]] - t[sel]))      # only the resumed frames are emulated
    for j, i in enumerate(sel):
        m, ti = int(idx[i]), int(t[i])
        assert (res["rewards"][j], res["frames"][j]) == (full["rewards"][m], full["frames"][m]), (m, ti)
        assert np.array_equal(res["scores"][j], full["scores"][m]), (m, ti)
        T = int(full["frames"][m])
        assert res["record"][j, ti:T].tobytes() == full["record"][m, ti:T].tobytes(), (m, ti)
        assert np.all(res["record"][j, :ti]["timeout"] == SENTINEL) and np.all(res["record"][j, T:]["timeout"] == SENTINEL), (m, ti)


def test_captures_do_not_depend_on_the_core(hs):
    genomes, right, left, mult = _lists()
    caps = [_capture(hs, core, genomes, right, left, mult) for core in (0, 1)]
    assert np.array_equal(caps[0][3], caps[1][3])
    assert caps[0][4]["capture"].tobytes() == caps[1][4]["capture"].tobytes()
    # resume core 1's captures on core 0 and the other way round
    full, _, idx, t, _ = caps[0]
    sel = np.nonzero(t < full["frames"][idx])[0].astype(np.int32)
    results = []
    for core, (_, _, _, _, cap) in ((0, caps[1]), (1, caps[0])):
        faults, res = play(hs, core, genomes, right[idx[sel]], left[idx[sel]], mult[idx[sel]], key=idx[sel],
                           states=np.ascontiguousarray(cap["capture"][sel]), start=np.arange(len(sel), dtype=np.int32))
        assert faults == 0
        assert np.array_equal(res["rewards"], full["rewards"][idx[sel]]) and np.array_equal(res["frames"], full["frames"][idx[sel]])
        results.append(res)
    assert results[0]["record"].tobytes() == results[1]["record"].tobytes()


def _oracle_opp(genomes, l):
    return ("mlp", genomes[l]) if l >= 0 else ("score", None) if l == OPP_SCORE_HARDCODED else ("hardcoded", None)


@pytest.mark.parametrize("core", [0, 1])
def test_fresh_start_equals_the_oracle(hs, core):
    """fresh = 1 from the capture at t against the oracle: reset to the match's start state, step it with the recorded action
    vectors for t frames, then a new perform_episode from there with env_id = the match's key."""
    genomes, right, left, mult = _lists()
    full = play(hs, core, genomes, right, left, mult)[1]
    picks = [4, 3, 1, 10]                         # robot, scripted opponent, genome vs genome, robot with a multiplier
    assert left[4] == OPP_ROBOT and left[3] == OPP_SCORE_HARDCODED and left[1] >= 0
    idx = np.array(picks, np.int32)
    t = np.array([max(1, int(full["frames"][m]) // 3) for m in picks], np.int32)
    _, cap = play(hs, core, genomes, right[idx], left[idx], mult[idx], key=idx, capture_at=t, record=False)
    faults, res = play(hs, core, genomes, right[idx], left[idx], mult[idx], key=idx, states=cap["capture"],
                       start=np.arange(len(idx), dtype=np.int32), fresh=1)
    assert faults == 0
    shape = oracle.Shape.make([6, 2, 2])
    for j, m in enumerate(picks):
        env = oracle.Atari()
        env.reset_to_state(oracle.STATE_START_1P if left[m] == OPP_ROBOT else oracle.STATE_START_2P)
        act = full["record"][m]["act"]
        for step in range(int(t[j])):
            a = np.zeros(16, np.uint8)
            a[0] = a[15] = 1                                                      # BLANK_ACTION, config.py:21-23
            if step > 0:
                ra, la = int(act[step - 1]) >> 2, int(act[step - 1]) & 3
                a[4], a[5], a[6], a[7] = ra == oracle.ACT_UP, ra == oracle.ACT_DOWN, la == oracle.ACT_UP, la == oracle.ACT_DOWN
            env.step(a, want_frame=False)
        r, _ = env.episode(shape, _oracle_opp(genomes, int(left[m])), ("mlp", genomes[right[m]]), mult=float(mult[m]), seed=SEED,
                           env_id=m, generation=GENERATION)
        assert (res["rewards"][j], res["frames"][j], res["scores"][j, 0], res["scores"][j, 1]) == (r.reward, r.frames, r.score1,
                                                                                                  r.score2), m


def test_validation_refuses_every_corruption(hs):
    L, _, cart = hs
    genomes, right, left, mult = _lists()
    _, cap = play(hs, 1, genomes, right[:2], left[:2], mult[:2], capture_at=np.array([40, 0], np.int32), record=False)
    for st in cap["capture"]:
        assert L.hs_validate_state(P(st), cart) == 2
        assert np.array_equal(seal(st), st)                          # the documented checksum is the one written
        for i in range(STATE_BYTES):
            for flip in (0x01, 0x80):
                bad = st.copy()
                bad[i] ^= flip
                assert L.hs_validate_state(P(bad), cart) == 0, (i, flip)
        # the same state sealed for another cartridge
        other = st.copy()
        other[8:16] = np.frombuffer(np.uint64(cart ^ 1).tobytes(), np.uint8)
        other = seal(other)
        assert L.hs_validate_state(P(other), cart) == 0 and L.hs_validate_state(P(other), cart ^ 1) == 2
    # a bad state, a players value that disagrees with left[m], a start index out of range, a negative capture frame: the
    # list check refuses and nothing is written
    st = np.ascontiguousarray(cap["capture"][:1])
    bad = st.copy(); bad[0, 100] ^= 4
    zero = np.zeros(1, np.int32)
    robot = np.array([OPP_ROBOT], np.int32)
    for kwargs in ({"states": bad, "start": zero}, {"states": st, "start": zero, "left": robot}, {"states": st, "start": np.ones(1, np.int32)},
                   {"states": st, "start": np.array([-2], np.int32)}, {"states": st, "start": zero, "capture_at": np.array([-1], np.int32)}):
        lft = kwargs.pop("left", left[:1])
        faults, res = play(hs, 1, genomes, right[:1], lft, mult[:1], capture_at=kwargs.pop("capture_at", np.zeros(1, np.int32)),
                           **kwargs)
        assert faults > 0
        assert res["rewards"][0] == -1.0 and res["frames"][0] == -1 and np.all(res["capture"] == 0xAB)
        assert np.all(res["record"]["timeout"] == SENTINEL)
    # the robot game's state is refused for a two-player match, and accepted for a robot match
    _, rc = play(hs, 1, genomes, right[4:5], left[4:5], mult[4:5], capture_at=np.array([10], np.int32), record=False)
    assert L.hs_validate_state(P(rc["capture"][0]), cart) == 1
    assert play(hs, 1, genomes, right[:1], left[:1], mult[:1], states=rc["capture"], start=zero)[0] > 0
    assert play(hs, 1, genomes, right[:1], robot, mult[:1], states=rc["capture"], start=zero)[0] == 0
