"""CPU-side check of the CUDA core's SOURCE: tests/host_sim compiles csrc/*.cuh for the host behind
an intrinsics shim and is compared with the oracle.  This is a debugging aid for the GPU-less build
container; the binding parity evidence is tests/test_gpu_parity.py on a real B200."""
import ctypes

import numpy as np
import pytest

import oracle
from host_sim_lib import library

vp = ctypes.c_void_p


@pytest.fixture(scope="module")
def hs():
    L = library()
    return L, vp(L.hs_create(oracle.load_rom()))


def P(a):
    return a.ctypes.data_as(vp)


@pytest.mark.parametrize("core", [0, 1])
@pytest.mark.parametrize("state,frames,hold", [(None, 120, 3), (0, 500, 4), (1, 700, 7)])
def test_core_matches_oracle_on_random_traces(hs, state, frames, hold, core):
    """core 0 = table-driven interpreter, core 1 = statically translated cartridge."""
    L, sim = hs
    rng = np.random.RandomState(frames)
    env = oracle.Atari()
    if state is None:
        env.power_on(); L.hs_env_power_on(sim)
    else:
        env.reset_to_state(state); L.hs_env_reset(sim, state)
    ram = np.zeros(128, np.uint8); fb = np.zeros((210, 160), np.uint8); loc = np.zeros(6); valid = np.zeros(3, np.uint8)
    regs = np.zeros(8, np.uint8); dig = np.zeros(8, np.uint32)
    act = np.zeros(16, np.uint8)
    for f in range(frames):
        if f % hold == 0:
            act = np.zeros(16, np.uint8); act[0] = act[15] = 1
            r, l = rng.randint(0, 3), rng.randint(0, 3)
            act[4] = r == 1; act[5] = r == 2; act[6] = l == 1; act[7] = l == 2
        ofb = env.step(act)
        assert L.hs_env_step(sim, core, P(act), P(ram), P(fb), P(loc), P(valid), P(regs), P(dig)) == 0
        assert np.array_equal(env.ram, ram), f
        assert np.array_equal(env.cpu_regs[:7], regs[:7]), f
        assert np.array_equal(ofb, fb), f
        assert np.array_equal(env.tia_digest, dig), f
        ol, ov = oracle.find_stuff(oracle.fb_to_rgb(ofb))
        assert np.array_equal(ov, valid) and np.array_equal(ol[ov == 1].ravel(), loc.reshape(3, 2)[valid == 1].ravel()), f


@pytest.mark.parametrize("core", [0, 1])
def test_fused_rollout_matches_oracle_evaluate(hs, core):
    L, sim = hs
    rng = np.random.RandomState(7)
    nodes = np.array([6, 2, 2], np.int32)
    genomes = (rng.random_sample((1, 20)) * 4 - 2).astype(np.float32)
    hof = (rng.random_sample((3, 20)) * 4 - 2).astype(np.float32); hof_fit = np.array([0.7, 0.3, 0.1])
    pick = np.array([[2, 0, 1]], np.int32)
    rew = np.zeros((1, 6)); frm = np.zeros((1, 6), np.int32)
    L.hs_evaluate(sim, core, P(nodes), 3, 1, 0, 6, 0, P(genomes), 1, P(hof), P(hof_fit), 3, P(pick), 5, 0, P(rew), P(frm))
    fit, r, f = oracle.evaluate([6, 2, 2], genomes[0], hof, hof_fit, pick[0], seed=5, genome_id=0)
    assert np.array_equal(r, rew[0]) and np.array_equal(f, frm[0])


@pytest.mark.parametrize("core", [0, 1])
def test_fused_mode_observation_matches_oracle(hs, core):
    """The no-framebuffer flavour (quick span accounting, what rollout_kernel runs): RAM and the
    find_stuff result of every frame against the oracle's frame + restated find_stuff."""
    L, sim = hs
    rng = np.random.RandomState(99 + core)
    for state in (0, 1):
        env = oracle.Atari(); env.reset_to_state(state); L.hs_env_reset(sim, state)
        ram = np.zeros(128, np.uint8); loc = np.zeros(6); valid = np.zeros(3, np.uint8)
        act = np.zeros(16, np.uint8)
        for f in range(900):
            if f % 5 == 0:
                act = np.zeros(16, np.uint8); act[0] = act[15] = 1
                r, l = rng.randint(0, 3), rng.randint(0, 3)
                act[4] = r == 1; act[5] = r == 2; act[6] = l == 1; act[7] = l == 2
            ofb = env.step(act)
            assert L.hs_env_step_fast(sim, core, P(act), P(ram), P(loc), P(valid)) == 0
            assert np.array_equal(env.ram, ram), f
            ol, ov = oracle.find_stuff(oracle.fb_to_rgb(ofb))
            assert np.array_equal(ov, valid) and np.array_equal(ol[ov == 1].ravel(), loc.reshape(3, 2)[valid == 1].ravel()), f


def _build_variant(name, *flags):
    L = library(name, flags)
    return L, vp(L.hs_create(oracle.load_rom()))


def _run_fast_against_oracle(L, sim, frames, seed):
    rng = np.random.RandomState(seed)
    env = oracle.Atari(); env.reset_to_state(1); L.hs_env_reset(sim, 1)
    ram = np.zeros(128, np.uint8); loc = np.zeros(6); valid = np.zeros(3, np.uint8)
    act = np.zeros(16, np.uint8)
    for f in range(frames):
        if f % 4 == 0:
            act = np.zeros(16, np.uint8); act[0] = act[15] = 1
            r, l = rng.randint(0, 3), rng.randint(0, 3)
            act[4] = r == 1; act[5] = r == 2; act[6] = l == 1; act[7] = l == 2
        ofb = env.step(act)
        assert L.hs_env_step_fast(sim, 1, P(act), P(ram), P(loc), P(valid)) == 0
        assert np.array_equal(env.ram, ram), f
        ol, ov = oracle.find_stuff(oracle.fb_to_rgb(ofb))
        assert np.array_equal(ov, valid) and np.array_equal(ol[ov == 1].ravel(), loc.reshape(3, 2)[valid == 1].ravel()), f


def test_superblocks_are_taken():
    """The hand-fused loops (csrc/pong_superblocks.cuh) must actually run: with the event counters compiled in, every frame
    enters the main display loop's block and the score loop's block, and the dispatcher is left with < 100 trips per frame
    (188 without the blocks)."""
    L, sim = _build_variant("stats", "-DA26_STATS")
    st = L.hs_stats().contents
    frames = 200
    for i in range(16):
        st[i] = 0
    _run_fast_against_oracle(L, sim, frames, seed=3)
    assert st[6] >= frames and st[7] >= frames and st[8] >= frames, (st[6], st[7], st[8])
    assert st[5] < 100 * frames, st[5]


def test_generic_translation_without_superblocks():
    """-DA26_NO_SUPERBLOCKS: the instruction-by-instruction translation the guards fall back to stays bit-exact too."""
    L, sim = _build_variant("nosb", "-DA26_NO_SUPERBLOCKS")
    _run_fast_against_oracle(L, sim, 300, seed=4)


def test_hot_latch_mirror_equals_poke_quick_on_random_states(hs):
    """csrc/a26_core.cuh keeps the sixteen hot TIA latches of the display loop in registers (HotLatches): hot_write and
    hot_display_writes must give poke_quick()'s verdict and tia_apply()'s latch bytes for ANY latch state -- the cartridge's own
    traces never delay a player or unlock a missile, so those rules are exercised here on random states."""
    L, _ = hs
    assert L.hs_hot_latch_selftest(1, 200000) == 0


def test_display_loop_event_queue_early_replay():
    """The display-loop block queues the TIA writes that change the picture and replays them when it is left; when fewer than
    eight slots are free it replays in the middle of the loop.  With the normal capacity that path is rare: a build with nine
    slots takes it at every other event, and must still match the oracle frame for frame (RAM and observation)."""
    L, sim = _build_variant("smallqueue", "-DA26_SB_MAX_EVENTS=9")
    _run_fast_against_oracle(L, sim, 400, seed=5)
    # the every-pixel flavour through the same queue: frame buffer, RAM and CPU registers
    rng = np.random.RandomState(6)
    env = oracle.Atari(); env.reset_to_state(0); L.hs_env_reset(sim, 0)
    ram = np.zeros(128, np.uint8); fb = np.zeros((210, 160), np.uint8); loc = np.zeros(6); valid = np.zeros(3, np.uint8)
    regs = np.zeros(8, np.uint8); dig = np.zeros(8, np.uint32)
    for f in range(200):
        if f % 5 == 0:
            act = np.zeros(16, np.uint8); act[0] = act[15] = 1
            r, l = rng.randint(0, 3), rng.randint(0, 3)
            act[4] = r == 1; act[5] = r == 2; act[6] = l == 1; act[7] = l == 2
        ofb = env.step(act)
        assert L.hs_env_step(sim, 1, P(act), P(ram), P(fb), P(loc), P(valid), P(regs), P(dig)) == 0
        assert np.array_equal(env.ram, ram) and np.array_equal(env.cpu_regs[:7], regs[:7]) and np.array_equal(ofb, fb), f
