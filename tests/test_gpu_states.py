"""Save states on the GPU: ngp_play_matches_states (match lists that start from states and capture their own, run by the
recording twins of the fused rollout) and ngp_env_get_state / ngp_env_set_state.  Without the new arguments the results are
ngp_play_matches' and ngp_record_matches' bits; a resumed capture replays the rest of the uninterrupted game at every launch
geometry; stepwise and fused states agree byte for byte; refusals write nothing; other entry points are unaffected."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

STATE = 512
EPISODE = slice(384, 432)             # DESIGN.md section 4: the episode words
HAS_EPISODE = 20                      # header word 5
CHECKSUM = slice(504, 512)


@pytest.fixture(scope="module")
def ngp():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import neuro_genetic_pong_self_play_b200 as m
    return m


def _dev(a, dtype=None):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype).cuda()


def _genomes(n, G, seed):
    return (np.random.RandomState(seed).standard_normal((n, G)) * 2).astype(np.float32)


def _matches():
    from test_host_sim_matches import MATCHES
    return (np.array([m[i] for m in MATCHES]) for i in range(3))


def _same(a, b, keys=("rewards", "frames", "scores")):
    for k in keys:
        assert torch.equal(a[k], b[k]), k


def _console(states: torch.Tensor) -> torch.Tensor:
    """the bytes of states that do not belong to the episode (header without has_episode, console, padding)"""
    keep = torch.ones(STATE, dtype=torch.bool, device=states.device)
    keep[EPISODE] = False
    keep[HAS_EPISODE] = False
    keep[CHECKSUM] = False
    return states[:, keep]


@pytest.mark.parametrize("core", [0, 1])
def test_without_new_arguments_the_bits_of_play_and_record_matches(ngp, core):
    eng = ngp.Engine(ngp.Config(CORE=core), device=0)
    right, left, mult = _matches()
    args = (_dev(_genomes(5, eng.gene_size, 3)), _dev(right, torch.int32), _dev(left, torch.int32), _dev(mult, torch.float64))
    pm = eng.play_matches(*args, seed=21, generation=3)
    ps = eng.play_matches_states(*args, seed=21, generation=3)
    _same(pm, ps)
    assert pm["frames_total"] == ps["frames_total"] and "capture" not in ps and "record" not in ps
    key = _dev(np.arange(len(right))[::-1], torch.int32)
    rm = eng.record_matches(*args, key=key, max_record=12000, seed=21, generation=3)
    rs = eng.play_matches_states(*args, key=key, max_record=12000, seed=21, generation=3)
    _same(rm, rs)
    assert rm["frames_total"] == rs["frames_total"]
    for m in range(len(right)):
        T = int(rm["frames"][m].item())
        assert torch.equal(rm["record"]["raw"][m, :T], rs["record"]["raw"][m, :T]), m
    eng.close()


def test_resume_equals_the_uninterrupted_game_at_every_geometry(ngp):
    eng = ngp.Engine(ngp.Config(MAX_FRAMES=150), device=0)
    a, b = eng.init_population(128, seed=8), eng.init_population(128, seed=9)     # 16 384 matches: CTA-synchronous flavour
    genomes = torch.cat([a, b])
    rows = torch.arange(256, dtype=torch.int32, device="cuda")
    right, left = rows[:128].repeat_interleave(128), rows[128:].repeat(128)
    M = right.shape[0]
    t = (torch.arange(M, device="cuda", dtype=torch.int32) * 37) % 160              # some past the end: never captured
    base = None
    for blk in (0, 32, 128, 256, 384, 512):
        eng.set_option("rollout_block", blk)
        try:
            full = eng.play_matches_states(genomes, right, left, capture_at=t, max_record=150, seed=6, generation=2)
            cap = full["capture"]
            written = t < full["frames"]
            assert bool((cap[~written] == 0).all())                                 # left untouched (zeros)
            # only written captures are passed: every state given is validated, whether a match starts from it or not
            idx = torch.nonzero(written).flatten()
            start = torch.full((M,), -1, dtype=torch.int32, device="cuda")
            start[idx] = torch.arange(idx.shape[0], dtype=torch.int32, device="cuda")
            res = eng.play_matches_states(genomes, right, left, states=cap[idx].contiguous(), start=start, max_record=150, seed=6,
                                          generation=2)
        finally:
            eng.set_option("rollout_block", 0)
        _same(full, res)
        assert res["frames_total"] == full["frames_total"] - int(t[written].sum().item())
        steps = torch.arange(150, device="cuda")[None, :]
        after = (steps >= torch.where(written, t, 0)[:, None]) & (steps < full["frames"][:, None])
        assert torch.equal(res["record"]["raw"][after], full["record"]["raw"][after]), blk
        if base is None:
            base = full
        else:
            _same(base, full)
            assert torch.equal(base["capture"], cap), blk
    eng.close()


def _replay_actions(ngp, act_prev: torch.Tensor) -> torch.Tensor:
    """BLANK_ACTION with the decisions of the previous frame (left | right << 2, per env) written to [4:8]"""
    a = torch.zeros((act_prev.shape[0], 16), dtype=torch.uint8, device="cuda")
    a[:, 0] = 1; a[:, 15] = 1
    ra, la = act_prev.long() >> 2, act_prev.long() & 3
    a[:, 4], a[:, 5] = (ra == ngp.ACT_UP).to(torch.uint8), (ra == ngp.ACT_DOWN).to(torch.uint8)
    a[:, 6], a[:, 7] = (la == ngp.ACT_UP).to(torch.uint8), (la == ngp.ACT_DOWN).to(torch.uint8)
    return a


def test_stepwise_states_agree_with_fused_captures(ngp):
    eng = ngp.Engine(ngp.Config(CORE=1), device=0)
    genomes = _dev(_genomes(5, eng.gene_size, 3))
    # env_reset('Start.2P') = a t = 0 capture of a two-player match, up to the episode part
    eng.env_reset(1, ngp.STATE_START_2P)
    s0 = eng.env_get_state()
    c0 = eng.play_matches_states(genomes, _dev([1], torch.int32), _dev([2], torch.int32), capture_at=_dev([0], torch.int32))
    assert torch.equal(_console(s0), _console(c0["capture"]))
    assert int(s0[0, HAS_EPISODE]) == 0 and int(c0["capture"][0, HAS_EPISODE]) == 1
    assert bool((s0[0, EPISODE] == 0).all())
    for players, r, l in ((2, [0, 1, 3, 1], [0, 2, -2, 4]), (1, [0, 2], [-3, -3])):
        r, l = _dev(r, torch.int32), _dev(l, torch.int32)
        n = r.shape[0]
        full = eng.play_matches_states(genomes, r, l, max_record=12000, seed=21, generation=3)
        t = torch.clamp(full["frames"] // 3, min=1)
        k = 25
        assert bool((t + k < full["frames"]).all())
        c_t = eng.play_matches_states(genomes, r, l, capture_at=t, seed=21, generation=3)["capture"]
        c_tk = eng.play_matches_states(genomes, r, l, capture_at=t + k, seed=21, generation=3)["capture"]
        rows = torch.arange(n, device="cuda")
        for frames in (False, True):
            eng.env_set_state(c_t)
            got = eng.env_get_state()
            assert torch.equal(_console(got), _console(c_t)) and bool((got[:, EPISODE] == 0).all())
            for j in range(k):
                step = t + j                                                  # env.step index of the whole episode
                a = _replay_actions(ngp, full["record"]["act"][rows, step - 1])
                out = eng.env_step(a, want_frames=frames, want_obs=False, core=ngp.CORE_TRANSLATED)
                rec = {f: full["record"][f][rows, step] for f in ("loc", "valid", "score")}
                assert torch.equal(out["ram"][:, 13:15], rec["score"]), (players, frames, j)
                if frames:
                    loc, valid = eng.find_stuff(out["frames"])
                    assert torch.equal(valid[:, 0] | valid[:, 1] << 1 | valid[:, 2] << 2, rec["valid"]), (players, j)
                    assert torch.equal(loc, rec["loc"]), (players, j)
            assert torch.equal(_console(eng.env_get_state()), _console(c_tk)), (players, frames)
    eng.close()


def test_key_reproduces_evaluate_from_a_capture(ngp):
    n, games = 64, 6
    eng = ngp.Engine(ngp.Config(SCHEDULE=ngp.SCHEDULE_ROUND_ROBIN, GAMES_TO_PLAY=games, POPULATION_SIZE=n), device=0)
    g = eng.init_population(n, seed=12)
    ev = eng.evaluate(g, seed=4, generation=7, want_detail=True)
    gi, k = np.meshgrid(np.arange(n), np.arange(games), indexing="ij")
    right, left = _dev(gi.reshape(-1), torch.int32), _dev(((gi + k + 1) % n).reshape(-1), torch.int32)
    key = torch.arange(n * games, dtype=torch.int32, device="cuda")
    t = (ev["frames"].reshape(-1) // 2).to(torch.int32).contiguous()
    cap = eng.play_matches_states(g, right, left, key=key, capture_at=t, seed=4, generation=7)["capture"]
    res = eng.play_matches_states(g, right, left, key=key, states=cap, start=key, seed=4, generation=7)
    assert torch.equal(res["rewards"], ev["rewards"].reshape(-1))
    assert torch.equal(res["frames"], ev["frames"].reshape(-1))
    eng.close()


def test_branch_and_render_from_the_start_state(ngp):
    from neuro_genetic_pong_self_play_b200 import reference_api as ref
    eng = ngp.Engine(ngp.Config(), device=0)
    tb = ref.Toolbox(eng.config, engine=eng, seed=2)
    g = eng.init_population(4, seed=13)
    right, left = [0, 1, 2], [3, ngp.OPP_HARDCODED, ngp.OPP_ROBOT]
    rm = eng.record_matches(g, _dev(right, torch.int32), _dev(left, torch.int32), max_record=12000, seed=2)
    for m in range(3):
        T = int(rm["frames"][m].item())
        t = T // 2
        same = ref.branch(tb, g, right, left, m, t, max_record=12000)              # the same players: the original game
        assert same["rewards"].item() == rm["rewards"][m].item() and int(same["frames"].item()) == T
        assert torch.equal(same["record"]["raw"][0, :T], rm["record"]["raw"][m, :T])
        other = ref.branch(tb, g, right, left, m, t, new_right=3, new_left=None if left[m] < 0 else 1, max_record=12000)
        T2 = int(other["frames"].item())
        assert T2 > t
        pix, ram = ref.render_recorded(tb, other, [0], want_ram=True, start_states=other["start_states"])[0]
        assert pix.shape == (T2 - t, 210, 160, 3)
        loc, valid = eng.find_stuff(pix)
        rec = other["record"]
        assert torch.equal(valid[:, 0] | valid[:, 1] << 1 | valid[:, 2] << 2, rec["valid"][0, t:T2]), m
        assert torch.equal(loc, rec["loc"][0, t:T2]) and torch.equal(ram[:, 13:15], rec["score"][0, t:T2]), m
        # the rendering of the whole game from the built-in start agrees with the one from the state
        whole = ref.render_recorded(tb, other, [0])[0]
        assert torch.equal(whole[t:], pix), m
    eng.close()


def test_refusals_write_nothing(ngp):
    from neuro_genetic_pong_self_play_b200.engine import _p, _stream
    eng = ngp.Engine(ngp.Config(), device=0)
    g = _dev(_genomes(8, eng.gene_size, 5))
    ok = _dev([0, 1, 2, 3], torch.int32)
    good = eng.play_matches_states(g, ok, ok, capture_at=_dev([5, 6, 7, 8], torch.int32))["capture"]
    robot = eng.play_matches_states(g, ok[:1], _dev([ngp.OPP_ROBOT], torch.int32), capture_at=_dev([5], torch.int32))["capture"]
    flipped = good.clone(); flipped[2, 77] ^= 1
    z = _dev([0, 1, 2, 3], torch.int32)
    cases = [  # (right, left, states, start, capture_at, with_capture)
        (_dev([0, 8, 2, 3], torch.int32), ok, good, z, None, False),           # a record_matches refusal
        (ok, ok, good, _dev([0, 1, 4, 3], torch.int32), None, False),          # start past n_states
        (ok, ok, good, _dev([0, -2, 2, 3], torch.int32), None, False),
        (ok, ok, flipped, z, None, False),                                     # a state that fails validation
        (ok, ok, flipped, None, None, False),                                  # ... even when no match starts from it
        (ok, ok, torch.cat([good[:3], robot]), z, None, False),                # players 1 for a two-player match
        (ok, _dev([0, 1, 2, ngp.OPP_ROBOT], torch.int32), good, z, None, False),   # players 2 for a robot match
        (ok, ok, good, z, _dev([0, 1, -1, 3], torch.int32), True),             # a negative capture frame
        (ok, ok, good, z, _dev([0, 1, 2, 3], torch.int32), False),             # capture_at without capture
    ]
    for i, (r, l, states, start, cap_at, with_capture) in enumerate(cases):
        rew = torch.full((4,), -7.0, dtype=torch.float64, device="cuda")
        frm = torch.full((4,), -7, dtype=torch.int32, device="cuda")
        sc = torch.full((4, 2), -7, dtype=torch.int32, device="cuda")
        raw = torch.full((4, 16, 32), 0xAB, dtype=torch.uint8, device="cuda")
        cap = torch.full((4, STATE), 0xAB, dtype=torch.uint8, device="cuda")
        rc = eng._L.ngp_play_matches_states(eng._h, _p(g), 8, _p(r), _p(l), None, None, 4, _p(states), states.shape[0], _p(start), 0,
                                            _p(cap_at), _p(cap) if with_capture else None, 16, _p(raw), 0, 0, _p(rew), _p(frm), _p(sc),
                                            None, _stream(eng.device))
        assert rc == -1, i                                                                        # NGP_ERR_INVALID
        torch.cuda.synchronize()
        assert bool((rew == -7.0).all()) and bool((frm == -7).all()) and bool((sc == -7).all()), i
        assert bool((raw == 0xAB).all()) and bool((cap == 0xAB).all()), i
    with pytest.raises(ngp.NgpError):
        eng.play_matches_states(g, ok, ok, states=flipped, start=z)
    # a refused env_set_state leaves the stepwise environments as they were
    eng.env_set_state(good)
    before = eng.env_get_state()
    for bad in (flipped, torch.cat([good[:3], robot])):
        with pytest.raises(ngp.NgpError):
            eng.env_set_state(bad)
        assert torch.equal(eng.env_get_state(), before)
    from test_host_sim_states import seal
    foreign = good[:1].cpu().numpy()[0].copy()
    foreign[8] ^= 1                                                                             # another cartridge's hash
    with pytest.raises(ngp.NgpError):
        eng.env_set_state(_dev(seal(foreign)[None]))
    assert torch.equal(eng.env_get_state(), before)
    eng.close()
    wide = ngp.Engine(ngp.Config(NETWORK_SHAPE=(6, 48, 2)), device=0)
    gw = _dev(_genomes(2, wide.gene_size, 6))
    rew = torch.zeros(1, dtype=torch.float64, device="cuda")
    rt, lt = _dev([0], torch.int32), _dev([1], torch.int32)
    rc = wide._L.ngp_play_matches_states(wide._h, _p(gw), 2, _p(rt), _p(lt), None, None, 1, None, 0, None, 0, None, None, 0, None, 0, 0,
                                         _p(rew), None, None, None, _stream(wide.device))
    assert rc == -3 and b"wider" in wide._L.ngp_last_error()                                    # NGP_ERR_UNSUPPORTED
    wide.close()


def test_states_leave_evaluate_play_and_record_matches_unchanged(ngp):
    n = 32
    eng = ngp.Engine(ngp.Config(SCHEDULE=ngp.SCHEDULE_ROUND_ROBIN, POPULATION_SIZE=n, MAX_FRAMES=600), device=0)
    g = _dev(_genomes(n, eng.gene_size, 7))
    right, left = _dev(np.arange(n), torch.int32), _dev((np.arange(n) + 3) % n, torch.int32)

    def run():
        return (eng.evaluate(g, seed=3, generation=1, want_detail=True), eng.play_matches(g, right, left, seed=3, generation=1),
                eng.record_matches(g, right, left, max_record=600, seed=3, generation=1))

    before = run()
    cap = eng.play_matches_states(g, right, left, capture_at=_dev(np.arange(n) * 5, torch.int32), seed=9, generation=4)["capture"]
    written = torch.nonzero(cap.any(dim=1)).flatten().to(torch.int32)
    eng.play_matches_states(g, right[written].contiguous(), left[written].contiguous(), states=cap[written.long()].contiguous(),
                            start=torch.arange(written.shape[0], dtype=torch.int32, device="cuda"), fresh=True, max_record=50,
                            seed=9, generation=4)
    after = run()
    for k in ("fitness", "rewards", "frames"):
        assert torch.equal(before[0][k], after[0][k]), k
    assert before[0]["frames_total"] == after[0]["frames_total"]
    _same(before[1], after[1]); _same(before[2], after[2])
    for m in range(n):
        T = int(before[2]["frames"][m].item())
        assert torch.equal(before[2]["record"]["raw"][m, :T], after[2]["record"]["raw"][m, :T]), m
    eng.close()
