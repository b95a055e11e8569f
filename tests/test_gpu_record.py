"""ngp_record_matches on the GPU: match lists played by the recording twins of the fused rollout.  Results must be
ngp_play_matches' bits; every recorded frame must equal the oracle's trace; the key must reproduce ngp_evaluate's games;
recorded games must re-render through ngp_env_step to pixels whose find_stuff and RAM scores are the recorded ones;
truncation and refusals must leave untouched what they promise to."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

SENTINEL = 0xAB


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


def _same_results(pm, rm):
    for k in ("rewards", "frames", "scores"):
        assert torch.equal(pm[k], rm[k]), k
    assert pm["frames_total"] == rm["frames_total"]


def _fallback_frames(valid: torch.Tensor) -> torch.Tensor:
    """per match: frames on which the ball was found and a paddle was not (get_actions' random fall-back)"""
    v = valid.to(torch.int32)
    return (((v & 1) == 1) & (v != 7)).sum(dim=1)


@pytest.mark.parametrize("core", [0, 1])
def test_irregular_list_same_as_play_matches_and_oracle_trace(ngp, core):
    from test_host_sim_record import FRAME_RECORD, MAX_RECORD, check_against_oracle
    eng = ngp.Engine(ngp.Config(CORE=core), device=0)
    genomes = _genomes(5, eng.gene_size, 3)
    right, left, mult = _matches()
    args = (_dev(genomes), _dev(right, torch.int32), _dev(left, torch.int32), _dev(mult, torch.float64))
    pm = eng.play_matches(*args, seed=21, generation=3)
    rm = eng.record_matches(*args, max_record=MAX_RECORD, seed=21, generation=3)
    _same_results(pm, rm)
    rec = rm["record"]["raw"].cpu().numpy().view(FRAME_RECORD)[..., 0]
    check_against_oracle(rec, *(rm[k].cpu().numpy() for k in ("rewards", "frames", "scores")), genomes, right, left, mult,
                         np.arange(len(right)), 21, 3, sentinel=None)
    eng.close()


@pytest.mark.parametrize("core", [0, 1])
def test_round_robin_list_same_as_play_matches(ngp, core):
    n, games = 64, 6
    eng = ngp.Engine(ngp.Config(SCHEDULE=ngp.SCHEDULE_ROUND_ROBIN, GAMES_TO_PLAY=games, POPULATION_SIZE=n, CORE=core), device=0)
    g = _dev(_genomes(n, eng.gene_size, 1))
    gi, k = np.meshgrid(np.arange(n), np.arange(games), indexing="ij")
    right, left = _dev(gi.reshape(-1), torch.int32), _dev(((gi + k + 1) % n).reshape(-1), torch.int32)
    pm = eng.play_matches(g, right, left, seed=5, generation=2)
    rm = eng.record_matches(g, right, left, seed=5, generation=2)
    _same_results(pm, rm)
    # the record ends where the game does: the last recorded frame holds the final scores
    T = torch.clamp(rm["frames"], max=2048).long() - 1
    last = rm["record"]["score"][torch.arange(n * games, device="cuda"), T].to(torch.int32)
    full = rm["frames"] <= 2048
    assert torch.equal(last[full], rm["scores"][full])
    eng.close()


def test_cross_table_same_as_play_matches_at_every_geometry(ngp):
    eng = ngp.Engine(ngp.Config(MAX_FRAMES=150), device=0)
    a, b = eng.init_population(128, seed=8), eng.init_population(128, seed=9)     # 16 384 matches: CTA-synchronous flavour
    genomes = torch.cat([a, b])
    rows = torch.arange(256, dtype=torch.int32, device="cuda")
    right, left = rows[:128].repeat_interleave(128), rows[128:].repeat(128)
    base = None
    # 0 = automatic; 32 one-warp CTAs; 128 / 256 the full-register CTA-synchronous flavour; 384 and 512 (43 and 32 CTAs) the
    # register-capped CTA-synchronous flavours <1,true,384> and <1,true,512> and their recording twins
    for blk in (0, 32, 128, 256, 384, 512):
        eng.set_option("rollout_block", blk)
        try:
            pm = eng.play_matches(genomes, right, left, seed=6, generation=2)
            rm = eng.record_matches(genomes, right, left, max_record=150, seed=6, generation=2)
        finally:
            eng.set_option("rollout_block", 0)
        _same_results(pm, rm)
        assert int(rm["frames"].max().item()) <= 150
        if base is None:
            base = rm
        else:
            _same_results(base, rm)
            assert torch.equal(rm["record"]["raw"], base["record"]["raw"]), blk
    eng.close()


@pytest.mark.parametrize("blind_left", [False, True])
def test_key_reproduces_evaluate(ngp, blind_left):
    """A shuffled round-robin list with key = the original environment index gives evaluate's games, and replay_selfplay
    plays them again.  blind_left: a left-paddle colour that matches nothing, so that every frame with the ball in view takes
    get_actions' random fall-back and the key decides the game (self-play between visible paddles rarely if ever does)."""
    from neuro_genetic_pong_self_play_b200 import reference_api as ref
    n, games = 256, 6
    colour = {"LEFT_GUY_COLOUR": (1, 2, 3)} if blind_left else {}
    eng = ngp.Engine(ngp.Config(SCHEDULE=ngp.SCHEDULE_ROUND_ROBIN, GAMES_TO_PLAY=games, POPULATION_SIZE=n, **colour), device=0)
    g = eng.init_population(n, seed=12)
    ev = eng.evaluate(g, seed=4, generation=7, want_detail=True)
    gi, k = np.meshgrid(np.arange(n), np.arange(games), indexing="ij")
    perm = np.random.RandomState(0).permutation(n * games)
    right = _dev(gi.reshape(-1)[perm], torch.int32)
    left = _dev(((gi + k + 1) % n).reshape(-1)[perm], torch.int32)
    rm = eng.record_matches(g, right, left, key=_dev(perm, torch.int32), seed=4, generation=7)
    inv = torch.as_tensor(np.argsort(perm), device="cuda")
    assert torch.equal(rm["rewards"][inv], ev["rewards"].reshape(-1))
    assert torch.equal(rm["frames"][inv], ev["frames"].reshape(-1))
    fb = _fallback_frames(rm["record"]["valid"])[inv].cpu().numpy()
    if blind_left:
        assert fb.min() > 0, "every game must take the random fall-back"
        # without the key (environment index = list position) the same list plays other games
        other = eng.record_matches(g, right, left, seed=4, generation=7)
        assert not torch.equal(other["frames"], rm["frames"])
    tb = ref.Toolbox(eng.config, engine=eng, seed=4)
    tb.generation = 7
    for e in (0, 7, int(np.argmax(fb))):
        gg, kk = divmod(e, games)
        out = ref.replay_selfplay(tb, g, gg, kk, upsample=(1, 1))
        assert out["reward"] == ev["rewards"][gg, kk].item() and out["steps"] == ev["frames"][gg, kk].item(), (gg, kk)
        assert out["frames"].shape == (out["steps"], 210, 160, 3)
    eng.close()


def test_render_round_trip(ngp):
    from neuro_genetic_pong_self_play_b200 import reference_api as ref
    eng = ngp.Engine(ngp.Config(), device=0)
    tb = ref.Toolbox(eng.config, engine=eng, seed=2)
    g = eng.init_population(4, seed=13)
    right = _dev([0, 1, 2, 3], torch.int32)
    left = _dev([3, ngp.OPP_HARDCODED, ngp.OPP_SCORE_HARDCODED, ngp.OPP_ROBOT], torch.int32)
    rm = eng.record_matches(g, right, left, max_record=12000, seed=2)
    rec = rm["record"]
    assert int(rm["frames"].max().item()) <= 12000
    r_int = ref.render_recorded(tb, rm, range(4), core=ngp.CORE_INTERPRETER, want_ram=True)
    r_tr = ref.render_recorded(tb, rm, range(4), core=ngp.CORE_TRANSLATED, want_ram=True)
    for m in range(4):
        T = int(rm["frames"][m].item())
        (pix, ram), (pix_t, ram_t) = r_int[m], r_tr[m]
        assert pix.shape == (T, 210, 160, 3)
        assert torch.equal(pix, pix_t) and torch.equal(ram, ram_t), m
        loc, valid = eng.find_stuff(pix)
        bits = valid[:, 0] | valid[:, 1] << 1 | valid[:, 2] << 2
        assert torch.equal(bits, rec["valid"][m, :T]), m
        assert torch.equal(loc, rec["loc"][m, :T]), m
        assert torch.equal(ram[:, 13:15], rec["score"][m, :T]), m
    eng.close()


def test_truncation_and_untouched_entries(ngp):
    from neuro_genetic_pong_self_play_b200.engine import _p, _stream, record_views
    eng = ngp.Engine(ngp.Config(CORE=1), device=0)
    genomes = _dev(_genomes(5, eng.gene_size, 3))
    right, left, mult = _matches()
    r, l, mu = _dev(right, torch.int32), _dev(left, torch.int32), _dev(mult, torch.float64)
    full = eng.record_matches(genomes, r, l, mu, max_record=12000, seed=21, generation=3)
    M = len(right)
    for T in (40, 12000):
        raw = torch.full((M, T, 32), SENTINEL, dtype=torch.uint8, device="cuda")
        rew = torch.empty(M, dtype=torch.float64, device="cuda")
        frm = torch.empty(M, dtype=torch.int32, device="cuda")
        rc = eng._L.ngp_record_matches(eng._h, _p(genomes), 5, _p(r), _p(l), _p(mu), None, M, 21, 3, T, _p(raw), _p(rew), _p(frm),
                                       None, None, _stream(eng.device))
        assert rc == 0
        assert torch.equal(frm, full["frames"]) and torch.equal(rew, full["rewards"])         # full lengths whatever T is
        for m in range(M):
            n = min(int(frm[m].item()), T)
            assert torch.equal(raw[m, :n], full["record"]["raw"][m, :n]), (T, m)
            assert bool((raw[m, n:] == SENTINEL).all()), (T, m)
        if T == 40:
            assert record_views(raw)["timeout"].shape == (M, 40)
    eng.close()


def test_refusals_write_nothing(ngp):
    from neuro_genetic_pong_self_play_b200.engine import _p, _stream
    eng = ngp.Engine(ngp.Config(), device=0)
    g = _dev(_genomes(8, eng.gene_size, 5))
    ok = np.array([0, 1, 2, 3], np.int32)
    cases = [(np.array([0, 8, 2, 3]), ok, None, 16, True), (ok, np.array([0, 1, 8, 3]), None, 16, True),
             (ok, np.array([0, -4, 2, 3]), None, 16, True), (ok, ok, np.array([0, 1, -1, 3]), 16, True),
             (ok, ok, None, 0, True), (ok, ok, None, 16, False)]
    for r, l, key, T, with_record in cases:
        rew = torch.full((4,), -7.0, dtype=torch.float64, device="cuda")
        frm = torch.full((4,), -7, dtype=torch.int32, device="cuda")
        sc = torch.full((4, 2), -7, dtype=torch.int32, device="cuda")
        raw = torch.full((4, 16, 32), SENTINEL, dtype=torch.uint8, device="cuda")
        rt, lt = _dev(r, torch.int32), _dev(l, torch.int32)
        kt = None if key is None else _dev(key, torch.int32)
        rc = eng._L.ngp_record_matches(eng._h, _p(g), 8, _p(rt), _p(lt), None, _p(kt), 4, 0, 0, T, _p(raw) if with_record else None,
                                       _p(rew), _p(frm), _p(sc), None, _stream(eng.device))
        assert rc == -1, (r, l, key, T, with_record)                                            # NGP_ERR_INVALID
        torch.cuda.synchronize()
        assert bool((rew == -7.0).all()) and bool((frm == -7).all()) and bool((sc == -7).all())
        assert bool((raw == SENTINEL).all())
    with pytest.raises(ngp.NgpError):
        eng.record_matches(g, _dev(ok, torch.int32), _dev(ok, torch.int32), key=_dev([0, 1, -1, 3], torch.int32))
    eng.close()
    wide = ngp.Engine(ngp.Config(NETWORK_SHAPE=(6, 48, 2)), device=0)
    gw = _dev(_genomes(2, wide.gene_size, 6))
    rew = torch.zeros(1, dtype=torch.float64, device="cuda")
    raw = torch.zeros((1, 4, 32), dtype=torch.uint8, device="cuda")
    rt, lt = _dev([0], torch.int32), _dev([1], torch.int32)
    rc = wide._L.ngp_record_matches(wide._h, _p(gw), 2, _p(rt), _p(lt), None, None, 1, 0, 0, 4, _p(raw), _p(rew), None, None, None,
                                    _stream(wide.device))
    assert rc == -3 and b"wider" in wide._L.ngp_last_error()                                    # NGP_ERR_UNSUPPORTED
    wide.close()


def test_record_leaves_evaluate_and_play_matches_unchanged(ngp):
    n = 32
    eng = ngp.Engine(ngp.Config(SCHEDULE=ngp.SCHEDULE_ROUND_ROBIN, POPULATION_SIZE=n, MAX_FRAMES=600), device=0)
    g = _dev(_genomes(n, eng.gene_size, 7))
    right, left = _dev(np.arange(n), torch.int32), _dev((np.arange(n) + 3) % n, torch.int32)
    ev0 = eng.evaluate(g, seed=3, generation=1, want_detail=True)
    pm0 = eng.play_matches(g, right, left, seed=3, generation=1)
    eng.record_matches(g, right.flip(0).contiguous(), _dev(np.full(n, ngp.OPP_ROBOT), torch.int32), key=right, seed=9, generation=4)
    ev1 = eng.evaluate(g, seed=3, generation=1, want_detail=True)
    pm1 = eng.play_matches(g, right, left, seed=3, generation=1)
    for k in ("fitness", "rewards", "frames"):
        assert torch.equal(ev0[k], ev1[k]), k
    assert ev0["frames_total"] == ev1["frames_total"]
    _same_results(pm0, pm1)
    eng.close()
