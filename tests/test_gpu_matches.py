"""ngp_play_matches on the GPU: an explicit match list through the fused rollout.  Both built-in schedules written as lists
must give ngp_evaluate's bits; irregular lists must give the oracle's; results must not depend on the launch geometry; bad
lists are refused before anything is played."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


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


@pytest.mark.parametrize("core", [0, 1])
def test_round_robin_as_a_list_equals_evaluate(ngp, core):
    n, games = 64, 6
    eng = ngp.Engine(ngp.Config(SCHEDULE=ngp.SCHEDULE_ROUND_ROBIN, GAMES_TO_PLAY=games, POPULATION_SIZE=n, CORE=core), device=0)
    g = _dev(_genomes(n, eng.gene_size, 1))
    ev = eng.evaluate(g, seed=5, generation=2, want_detail=True)
    gi, k = np.meshgrid(np.arange(n), np.arange(games), indexing="ij")              # m = g * games + k
    right, left = _dev(gi.reshape(-1), torch.int32), _dev(((gi + k + 1) % n).reshape(-1), torch.int32)
    pm = eng.play_matches(g, right, left, seed=5, generation=2)
    assert torch.equal(pm["rewards"], ev["rewards"].reshape(-1)) and torch.equal(pm["frames"], ev["frames"].reshape(-1))
    assert pm["frames_total"] == ev["frames_total"]
    eng.close()


@pytest.mark.parametrize("core", [0, 1])
def test_reference_schedule_as_a_list_equals_evaluate(ngp, core):
    n, n_hof = 24, 5
    eng = ngp.Engine(ngp.Config(POPULATION_SIZE=n, CORE=core), device=0)
    pop = _genomes(n, eng.gene_size, 2)
    hof = _genomes(n_hof, eng.gene_size, 3)
    hof_fit = np.linspace(0.9, -0.3, n_hof)
    pick = np.random.RandomState(4).randint(0, n_hof, (n, 3)).astype(np.int32)
    table = _dev(np.concatenate([pop, hof]))
    right = _dev(np.repeat(np.arange(n), 6), torch.int32)
    for with_hof in (True, False):
        if with_hof:
            ev = eng.evaluate(_dev(pop), _dev(hof), _dev(hof_fit), _dev(pick), seed=7, generation=1, want_detail=True)
            left = np.concatenate([np.tile([ngp.OPP_HARDCODED, ngp.OPP_ROBOT, ngp.OPP_SCORE_HARDCODED], (n, 1)), n + pick], axis=1)
            mult = np.concatenate([np.ones((n, 3)), hof_fit[pick]], axis=1)
        else:                                               # no hall of fame: games 3-5 are HardcodedAi games (main.py:44-58)
            ev = eng.evaluate(_dev(pop), seed=7, generation=1, want_detail=True)
            left = np.tile([ngp.OPP_HARDCODED, ngp.OPP_ROBOT, ngp.OPP_SCORE_HARDCODED] + [ngp.OPP_HARDCODED] * 3, (n, 1))
            mult = np.ones((n, 6))
        pm = eng.play_matches(table, right, _dev(left.reshape(-1), torch.int32), _dev(mult.reshape(-1)), seed=7, generation=1)
        assert torch.equal(pm["rewards"], ev["rewards"].reshape(-1)), with_hof
        assert torch.equal(pm["frames"], ev["frames"].reshape(-1)), with_hof
    eng.close()


@pytest.mark.parametrize("core", [0, 1])
def test_irregular_list_matches_oracle(ngp, core):
    import oracle
    from test_host_sim_matches import MATCHES, oracle_match
    eng = ngp.Engine(ngp.Config(CORE=core), device=0)
    genomes = _genomes(5, eng.gene_size, 3)
    right, left, mult = (np.array([m[i] for m in MATCHES]) for i in range(3))
    pm = eng.play_matches(_dev(genomes), _dev(right, torch.int32), _dev(left, torch.int32), _dev(mult, torch.float64), seed=21,
                          generation=3)
    rew, frm, sc = (pm[k].cpu().numpy() for k in ("rewards", "frames", "scores"))
    shape = oracle.Shape.make([6, 2, 2])
    for m in range(len(MATCHES)):
        res = oracle_match(shape, genomes, int(right[m]), int(left[m]), float(mult[m]), 21, 3, m)
        assert (rew[m], frm[m], sc[m, 0], sc[m, 1]) == (res.reward, res.frames, res.score1, res.score2), m
    eng.close()


def test_cross_play_is_independent_of_launch_geometry(ngp):
    from neuro_genetic_pong_self_play_b200 import reference_api as ref
    eng = ngp.Engine(ngp.Config(MAX_FRAMES=150), device=0)
    tb = ref.Toolbox(eng.config, engine=eng, seed=6)
    tb.generation = 2
    a, b = eng.init_population(128, seed=8), eng.init_population(128, seed=9)       # 16 384 matches: CTA-synchronous flavour
    base = ref.cross_play(tb, a, b)
    assert base["reward"].shape == (128, 128) and base["score"].shape == (128, 128, 2) and base["frames"].shape == (128, 128)
    for blk in (32, 128, 256):
        eng.set_option("rollout_block", blk)
        try:
            out = ref.cross_play(tb, a, b)
        finally:
            eng.set_option("rollout_block", 0)
        for k in ("reward", "score", "frames"):
            assert torch.equal(out[k], base[k]), (blk, k)
    # entry (i, j) is right row i of a against left row j of b
    one = eng.play_matches(torch.cat([a, b]), _dev([5], torch.int32), _dev([128 + 77], torch.int32), seed=6, generation=2)
    assert one["frames"].item() == base["frames"][5, 77].item() and one["rewards"].item() == base["reward"][5, 77].item()
    eng.close()


def test_accounting_against_the_scripted_opponents(ngp):
    n = 256
    eng = ngp.Engine(ngp.Config(), device=0)
    g = eng.init_population(n, seed=10)
    codes = [ngp.OPP_HARDCODED, ngp.OPP_SCORE_HARDCODED, ngp.OPP_ROBOT]
    right = _dev(np.repeat(np.arange(n), 3), torch.int32)
    left = _dev(np.tile(codes, n), torch.int32)
    pm = eng.play_matches(g, right, left, seed=1)
    frames, scores, rewards = pm["frames"].cpu().numpy(), pm["scores"].cpu().numpy(), pm["rewards"].cpu().numpy()
    assert pm["frames_total"] == int(frames.astype(np.int64).sum())
    assert scores.min() >= 0 and scores.max() <= eng.config.WIN_SCORE
    tie = scores[:, 0] == scores[:, 1]
    assert np.all(rewards[tie] == 0.0)
    # the reward's sign follows the score difference (calculate_reward: (s2 - s1 + s2 * mult) / scaled time, mult = 1)
    assert np.all(np.sign(rewards[~tie]) == np.sign(scores[~tie, 1] - scores[~tie, 0] + scores[~tie, 1]))
    eng.close()


def test_bad_lists_are_refused_and_nothing_is_written(ngp):
    from neuro_genetic_pong_self_play_b200.engine import _p, _stream
    eng = ngp.Engine(ngp.Config(), device=0)
    g = _dev(_genomes(8, eng.gene_size, 5))
    ok = np.array([0, 1, 2, 3], np.int32)
    cases = [(np.array([0, 8, 2, 3]), ok), (np.array([0, -1, 2, 3]), ok), (ok, np.array([0, 1, 8, 3])),
             (ok, np.array([0, -4, 2, 3])), (ok, np.array([ngp.OPP_ROBOT, 2**31 - 1, 2, 3]))]
    for r, l in cases:
        rew = torch.full((4,), -7.0, dtype=torch.float64, device="cuda")
        frm = torch.full((4,), -7, dtype=torch.int32, device="cuda")
        sc = torch.full((4, 2), -7, dtype=torch.int32, device="cuda")
        rt, lt = _dev(r, torch.int32), _dev(l, torch.int32)
        rc = eng._L.ngp_play_matches(eng._h, _p(g), 8, _p(rt), _p(lt), None, 4, 0, 0, _p(rew), _p(frm), _p(sc), None, _stream(eng.device))
        assert rc == -1, (r, l)                                                      # NGP_ERR_INVALID
        torch.cuda.synchronize()
        assert bool((rew == -7.0).all()) and bool((frm == -7).all()) and bool((sc == -7).all())
        with pytest.raises(ngp.NgpError):
            eng.play_matches(g, rt, lt)
    empty = torch.empty(0, dtype=torch.int32, device="cuda")
    with pytest.raises(ngp.NgpError):
        eng.play_matches(g, empty, empty)
    eng.close()
    wide = ngp.Engine(ngp.Config(NETWORK_SHAPE=(6, 48, 2)), device=0)
    gw = _dev(_genomes(2, wide.gene_size, 6))
    rew = torch.zeros(1, dtype=torch.float64, device="cuda")
    rt, lt = _dev([0], torch.int32), _dev([1], torch.int32)
    rc = wide._L.ngp_play_matches(wide._h, _p(gw), 2, _p(rt), _p(lt), None, 1, 0, 0, _p(rew), None, None, None, _stream(wide.device))
    assert rc == -3 and b"wider" in wide._L.ngp_last_error()                          # NGP_ERR_UNSUPPORTED
    wide.close()


def test_play_matches_leaves_evaluate_unchanged(ngp):
    n = 32
    eng = ngp.Engine(ngp.Config(SCHEDULE=ngp.SCHEDULE_ROUND_ROBIN, POPULATION_SIZE=n, MAX_FRAMES=600), device=0)
    g = _dev(_genomes(n, eng.gene_size, 7))
    before = eng.evaluate(g, seed=3, generation=1, want_detail=True)
    eng.play_matches(g, _dev(np.arange(n), torch.int32), _dev(np.full(n, ngp.OPP_ROBOT), torch.int32), seed=9, generation=4)
    after = eng.evaluate(g, seed=3, generation=1, want_detail=True)
    for k in ("fitness", "rewards", "frames"):
        assert torch.equal(before[k], after[k]), k
    assert before["frames_total"] == after["frames_total"]
    eng.close()
