"""ngp_play_matches_stepwise on the GPU: match lists, records and save states on the per-frame driver, for networks of any
width.  Networks the fused rollout takes must give the fused entry points' bits (the decide kernel runs the same FP64
policies), wide networks must give the FP64 oracle's games (the MLP rows gathered into per-genome chunks), and every
refusal of the fused calls must be the same here."""
import concurrent.futures as cf
import ctypes
import os

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


def _wide_genomes(rng, n, nodes, bias=True):
    """test_gpu_wide_evaluate's scaling: weights scaled by 1/sqrt(fan-in) per layer, so that decisions depend on the inputs"""
    b = 1 if bias else 0
    G = sum((a + b) * c for a, c in zip(nodes[:-1], nodes[1:]))
    g = np.zeros((n, G), np.float32)
    off = 0
    for a, c in zip(nodes[:-1], nodes[1:]):
        cnt = (a + b) * c
        g[:, off:off + cnt] = (rng.standard_normal((n, cnt)) * 3.0 / np.sqrt(a + 1)).astype(np.float32)
        off += cnt
    return g


def _matches():
    from test_host_sim_matches import MATCHES
    return (np.array([m[i] for m in MATCHES]) for i in range(3))


def _skewed(n_genomes):
    """genome 0 on the right against rows 1..36 (36 rows: three chunks of 16), rows 37.. once each against the scripted players"""
    right = np.concatenate([np.zeros(36, np.int64), np.arange(37, n_genomes)])
    codes = np.array([-1, -2, -3])
    left = np.concatenate([np.arange(1, 37), codes[np.arange(n_genomes - 37) % 3]])
    return right, left, np.ones(len(right))


def _call(eng, driver, genomes, right, left, mult=None, key=None, states=None, start=None, fresh=False, capture_at=None,
          capture=None, max_record=0, record=None, seed=0, generation=0):
    """One raw ngp_play_matches_states / ngp_play_matches_stepwise call with sentinel-filled outputs; returns (rc, outputs)."""
    from neuro_genetic_pong_self_play_b200.engine import _p, _stream
    fn = eng._L.ngp_play_matches_stepwise if driver == "stepwise" else eng._L.ngp_play_matches_states
    M = right.shape[0]
    out = {"rewards": torch.full((M,), -7.0, dtype=torch.float64, device="cuda"),
           "frames": torch.full((M,), -7, dtype=torch.int32, device="cuda"),
           "scores": torch.full((M, 2), -7, dtype=torch.int32, device="cuda")}
    total = ctypes.c_uint64(0)
    rec_p = record if isinstance(record, ctypes.c_void_p) else _p(record)
    rc = fn(eng._h, _p(genomes), genomes.shape[0], _p(right), _p(left), _p(mult), _p(key), M, _p(states),
            0 if states is None else states.shape[0], _p(start), 1 if fresh else 0, _p(capture_at), _p(capture), int(max_record), rec_p,
            seed, generation, _p(out["rewards"]), _p(out["frames"]), _p(out["scores"]), ctypes.byref(total), _stream(eng.device))
    torch.cuda.synchronize()
    out["frames_total"] = int(total.value)
    return rc, out


def _same(a, b, keys=("rewards", "frames", "scores", "frames_total"), what=""):
    for k in keys:
        if k == "frames_total":
            assert a[k] == b[k], (what, k, a[k], b[k])
        else:
            assert torch.equal(a[k], b[k]), (what, k)


def _both(eng, *args, **kw):
    rf, f = _call(eng, "fused", *args, **kw)
    rs, s = _call(eng, "stepwise", *args, **kw)
    assert rf == 0 and rs == 0, (rf, rs, eng._L.ngp_last_error())
    return f, s


def _narrow_lists(ngp, eng):
    """(name, genomes, right, left, mult): round robin 64 x 6, the reference schedule with hall-of-fame rows, bots and the
    robot, test_host_sim_matches' MATCHES and a 4 096-match cross table"""
    G = eng.gene_size
    n, games = 64, 6
    gi, k = np.meshgrid(np.arange(n), np.arange(games), indexing="ij")
    rr = ("round robin", _dev(_genomes(n, G, 1)), gi.reshape(-1), ((gi + k + 1) % n).reshape(-1), None)
    n, n_hof = 24, 5
    pick = np.random.RandomState(4).randint(0, n_hof, (n, 3))
    left = np.concatenate([np.tile([ngp.OPP_HARDCODED, ngp.OPP_ROBOT, ngp.OPP_SCORE_HARDCODED], (n, 1)), n + pick], axis=1)
    hof_fit = np.linspace(0.9, -0.3, n_hof)
    mult = np.concatenate([np.ones((n, 3)), hof_fit[pick]], axis=1)
    ref = ("reference", _dev(np.concatenate([_genomes(n, G, 2), _genomes(n_hof, G, 3)])), np.repeat(np.arange(n), 6),
           left.reshape(-1), mult.reshape(-1))
    right, left, mult = _matches()
    irr = ("irregular", _dev(_genomes(5, G, 3)), right, left, mult)
    a = np.arange(64)
    cross = ("cross", _dev(_genomes(128, G, 8)), np.repeat(a, 64), 64 + np.tile(a, 64), None)
    return [rr, ref, irr, cross]


def _lists_dev(right, left, mult):
    return _dev(right, torch.int32), _dev(left, torch.int32), None if mult is None else _dev(mult, torch.float64)


# ---- 1. narrow networks: both drivers, same arguments, same bits ---------------------------------------------------------
@pytest.mark.parametrize("core", [0, 1])
def test_narrow_lists_same_bits_on_both_drivers(ngp, core):
    # the interpreter core is much slower per frame on the per-frame driver: its games stop at 600 frames
    eng = ngp.Engine(ngp.Config(CORE=core, MAX_FRAMES=0 if core else 600), device=0)
    for name, genomes, right, left, mult in _narrow_lists(ngp, eng):
        r, l, mu = _lists_dev(right, left, mult)
        f, s = _both(eng, genomes, r, l, mu, seed=21, generation=3)
        _same(f, s, what=name)
        if name == "cross":
            continue
        M = r.shape[0]
        # records: max_record shorter than some games, with and without a key, sentinel-filled buffers
        T = 300
        for key in (None, _dev(np.arange(M)[::-1] * 3, torch.int32)):
            recs = [torch.full((M, T, 32), SENTINEL, dtype=torch.uint8, device="cuda") for _ in range(2)]
            rf, fo = _call(eng, "fused", genomes, r, l, mu, key=key, max_record=T, record=recs[0], seed=21, generation=3)
            rs, so = _call(eng, "stepwise", genomes, r, l, mu, key=key, max_record=T, record=recs[1], seed=21, generation=3)
            assert rf == 0 and rs == 0
            _same(fo, so, what=(name, key is None))
            assert torch.equal(recs[0], recs[1]), (name, key is None)
            n_written = torch.clamp(so["frames"], max=T)
            past = torch.arange(T, device="cuda")[None, :] >= n_written[:, None]
            assert bool((recs[1][past] == SENTINEL).all()) and bool((so["frames"] > T).any())
        # states: captures at 0, mid-game and after the end; resumed and fresh starts
        t = torch.tensor([0, 1, 50, 333, 100000], device="cuda", dtype=torch.int32)[torch.arange(M, device="cuda") % 5].contiguous()
        caps = [torch.zeros((M, 512), dtype=torch.uint8, device="cuda") for _ in range(2)]
        _, fo = _call(eng, "fused", genomes, r, l, mu, capture_at=t, capture=caps[0], seed=21, generation=3)
        _, so = _call(eng, "stepwise", genomes, r, l, mu, capture_at=t, capture=caps[1], seed=21, generation=3)
        _same(fo, so, what=(name, "capture"))
        assert torch.equal(caps[0], caps[1]), name
        written = t < so["frames"]
        assert bool((caps[1][~written] == 0).all()) and bool(written.any()) and bool((~written).any())
        idx = torch.nonzero(written).flatten()
        start = torch.full((M,), -1, dtype=torch.int32, device="cuda")
        start[idx] = torch.arange(idx.shape[0], dtype=torch.int32, device="cuda")
        states = caps[1][idx].contiguous()
        for fresh in (False, True):
            f, s = _both(eng, genomes, r, l, mu, states=states, start=start, fresh=fresh, seed=21, generation=3)
            _same(f, s, what=(name, "resume", fresh))
            if not fresh:
                _same(s, so, keys=("rewards", "frames", "scores"), what=(name, "uninterrupted"))
    eng.close()


# ---- 2. wide networks against the FP64 oracle ------------------------------------------------------------------------------
def _oracle(args):
    import oracle
    nodes, bias, genomes, right, left, mult, seed, generation, env_id, max_frames = args
    env = oracle.Atari()
    env.reset_to_state(oracle.STATE_START_1P if left == -3 else oracle.STATE_START_2P)
    opp = ("mlp", genomes[left]) if left >= 0 else ("score", None) if left == -2 else ("hardcoded", None)
    res, tr = env.episode(oracle.Shape.make(list(nodes), bias), opp, ("mlp", genomes[right]), mult=mult, seed=seed, env_id=env_id,
                          max_frames=max_frames, trace_cap=max_frames, generation=generation)
    return res.reward, res.frames, res.score1, res.score2, tr[:, 128:140].copy()


def _oracle_games(nodes, bias, genomes, right, left, mult, seed, generation, max_frames, keys=None):
    keys = np.arange(len(right)) if keys is None else keys
    jobs = [(nodes, bias, genomes, int(right[m]), int(left[m]), float(mult[m]), seed, generation, int(keys[m]), max_frames)
            for m in range(len(right))]
    with cf.ProcessPoolExecutor(max_workers=min(16, os.cpu_count() or 1)) as ex:
        return list(ex.map(_oracle, jobs))


def _check_oracle(out, rec, ref):
    rew, frm, sc = (out[k].cpu().numpy() for k in ("rewards", "frames", "scores"))
    rec = rec.cpu().numpy()
    for m, (r, f, s1, s2, tr) in enumerate(ref):
        assert (rew[m], frm[m], sc[m, 0], sc[m, 1]) == (r, f, s1, s2), m
        e = rec[m, :f]
        assert np.array_equal(e[:, 27] & 3, tr[:, 0]) and np.array_equal(e[:, 27] >> 2, tr[:, 1]), m          # decisions
        assert np.array_equal(e[:, 25], tr[:, 2]) and np.array_equal(e[:, 26], tr[:, 3]), m                     # scores
        valid = tr[:, 4].astype(np.int32) | tr[:, 5].astype(np.int32) << 1 | tr[:, 6].astype(np.int32) << 2
        assert np.array_equal(e[:, 24], valid), m
        assert np.array_equal(e[:, 28:32].copy().view("<i4")[:, 0], tr[:, 8:12].copy().view("<i4")[:, 0]), m      # timeout
        assert bool((rec[m, f:] == SENTINEL).all()), m


@pytest.mark.parametrize("nodes,bias", [((6, 48, 2), True), ((6, 64, 40, 2), True), ((6, 512, 512, 2), True), ((6, 48, 2), False)])
def test_wide_lists_match_the_oracle(ngp, nodes, bias):
    MF = 400
    eng = ngp.Engine(ngp.Config(NETWORK_SHAPE=nodes, BIAS=bias, MAX_FRAMES=MF), device=0)
    rng = np.random.RandomState(sum(nodes) + bias)
    genomes = _wide_genomes(rng, 44, nodes, bias)
    assert genomes.shape[1] == eng.gene_size
    g = _dev(genomes)
    ir, il, imu = _matches()
    for name, (right, left, mult) in (("irregular", (ir, il, imu)), ("skewed", _skewed(44))):
        r, l, mu = _lists_dev(right, left, mult)
        rec = torch.full((len(right), MF, 32), SENTINEL, dtype=torch.uint8, device="cuda")
        rc, out = _call(eng, "stepwise", g, r, l, mu, max_record=MF, record=rec, seed=9, generation=2)
        assert rc == 0, eng._L.ngp_last_error()
        _check_oracle(out, rec, _oracle_games(nodes, bias, genomes, right, left, mult, 9, 2, MF))
        rc, plain = _call(eng, "stepwise", g, r, l, mu, seed=9, generation=2)
        assert rc == 0
        _same(out, plain, what=name)
        assert out["frames_total"] == int(out["frames"].sum().item())
    eng.close()


# ---- 3. a wide round robin as a list gives ngp_evaluate's outcomes; replay_selfplay reproduces a game --------------------
@pytest.mark.parametrize("nodes,n,games", [((6, 64, 40, 2), 6, 3), ((6, 512, 512, 2), 4, 2)])
def test_wide_round_robin_list_equals_evaluate(ngp, nodes, n, games):
    from neuro_genetic_pong_self_play_b200 import reference_api as ref
    cfg = ngp.Config(SCHEDULE=ngp.SCHEDULE_ROUND_ROBIN, GAMES_TO_PLAY=games, NETWORK_SHAPE=nodes, POPULATION_SIZE=n, MAX_FRAMES=1500)
    eng = ngp.Engine(cfg, device=0)
    g = _dev(_wide_genomes(np.random.RandomState(5), n, nodes))
    ev = eng.evaluate(g, seed=21, generation=1, want_detail=True)
    gi, k = np.meshgrid(np.arange(n), np.arange(games), indexing="ij")
    r, l, _ = _lists_dev(gi.reshape(-1), ((gi + k + 1) % n).reshape(-1), None)
    pm = eng.play_matches(g, r, l, seed=21, generation=1)                      # driver=None: the per-frame driver for wide networks
    assert torch.equal(pm["rewards"], ev["rewards"].reshape(-1)) and torch.equal(pm["frames"], ev["frames"].reshape(-1))
    assert pm["frames_total"] == ev["frames_total"]
    with pytest.raises(ngp.NgpError):
        eng.play_matches(g, r, l, seed=21, generation=1, driver="fused")
    tb = ref.Toolbox(eng.config, engine=eng, seed=21)
    tb.generation = 1
    gg, kk = n - 1, games - 1
    rp = ref.replay_selfplay(tb, g, gg, kk, upsample=(1, 1))
    assert rp["steps"] == int(ev["frames"][gg, kk].item()) and rp["reward"] == ev["rewards"][gg, kk].item()
    assert rp["frames"].shape[0] == rp["steps"]
    eng.close()


# ---- 4. wide resume ----------------------------------------------------------------------------------------------------------
def test_wide_resume_and_captures_on_both_cores(ngp):
    nodes, MF = (6, 64, 40, 2), 300
    caps, fulls = [], []
    for core in (0, 1):
        eng = ngp.Engine(ngp.Config(NETWORK_SHAPE=nodes, MAX_FRAMES=MF, CORE=core), device=0)
        g = _dev(_wide_genomes(np.random.RandomState(11), 16, nodes))
        a = np.arange(8)
        right = np.concatenate([np.repeat(a, 8), [0, 3, 5]])
        left = np.concatenate([8 + np.tile(a, 8), [-1, -2, -3]])
        r, l, _ = _lists_dev(right, left, None)
        M = len(right)
        t = _dev((np.arange(M) * 37) % (MF + 40), torch.int32)                        # some past the end: never captured
        full = eng.play_matches_states(g, r, l, capture_at=t, max_record=MF, seed=6, generation=2)
        cap = full["capture"]
        written = t < full["frames"]
        assert bool(written.any()) and bool((~written).any()) and bool((cap[~written] == 0).all())
        idx = torch.nonzero(written).flatten()
        start = torch.full((M,), -1, dtype=torch.int32, device="cuda")
        start[idx] = torch.arange(idx.shape[0], dtype=torch.int32, device="cuda")
        res = eng.play_matches_states(g, r, l, states=cap[idx].contiguous(), start=start, max_record=MF, seed=6, generation=2)
        for k in ("rewards", "frames", "scores"):
            assert torch.equal(res[k], full[k]), (core, k)
        assert res["frames_total"] == full["frames_total"] - int(t[written].sum().item())
        steps = torch.arange(MF, device="cuda")[None, :]
        after = (steps >= torch.where(written, t, 0)[:, None]) & (steps < full["frames"][:, None])
        assert torch.equal(res["record"]["raw"][after], full["record"]["raw"][after]), core
        caps.append(cap)
        fulls.append(full)
        eng.close()
    assert torch.equal(caps[0], caps[1])
    for k in ("rewards", "frames", "scores"):
        assert torch.equal(fulls[0][k], fulls[1][k]), k


# ---- 5. beyond the grid limit: 65 536 chunks of 16 rows, the packed tcgen05 layer ----------------------------------------
def test_more_chunks_than_the_grid_limit(ngp):
    nodes, MF = (6, 64, 64, 2), 40
    eng = ngp.Engine(ngp.Config(NETWORK_SHAPE=nodes, MAX_FRAMES=MF), device=0)
    n = 65536
    genomes = _wide_genomes(np.random.RandomState(12), n, nodes)
    g = _dev(genomes)
    right, left = np.arange(0, n, 2), np.arange(1, n, 2)                     # chunk c = genome c; 65 535 is the second slice's
    r, l, _ = _lists_dev(right, left, None)
    M = len(right)
    rc, out = _call(eng, "stepwise", g, r, l, seed=3, generation=1)
    assert rc == 0, eng._L.ngp_last_error()
    # a second call on matches around chunk 65 535 (and at the start), with their keys: other chunk positions, same games
    sub = np.array([0, 1, 2, M - 3, M - 2, M - 1])
    rs, so = _call(eng, "stepwise", g, _dev(right[sub], torch.int32), _dev(left[sub], torch.int32), key=_dev(sub, torch.int32), seed=3,
                   generation=1)
    assert rs == 0
    for k in ("rewards", "frames", "scores"):
        assert torch.equal(so[k], out[k][torch.as_tensor(sub, device="cuda")]), k
    ref = _oracle_games(nodes, True, genomes, right[sub], left[sub], np.ones(len(sub)), 3, 1, MF, keys=sub)
    rew, frm, sc = (out[k].cpu().numpy() for k in ("rewards", "frames", "scores"))
    for i, m in enumerate(sub):
        assert (rew[m], frm[m], sc[m, 0], sc[m, 1]) == ref[i][:4], m
    eng.close()


# ---- 6. refusals -----------------------------------------------------------------------------------------------------------
def test_refusals_are_the_fused_calls_and_write_nothing(ngp):
    eng = ngp.Engine(ngp.Config(), device=0)
    g = _dev(_genomes(8, eng.gene_size, 5))
    ok = np.array([0, 1, 2, 3], np.int32)
    good_state = eng.play_matches_states(g, _dev(ok, torch.int32), _dev(ok, torch.int32), capture_at=_dev([0, 0, 0, 0], torch.int32),
                                         seed=1)["capture"]
    bad_state = good_state.clone()
    bad_state[0, 100] ^= 1
    i32 = lambda a: _dev(a, torch.int32)                                                   # noqa: E731
    cases = [dict(right=i32([0, 8, 2, 3])), dict(right=i32([0, -1, 2, 3])), dict(left=i32([0, 1, 8, 3])), dict(left=i32([0, -4, 2, 3])),
             dict(key=i32([0, 1, -1, 3])), dict(capture_at=i32([0, -1, 0, 0]), capture=True), dict(capture_at=i32([0, 1, 0, 0])),
             dict(start=i32([0, 4, -1, -1]), states=good_state), dict(start=i32([0, -2, -1, -1]), states=good_state),
             dict(start=i32([0, -1, -1, -1]), states=bad_state), dict(start=i32([0, -1, -1, -1]), states=good_state, left=i32([-3, 1, 2, 3])),
             dict(max_record=0, record=True), dict(max_record=16, record="misaligned")]
    wide = ngp.Engine(ngp.Config(NETWORK_SHAPE=(6, 48, 2)), device=0)
    gw = _dev(_genomes(8, wide.gene_size, 6))
    for e, genomes in ((eng, g), (wide, gw)):
        for case in cases:
            for driver in ("fused", "stepwise"):
                kw = dict(right=i32(ok), left=i32(ok))
                kw.update({k: v for k, v in case.items() if k not in ("capture", "record")})
                cap = torch.full((4, 512), SENTINEL, dtype=torch.uint8, device="cuda")
                raw = torch.full((4 * 16 * 32 + 64,), SENTINEL, dtype=torch.uint8, device="cuda")
                if case.get("capture"):
                    kw["capture"] = cap
                if case.get("record") is True:
                    kw["record"] = raw
                elif case.get("record") == "misaligned":
                    kw["record"] = ctypes.c_void_p(raw.data_ptr() + 4)
                if e is wide and driver == "fused":
                    continue
                rc, out = _call(e, driver, genomes, kw.pop("right"), kw.pop("left"), **kw)
                assert rc == -1, (case, driver, rc)                                              # NGP_ERR_INVALID
                assert bool((out["rewards"] == -7.0).all()) and bool((out["frames"] == -7).all()) and bool((out["scores"] == -7).all())
                assert bool((cap == SENTINEL).all()) and bool((raw == SENTINEL).all())
    rc, _ = _call(wide, "fused", gw, i32(ok), i32(ok))
    assert rc == -3 and b"wider" in wide._L.ngp_last_error()                                     # NGP_ERR_UNSUPPORTED
    with pytest.raises(ngp.NgpError):
        wide.record_matches(gw, i32(ok), i32(ok), driver="fused")
    wide.close()
    nine = ngp.Engine(ngp.Config(NETWORK_SHAPE=(6, 48, 9)), device=0)
    rc, _ = _call(nine, "stepwise", _dev(_genomes(8, nine.gene_size, 6)), i32(ok), i32(ok))
    assert rc == -1 and b"at most 8 outputs" in nine._L.ngp_last_error()
    nine.close()
    eng.close()


# ---- 7. scratch: repeated and interleaved calls, a fresh handle, evaluate ----------------------------------------------------
def test_scratch_reuse_and_evaluate_unchanged(ngp):
    nodes = (6, 64, 40, 2)
    cfg = ngp.Config(NETWORK_SHAPE=nodes, MAX_FRAMES=200, SCHEDULE=ngp.SCHEDULE_ROUND_ROBIN, POPULATION_SIZE=16, GAMES_TO_PLAY=2)
    eng = ngp.Engine(cfg, device=0)
    g = _dev(_wide_genomes(np.random.RandomState(13), 128, nodes))
    ev0 = eng.evaluate(g[:16].contiguous(), seed=2, want_detail=True)
    a = np.arange(64)
    small = _lists_dev(np.arange(8), np.array([9, 10, -1, -2, -3, 0, 1, 2]), None)
    big = _lists_dev(np.repeat(a, 64), 64 + np.tile(a, 64), None)
    runs = []
    for r, l, _ in (small, big, small):
        rc, out = _call(eng, "stepwise", g, r, l, seed=4, generation=1)
        assert rc == 0
        runs.append(out)
    _same(runs[0], runs[2])
    fresh = ngp.Engine(cfg, device=0)
    for (r, l, _), out in zip((small, big), runs):
        rc, f = _call(fresh, "stepwise", g, r, l, seed=4, generation=1)
        assert rc == 0
        _same(out, f)
    fresh.close()
    ev1 = eng.evaluate(g[:16].contiguous(), seed=2, want_detail=True)
    for k in ("fitness", "rewards", "frames"):
        assert torch.equal(ev0[k], ev1[k]), k
    assert ev0["frames_total"] == ev1["frames_total"]
    eng.close()


# ---- the reference API on a wide config ------------------------------------------------------------------------------------
def test_cross_play_and_branch_on_a_wide_config(ngp):
    from neuro_genetic_pong_self_play_b200 import reference_api as ref
    nodes = (6, 512, 512, 2)
    eng = ngp.Engine(ngp.Config(NETWORK_SHAPE=nodes, MAX_FRAMES=600), device=0)
    tb = ref.Toolbox(eng.config, engine=eng, seed=6)
    tb.generation = 2
    rng = np.random.RandomState(14)
    a, b = _dev(_wide_genomes(rng, 4, nodes)), _dev(_wide_genomes(rng, 3, nodes))
    ct = ref.cross_play(tb, a, b)                                              # (i, j) is list entry i * 3 + j: its key
    assert ct["reward"].shape == (4, 3)
    genomes = torch.cat([a, b])
    right, left = [2, 0, 3], [4 + 1, -3, 4 + 2]
    full = eng.record_matches(genomes, _dev(right, torch.int32), _dev(left, torch.int32), key=_dev([2 * 3 + 1, 1, 3 * 3 + 2], torch.int32),
                              max_record=600, seed=6, generation=2)
    assert full["frames"][0].item() == ct["frames"][2, 1].item() and full["rewards"][0].item() == ct["reward"][2, 1].item()
    assert full["frames"][2].item() == ct["frames"][3, 2].item() and full["rewards"][2].item() == ct["reward"][3, 2].item()
    for m in (0, 1):
        t = int(full["frames"][m].item()) // 2
        br = ref.branch(tb, genomes, right, left, m, t, key=int([7, 1, 11][m]))
        assert br["rewards"].item() == full["rewards"][m].item() and br["frames"].item() == full["frames"][m].item(), m
        T = int(full["frames"][m].item())
        assert torch.equal(br["record"]["raw"][0, :T], full["record"]["raw"][m, :T]), m
    eng.close()
