"""Match sessions on the GPU (ngp_session_*, Engine.session, reference_api.play_policy): a match list advanced one env.step at a
time, with seats whose decisions the caller supplies.  Without external seats a session must give ngp_play_matches_stepwise's
and the fused rollout's bits; external seats fed the decisions a recorded game took must replay it bit for bit; NEED, obs and
captures must be what the record and ngp_play_matches_states say; refusals write nothing; other calls between two steps do not
disturb a session; a step neither synchronises nor launches more than the decide and the frame kernels (narrow networks)."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

SENTINEL = 0xAB
EXT = -4


@pytest.fixture(scope="module")
def ngp():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import neuro_genetic_pong_self_play_b200 as m
    return m


def _dev(a, dtype=None):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype).cuda()


def _i32(a):
    return _dev(np.asarray(a), torch.int32)


def _genomes(n, G, seed):
    return (np.random.RandomState(seed).standard_normal((n, G)) * 2).astype(np.float32)


def _wide_genomes(rng, n, nodes):
    G = sum((a + 1) * c for a, c in zip(nodes[:-1], nodes[1:]))
    g = np.zeros((n, G), np.float32)
    off = 0
    for a, c in zip(nodes[:-1], nodes[1:]):
        cnt = (a + 1) * c
        g[:, off:off + cnt] = (rng.standard_normal((n, cnt)) * 3.0 / np.sqrt(a + 1)).astype(np.float32)
        off += cnt
    return g


def _narrow_lists(ngp, eng):
    from test_gpu_matches_stepwise import _narrow_lists as lists
    return lists(ngp, eng)


def _run(sess, feed=None, every=None, capture_at=None):
    """Steps `sess` until no match runs.  feed(k) -> u8[M, 2] actions of step k (None: zeros); every(k, sess) is called after
    begin (k = 0) and after every step k.  capture_at: the step whose capture is returned (cloned)."""
    M = sess.n
    zeros = torch.zeros((M, 2), dtype=torch.uint8, device="cuda")
    cap = None
    if every:
        every(0, sess)
    k = 0
    while k % 8 or sess.running():
        k += 1
        c = sess.step(zeros if feed is None else feed(k), capture=capture_at == k)
        if c is not None:
            cap = c.clone()
        if every:
            every(k, sess)
    return cap


def _stepwise(ngp, eng, genomes, right, left, mult=None, key=None, states=None, start=None, fresh=False, capture_at=None, max_record=0,
              seed=0, generation=0, driver="stepwise"):
    out = eng.play_matches_states(genomes, right, left, mult, key=key, states=states, start=start, fresh=fresh, capture_at=capture_at,
                                  max_record=max_record, seed=seed, generation=generation, driver=driver)
    return out


def _same(a, b, what="", record=True, t0=None):
    """rewards, frames, scores, frames_total and the record entries written (from t0[m], the start frame of a resumed match)"""
    for k in ("rewards", "frames", "scores"):
        assert torch.equal(a[k], b[k]), (what, k)
    assert a["frames_total"] == b["frames_total"], (what, a["frames_total"], b["frames_total"])
    if record and "record" in a and "record" in b:
        steps = torch.arange(a["record"]["raw"].shape[1], device="cuda")[None, :]
        written = steps < a["frames"][:, None]
        if t0 is not None:
            written &= steps >= torch.as_tensor(t0, device="cuda")[:, None]
        assert torch.equal(a["record"]["raw"][written], b["record"]["raw"][written]), what


# ---- 1. no external seat: ngp_play_matches_stepwise's and the fused rollout's bits ----------------------------------------------
@pytest.mark.parametrize("core", [0, 1])
def test_session_without_external_seats_equals_both_drivers(ngp, core):
    eng = ngp.Engine(ngp.Config(CORE=core, MAX_FRAMES=0 if core else 500), device=0)
    T = 400
    for name, genomes, right, left, mult in _narrow_lists(ngp, eng):
        if not core and name != "irregular":
            continue
        r, l = _i32(right), _i32(left)
        mu = None if mult is None else _dev(mult, torch.float64)
        with eng.session(genomes, r, l, mu, max_record=T, seed=21, generation=3) as s:
            _run(s)
            got = s.result()
        for driver in ("stepwise", "fused"):
            ref = _stepwise(ngp, eng, genomes, r, l, mu, max_record=T, seed=21, generation=3, driver=driver)
            _same(got, ref, (name, driver))
        if name != "irregular":
            continue
        # resumed and fresh starts from captured states
        M = r.shape[0]
        t = _i32((np.arange(M) * 53) % 700)
        full = _stepwise(ngp, eng, genomes, r, l, mu, capture_at=t, seed=21, generation=3)
        written = t < full["frames"]
        idx = torch.nonzero(written).flatten()
        start = torch.full((M,), -1, dtype=torch.int32, device="cuda")
        start[idx] = torch.arange(idx.shape[0], dtype=torch.int32, device="cuda")
        states = full["capture"][idx].contiguous()
        for fresh in (False, True):
            with eng.session(genomes, r, l, mu, states=states, start=start, fresh=fresh, max_record=T, seed=21, generation=3) as s:
                _run(s)
                got = s.result()
            ref = _stepwise(ngp, eng, genomes, r, l, mu, states=states, start=start, fresh=fresh, max_record=T, seed=21, generation=3)
            _same(got, ref, (name, "start", fresh), t0=None if fresh else torch.where(written, t, 0))
            if not fresh:
                for k in ("rewards", "frames", "scores"):
                    assert torch.equal(got[k], full[k]), k
    eng.close()


def test_wide_session_without_external_seats_equals_stepwise(ngp):
    nodes = (6, 512, 512, 2)
    eng = ngp.Engine(ngp.Config(NETWORK_SHAPE=nodes, MAX_FRAMES=300), device=0)
    g = _dev(_wide_genomes(np.random.RandomState(3), 12, nodes))
    right = np.array([0, 1, 2, 3, 4, 5, 6, 7, 0, 0, 1, 2])
    left = np.array([8, 9, 10, 11, -1, -2, -3, 1, 2, 3, -3, 9])
    r, l = _i32(right), _i32(left)
    with eng.session(g, r, l, max_record=300, seed=5, generation=1) as s:
        _run(s)
        got = s.result()
    _same(got, _stepwise(ngp, eng, g, r, l, max_record=300, seed=5, generation=1), "wide")
    eng.close()


# ---- 2 + 3. external seats fed a recorded game's decisions replay it; NEED and obs follow the record ------------------------------
def _expected_obs(rec_loc, k, have_last):
    """utils.inference's rows (left mirrored, right) of frame k from the record's float loc, in float64"""
    loc = rec_loc[:, k].astype(np.float64)                      # [M, 3, 2]
    prev = rec_loc[:, k - 1].astype(np.float64) if k > 0 else loc
    last = np.where(have_last[:, None], prev[:, 0], loc[:, 0])  # [M, 2]
    ball = loc[:, 0]
    right = np.stack([ball[:, 1], ball[:, 0], last[:, 1], last[:, 0], loc[:, 2, 0], loc[:, 1, 0]], axis=1) / 160.0
    left = np.stack([160.0 - ball[:, 1], ball[:, 0], 160.0 - last[:, 1], last[:, 0], loc[:, 1, 0], loc[:, 2, 0]], axis=1) / 160.0
    return np.stack([left, right], axis=1)                      # [M, 2, 6]


def _replay_check(ngp, eng, genomes, right, left, ext_right, ext_left, T, states=None, start=None, t0=None, check_obs=True):
    """Records the list, then replays it in a session whose seats (ext_right, ext_left masks) are external, fed the recorded
    decisions; checks the result bit for bit and NEED / obs on every step (fresh starts)."""
    M = len(right)
    r, l = _i32(right), _i32(left)
    kw = dict(states=states, start=start, max_record=T, seed=7, generation=2)
    orig = _stepwise(ngp, eng, genomes, r, l, **kw)
    sr = np.where(ext_right, EXT, right)
    sl = np.where(ext_left, EXT, left)
    act = orig["record"]["act"]
    t0 = np.zeros(M, np.int64) if t0 is None else np.asarray(t0)
    t0d = torch.as_tensor(t0, device="cuda")
    rec_loc = orig["record"]["loc"].cpu().numpy()
    rec_valid = orig["record"]["valid"].cpu().numpy()
    frames = orig["frames"].cpu().numpy()
    has_ext = ext_left | ext_right
    n_need = [0]
    assert not (ext_left & ~(ext_right | (left >= 0))).any()       # an external left seat faces a genome or an external right seat

    def feed(k):
        a = act[torch.arange(M, device="cuda"), (t0d + k - 1).clamp(max=T - 1)].long()
        return torch.stack([a & 3, a >> 2], dim=1).to(torch.uint8).contiguous()

    def every(k, s):
        if not check_obs:
            return
        flags = s.flags.cpu().numpy()
        f = t0 + k                                             # the frame each match has just played
        running = f < frames
        need = (flags & 1) != 0
        fc = np.minimum(f, T - 1)
        expect = running & has_ext & (rec_valid[np.arange(M), fc] == 7)
        assert np.array_equal(need, expect), (k, np.nonzero(need != expect))
        assert np.array_equal((flags & 2) != 0, ~running), k
        if need.any():
            have_last = (rec_valid[np.arange(M), np.maximum(fc - 1, 0)] & 1).astype(bool) & (f > 0)
            loc_k = rec_loc[np.arange(M), fc]
            loc_p = rec_loc[np.arange(M), np.maximum(fc - 1, 0)]
            pair = np.stack([loc_p, loc_k], axis=1)
            exp = _expected_obs(pair, 1, have_last).astype(np.float32)
            obs = s.obs.cpu().numpy()
            seats = need[:, None] & np.stack([ext_left, ext_right], axis=1)
            got, want = obs[seats], exp[seats]
            tol = 2 * np.spacing(np.abs(want).astype(np.float32))
            assert bool((np.abs(got.astype(np.float64) - want.astype(np.float64)) <= tol).all()), k
            n_need[0] += int(seats.sum())

    with eng.session(genomes, _i32(sr), _i32(sl), **kw) as s:
        _run(s, feed, every)
        got = s.result()
    _same(got, orig, "replay", t0=t0)
    assert not check_obs or n_need[0] > 0
    return orig


def test_external_seats_replay_a_recorded_game(ngp):
    eng = ngp.Engine(ngp.Config(MAX_FRAMES=900), device=0)
    g = _dev(_genomes(10, eng.gene_size, 4))
    right = np.array([0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 0, 1])
    left = np.array([5, 6, 7, -3, -1, -2, 0, 1, 2, -3, 3, 4])
    T = 900
    xr = np.array([1, 0, 1, 1, 1, 1, 0, 0, 1, 1, 1, 0], bool)
    xl = np.array([0, 1, 1, 0, 0, 0, 1, 1, 1, 0, 0, 0], bool)          # left external only against a genome or an external right seat
    _replay_check(ngp, eng, g, right, left, xr, xl, T)
    # resumed from states captured mid-game: the session's steps continue from the captured frame
    M = len(right)
    t = np.array([30, 100, 5, 250, 0, 60, 400, 1, 90, 120, 33, 77])
    full = _stepwise(ngp, eng, g, _i32(right), _i32(left), capture_at=_i32(t), seed=7, generation=2)
    assert bool((full["frames"] > _i32(t)).all())
    _replay_check(ngp, eng, g, right, left, xr, xl, T, states=full["capture"], start=_i32(np.arange(M)), t0=t, check_obs=False)
    eng.close()


def test_external_seats_replay_on_a_wide_network(ngp):
    nodes = (6, 512, 512, 2)
    eng = ngp.Engine(ngp.Config(NETWORK_SHAPE=nodes, MAX_FRAMES=300), device=0)
    g = _dev(_wide_genomes(np.random.RandomState(8), 8, nodes))
    right = np.array([0, 1, 2, 3, 4, 5, 6, 7])
    left = np.array([4, 5, -3, -1, 0, 1, 2, 3])
    xr = np.array([1, 0, 1, 1, 1, 0, 1, 0], bool)
    xl = np.array([0, 1, 0, 0, 1, 1, 0, 0], bool)
    _replay_check(ngp, eng, g, right, left, xr, xl, 300)
    # no genome row at all: genomes None, an external right seat against the bots
    sr, sl = _i32([EXT, EXT, EXT]), _i32([-1, -2, -3])
    with eng.session(None, sr, sl, seed=1) as s:
        _run(s)
        out = s.result()
    assert bool((out["frames"] > 0).all())
    eng.close()


# ---- 4. captures ---------------------------------------------------------------------------------------------------------------
def test_step_capture_equals_play_matches_states_and_resumes(ngp):
    eng = ngp.Engine(ngp.Config(MAX_FRAMES=1200), device=0)
    g = _dev(_genomes(6, eng.gene_size, 9))
    right, left = _i32([0, 1, 2, 3, 4, 5]), _i32([1, -3, 3, -1, -2, 0])
    t = 150
    with eng.session(g, right, left, seed=3, generation=4) as s:
        cap = _run(s, capture_at=t)
        got = s.result()
    ref = _stepwise(ngp, eng, g, right, left, capture_at=_i32([t] * 6), seed=3, generation=4)
    running = ref["frames"] > t
    assert bool(running.any())
    assert torch.equal(cap[running], ref["capture"][running])
    idx = torch.nonzero(running).flatten()
    start = torch.full((6,), -1, dtype=torch.int32, device="cuda")
    start[idx] = torch.arange(idx.shape[0], dtype=torch.int32, device="cuda")
    res = _stepwise(ngp, eng, g, right, left, states=cap[idx].contiguous(), start=start, seed=3, generation=4)
    for k in ("rewards", "frames", "scores"):
        assert torch.equal(res[k], got[k]), k
    eng.close()


# ---- 5. refusals, bad actions, steps after the end ------------------------------------------------------------------------------
def _begin_raw(eng, genomes, right, left, states=None, start=None, record=None, max_record=0, obs=None):
    from neuro_genetic_pong_self_play_b200.engine import _p, _stream
    M = right.shape[0]
    out = {"rewards": torch.full((M,), -7.0, dtype=torch.float64, device="cuda"),
           "frames": torch.full((M,), -7, dtype=torch.int32, device="cuda"),
           "scores": torch.full((M, 2), -7, dtype=torch.int32, device="cuda"),
           "obs": torch.full((M, 2, 6), -7.0, dtype=torch.float32, device="cuda"),
           "flags": torch.full((M,), SENTINEL, dtype=torch.uint8, device="cuda")}
    h = ctypes.c_void_p(12345)
    rec_p = record if isinstance(record, ctypes.c_void_p) else _p(record)
    st_p = states if isinstance(states, ctypes.c_void_p) else _p(states)
    rc = eng._L.ngp_session_begin(eng._h, _p(genomes), 0 if genomes is None else genomes.shape[0], _p(right), _p(left), None, None, M,
                                  st_p, 0 if states is None else 1, _p(start), 0, max_record, rec_p, 0, 0, _p(out["rewards"]),
                                  _p(out["frames"]), _p(out["scores"]), obs if obs is not None else _p(out["obs"]), _p(out["flags"]),
                                  _stream(eng.device), ctypes.byref(h))
    torch.cuda.synchronize()
    return rc, h, out


def test_refusals_write_nothing_and_create_no_session(ngp):
    eng = ngp.Engine(ngp.Config(), device=0)
    g = _dev(_genomes(8, eng.gene_size, 5))
    ok = [0, 1, 2, 3]
    good = eng.play_matches_states(g, _i32(ok), _i32(ok), capture_at=_i32([0, 0, 0, 0]), seed=1)["capture"]
    bad = good.clone()
    bad[0, 100] ^= 1
    raw = torch.full((4 * 16 * 32 + 64,), SENTINEL, dtype=torch.uint8, device="cuda")
    cases = [dict(right=[0, 8, 2, 3]), dict(right=[0, -1, 2, 3]), dict(right=[0, -5, 2, 3]), dict(left=[0, 1, 8, 3]), dict(left=[0, -5, 2, 3]),
             dict(start=[0, 1, -1, -1], states=good[:1].contiguous()), dict(start=[0, -2, -1, -1], states=good[:1].contiguous()),
             dict(start=[0, -1, -1, -1], states=bad[:1].contiguous()), dict(start=[0, -1, -1, -1], states=good[:1].contiguous(), left=[-3, 1, 2, 3]),
             dict(record=ctypes.c_void_p(raw.data_ptr() + 4), max_record=16), dict(states=ctypes.c_void_p(good.data_ptr() + 8), start=[0, -1, -1, -1]),
             dict(genomes=None), dict(right=[EXT, 1, 2, 3], genomes=None)]
    for case in cases:
        kw = dict(genomes=g, right=ok, left=ok)
        kw.update(case)
        rc, h, out = _begin_raw(eng, kw["genomes"], _i32(kw["right"]), _i32(kw["left"]), states=kw.get("states"),
                                start=None if "start" not in kw else _i32(kw["start"]), record=kw.get("record"), max_record=kw.get("max_record", 0))
        assert rc == -1, (case, rc)
        assert h.value is None, case
        for k in ("rewards", "frames", "scores", "obs"):
            assert bool((out[k] == -7).all()), (case, k)
        assert bool((out["flags"] == SENTINEL).all()) and bool((raw == SENTINEL).all()), case
    # the other match-list entry points keep refusing the external code
    with pytest.raises(ngp.NgpError):
        eng.play_matches(g, _i32([EXT, 1]), _i32([0, 1]))
    with pytest.raises(ngp.NgpError):
        eng.play_matches_states(g, _i32([0, 1]), _i32([EXT, 1]), driver="stepwise")
    eng.close()


def test_bad_actions_play_none_and_are_reported(ngp):
    eng = ngp.Engine(ngp.Config(MAX_FRAMES=400), device=0)
    g = _dev(_genomes(4, eng.gene_size, 2))
    r, l = _i32([EXT, EXT, 0, EXT]), _i32([-1, 0, 1, -3])
    M = 4
    runs = []
    for v in (0, 7):
        acts = torch.full((M, 2), v, dtype=torch.uint8, device="cuda")
        with eng.session(g, r, l, max_record=400, seed=2) as s:
            _run(s, feed=lambda k: acts)
            if v:
                assert s.running() == 0
                with pytest.raises(ngp.NgpError, match="outside 0..2"):
                    s.result()
                rc, running, total = s._status()
                assert rc == -1 and running == 0
                runs.append({"rewards": s.rewards.clone(), "frames": s.frames.clone(), "scores": s.scores.clone(), "frames_total": total,
                             "record": {"raw": s._raw.clone()}})
            else:
                runs.append(s.result())
                runs[-1]["record"] = {"raw": runs[-1]["record"]["raw"].clone()}
                # steps after the end change nothing
                before = {k: t.clone() for k, t in (("obs", s.obs), ("flags", s.flags), ("scores", s.scores), ("rewards", s.rewards),
                                                     ("frames", s.frames))}
                for _ in range(3):
                    s.step(torch.full((M, 2), 2, dtype=torch.uint8, device="cuda"))
                for k, t in before.items():
                    assert torch.equal(t, getattr(s, k)), k
                assert bool((s.flags & 2 != 0).all()) and s.result()["frames_total"] == runs[-1]["frames_total"]
    _same(runs[0], runs[1], "bad actions = NONE")
    eng.close()


# ---- 6. other calls between two steps ------------------------------------------------------------------------------------------
def test_other_calls_between_steps_do_not_disturb_a_session(ngp):
    for nodes in ((6, 2, 2), (6, 64, 64, 2)):
        cfg = ngp.Config(NETWORK_SHAPE=nodes, MAX_FRAMES=250, SCHEDULE=ngp.SCHEDULE_ROUND_ROBIN, POPULATION_SIZE=8, GAMES_TO_PLAY=2)
        eng = ngp.Engine(cfg, device=0)
        rng = np.random.RandomState(21)
        g = _dev(_wide_genomes(rng, 8, nodes))
        other = _dev(_wide_genomes(rng, 8, nodes))
        r, l = _i32([0, 1, 2, 3, EXT, 5]), _i32([4, 5, -3, EXT, 6, -1])
        r2, l2 = _i32([7, 6, EXT]), _i32([-2, 0, 1])

        def feed_for(n):
            def feed(k):
                return torch.tensor([[(k + i) % 3, (2 * k + i) % 3] for i in range(n)], dtype=torch.uint8, device="cuda")
            return feed

        with eng.session(g, r, l, max_record=250, seed=4) as s:
            _run(s, feed_for(6))
            alone = {k: v.clone() if torch.is_tensor(v) else v for k, v in s.result().items() if k != "record"}
            alone["record"] = {"raw": s.result()["record"]["raw"].clone()}
        with eng.session(g, r2, l2, max_record=250, seed=4) as s2:
            _run(s2, feed_for(3))
            alone2 = {k: v.clone() if torch.is_tensor(v) else v for k, v in s2.result().items() if k != "record"}
        a = eng.session(g, r, l, max_record=250, seed=4)
        b = eng.session(g, r2, l2, max_record=250, seed=4)
        fa, fb = feed_for(6), feed_for(3)
        k = 0
        while a.running() or b.running():
            for _ in range(8):
                k += 1
                a.step(fa(k))
                if k % 3 == 0:
                    eng.evaluate(other, seed=9, want_detail=True)               # re-packs the wide weights
                if k % 5 == 0:
                    eng.play_matches_states(other, _i32([0, 1]), _i32([2, -1]), seed=3, driver="stepwise")
                b.step(fb(k))
        _same(a.result(), alone, nodes)
        _same(b.result(), alone2, nodes, record=False)
        a.close()
        b.close()
        eng.close()


# ---- 7. launches and CUDA graphs -----------------------------------------------------------------------------------------------
def test_narrow_step_launches_and_graph_replay(ngp):
    eng = ngp.Engine(ngp.Config(MAX_FRAMES=700), device=0)
    g = _dev(_genomes(8, eng.gene_size, 6))
    r, l = _i32([EXT, 1, EXT, 3, EXT, 5]), _i32([0, 2, -3, EXT, -1, 4])
    M = 6

    def policy(obs):                                   # HardcodedAi's rule on obs (dumb_ais.py:1-8)
        return torch.where(obs[..., 1] < obs[..., 4], 1, torch.where(obs[..., 1] > obs[..., 4], 2, 0)).to(torch.uint8)

    with eng.session(g, r, l, max_record=700, seed=8) as s:
        acts = torch.zeros((M, 2), dtype=torch.uint8, device="cuda")
        n0 = eng.launches
        s.step(acts)
        assert eng.launches - n0 == 2
        n_steps = 1
        while s.running():
            acts.copy_(policy(s.obs))
            s.step(acts)
            n_steps += 1
        eager = {k: v.clone() if torch.is_tensor(v) else v for k, v in s.result().items() if k != "record"}
        eager["record"] = {"raw": s.result()["record"]["raw"].clone()}
    with eng.session(g, r, l, max_record=700, seed=8) as s:
        acts = torch.zeros((M, 2), dtype=torch.uint8, device="cuda")
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):              # the first step (all-zero decisions) eagerly, as above
            s.step(acts)
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for _ in range(16):
                acts.copy_(policy(s.obs))
                s.step(acts)
        replays = 0
        while s.running():
            graph.replay()
            replays += 1
        assert replays * 16 >= n_steps - 1
        _same(s.result(), eager, "graph")
    eng.close()


# ---- 8. play_policy: an outside policy plays a 1 024-match list; render_recorded re-renders a game ---------------------------------
def test_play_policy_with_a_torch_policy_and_render(ngp):
    from neuro_genetic_pong_self_play_b200 import reference_api as ref
    eng = ngp.Engine(ngp.Config(MAX_FRAMES=1500), device=0)
    tb = ref.Toolbox(eng.config, engine=eng, seed=11)
    tb.generation = 3
    g = _dev(_genomes(16, eng.gene_size, 12))
    M = 1024
    right = np.full(M, EXT)
    left = np.array([-1, -2, -3, 0, 5, 9, 15, -1])[np.arange(M) % 8]

    def policy(obs):
        return torch.where(obs[:, 1] < obs[:, 4], 1, torch.where(obs[:, 1] > obs[:, 4], 2, 0)).to(torch.uint8)

    calls = [0]

    def counted(obs):
        calls[0] += 1
        assert obs.dim() == 2 and obs.shape[1] == 6 and obs.shape[0] > 0
        return policy(obs)

    res = ref.play_policy(tb, g, right, left, counted)
    assert calls[0] > 0 and bool((res["frames"] > 0).all()) and res["frames_total"] == int(res["frames"].sum().item())
    m = 2                                                            # a robot match
    T = int(res["frames"][m].item())
    (pix, ram), = ref.render_recorded(tb, res, [m], want_ram=True)
    assert pix.shape[0] == T
    assert torch.equal(ram[:, 13], res["record"]["score"][m, :T, 0]) and torch.equal(ram[:, 14], res["record"]["score"][m, :T, 1])

    class Bot:                                                       # a reference-style model object (dumb_ais.HardcodedAi)
        def run(self, vec):
            return [1, 0] if vec[1] < vec[4] else ([0, 1] if vec[1] > vec[4] else [0, 0])

    few = ref.play_policy(tb, g, right[:8], left[:8], ref.model_policy(Bot()))
    again = ref.play_policy(tb, g, right[:8], left[:8], policy)
    for k in ("rewards", "frames", "scores"):
        assert torch.equal(few[k], again[k]), k
    eng.close()
