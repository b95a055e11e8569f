"""Every code path of the policy network against the FP64 oracle (numpy_nn.NeuralNetwork.run restated in oracle/episode_oracle.c).

- ngp_mlp_forward's dispatch: a table of shapes, each naming the kernels it must launch (checked in a torch.profiler trace, so a
  dispatch change cannot silently empty a case), with BIAS on and off, through mlp_forward, mlp_prepare + mlp_forward_prepared
  and the FP32 FFMA fall-back (mlp_no_tf32).  Bar: outputs within rtol 1e-5 / atol 1e-7, actions equal on the seeded data.
- The argmax rules on every one of those paths, exactly: an exact tie and two outputs that both saturate to 1.0 give UP (index 0
  wins), a maximum at output 2 or later gives DOWN, one output always gives UP.
- The fused rollout's generic FP64 loop (every shape but [6,2,2] with bias): evaluate, round robin and record_matches, bit for bit.
- The stepwise driver's tensor-core layers (mlp_layer_tmem_kernel<64> / <128>) in whole episodes, bit for bit.
- More than 65 535 genomes: the wide kernels take the genome from grid.y / grid.z, which CUDA caps at 65 535."""
import concurrent.futures as cf
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

UP, DOWN = 1, 2
RTOL, ATOL = 1e-5, 1e-7


@pytest.fixture(scope="module")
def ngp():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import neuro_genetic_pong_self_play_b200 as m
    return m


@pytest.fixture(scope="module")
def pool():
    with cf.ProcessPoolExecutor(max_workers=min(16, os.cpu_count() or 1)) as ex:
        yield ex


def _genomes(rng, n, nodes, bias):
    """Weights scaled by 1/sqrt(fan-in) per layer so that hidden units do not all saturate and decisions depend on the inputs."""
    b = 1 if bias else 0
    layers = [(rng.standard_normal((n, (a + b) * c)) * 3.0 / np.sqrt(a + b)) for a, c in zip(nodes[:-1], nodes[1:])]
    return np.concatenate(layers, axis=1).astype(np.float32)


def _oracle_rows(nodes, genomes, x, bias):
    import oracle
    n, envs = x.shape[:2]
    out = np.zeros((n, envs, nodes[-1])); act = np.zeros((n, envs), np.uint8)
    for g in range(n):
        for e in range(envs):
            out[g, e], act[g, e] = oracle.mlp_forward(list(nodes), genomes[g], x[g, e].astype(np.float64), bias=bias)
    return out, act


# ---------------------------------------------------------------------------------------------------------------------------
# 1a. dispatch matrix of ngp_mlp_forward
# ---------------------------------------------------------------------------------------------------------------------------
def _k(name, arg=None):
    """A kernel as the trace may name it: demangled (name<arg>) or mangled (nameILi6E / nameILb0E)."""
    if arg is None:
        return (name,)
    mangled = {"false": "Lb0E", "true": "Lb1E"}.get(arg, f"Li{arg}E")
    return (f"{name}<{arg}>", f"{name}I{mangled}")


SMALL = _k("mlp_small_kernel")
N6, N0 = _k("mlp_narrow_in_kernel", 6), _k("mlp_narrow_in_kernel", 0)
LF, LT, DEC = _k("mlp_layer_kernel", "false"), _k("mlp_layer_kernel", "true"), _k("mlp_decide_kernel")
TF32 = _k("mlp_layer_tf32_v2_kernel")
PACK, TM64, TM128 = _k("mlp_pack_layer_kernel"), _k("mlp_layer_tmem_kernel", 64), _k("mlp_layer_tmem_kernel", 128)
LS, LW1, LW2 = _k("mlp_last_small_kernel"), _k("mlp_last_wide_kernel", 1), _k("mlp_last_wide_kernel", 2)
ROUTES = ("plain", "prepared", "no_tf32")


def _same(*ks):
    return {r: set(ks) for r in ROUTES}


# (id, nodes, envs, {route: kernels that must run}); mlp_prepare packs nothing (and launches nothing) unless a hidden layer
# is at least 64 wide on both sides with a fan-in that is a multiple of 4
CASES = [
    ("small_1out", (6, 1), 5, _same(SMALL)),
    ("small_3out", (6, 4, 3), 7, _same(SMALL)),
    ("small_32out", (6, 32, 32), 3, _same(SMALL)),
    ("small_8layers", (6, 8, 8, 8, 8, 8, 8, 5), 4, _same(SMALL)),
    # a hidden layer after the first with fan-in + bias <= 8: the run-time fan-in narrow kernel
    ("narrow0", (6, 40, 4, 40, 2), 9, _same(N6, LF, N0, LS)),
    # fewer than 16 environments: no tensor-core layer, on any route
    ("ffma_few_envs", (6, 64, 64, 2), 8, _same(N6, LF, LS)),
    # fan-in 70 (not a multiple of 4: never packed), 100 outputs (not a multiple of 128)
    ("tf32_ragged", (6, 70, 100, 2), 20, {"plain": {N6, TF32, LS}, "prepared": {N6, TF32, LS}, "no_tf32": {N6, LF, LS}}),
] + [
    # fan-in 68 (a multiple of 4, not of 16), 200 outputs; 3 outputs on the warp-per-row action layer
    (f"tmem_envs{e}", (6, 68, 200, 3), e, {"plain": {N6, TF32, LS}, "prepared": {N6, PACK, TM64 if e <= 64 else TM128, LS},
                                           "no_tf32": {N6, LF, LS}})
    for e in (16, 17, 64, 65, 130)
] + [
    ("last_small_5out", (6, 40, 5), 11, _same(N6, LS)),
    ("last_small_8out", (6, 40, 8), 11, _same(N6, LS)),
    ("last_wide_1out", (6, 128, 1), 19, _same(N6, LW1)),
    ("last_wide_2out", (6, 64, 256, 2), 33, {"plain": {N6, TF32, LW2}, "prepared": {N6, PACK, TM64, LW2}, "no_tf32": {N6, LF, LW2}}),
    ("decide_9out", (6, 40, 9), 6, _same(N6, LT, DEC)),
    # action-layer weights over 48 KB: 8 x 1541 x 4 B with bias, 8 x 1540 x 4 B without
    ("decide_48kb", (6, 1540, 8), 3, _same(N6, LT, DEC)),
]
CASE_IDS = [c[0] for c in CASES]


def _profiled(fn):
    """fn()'s result and the names of the GPU kernels it launched (torch.profiler, CUDA activity)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    return res, {e.name for e in prof.events()}


def _run_route(eng, route, g, x):
    if route == "plain":
        return eng.mlp_forward(g, x)
    if route == "prepared":
        eng.mlp_prepare(g)
        return eng.mlp_forward_prepared(g, x)
    eng.set_option("mlp_no_tf32", 1)
    try:
        return eng.mlp_forward(g, x)
    finally:
        eng.set_option("mlp_no_tf32", 0)


def _check_route(route, act, out, ref_out, ref_act, what):
    np.testing.assert_allclose(out.cpu().numpy(), ref_out, rtol=RTOL, atol=ATOL, err_msg=f"{what} {route}")
    assert np.array_equal(act.cpu().numpy(), ref_act), (what, route, act.cpu().numpy(), ref_act)


@pytest.mark.parametrize("bias", [True, False])
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_mlp_dispatch_matrix(ngp, case, bias):
    name, nodes, envs, kernels = case
    eng = ngp.Engine(ngp.Config(NETWORK_SHAPE=nodes, BIAS=bias), device=0)
    rng = np.random.RandomState(sum(nodes) + envs + bias)
    n = 3
    genomes = _genomes(rng, n, nodes, bias)
    assert genomes.shape[1] == eng.gene_size
    x = rng.random_sample((n, envs, 6)).astype(np.float32)
    ref_out, ref_act = _oracle_rows(nodes, genomes, x, bias)
    g, xd = torch.from_numpy(genomes).cuda(), torch.from_numpy(x).cuda()
    for route in ROUTES:
        (act, out), names = _profiled(lambda: _run_route(eng, route, g, xd))
        for k in kernels[route]:
            assert any(alt in nm for alt in k for nm in names), (name, route, k[0], sorted(names))
        _check_route(route, act, out, ref_out, ref_act, name)
    eng.close()


# ---------------------------------------------------------------------------------------------------------------------------
# 1b. the argmax rules on every path: exact actions
# ---------------------------------------------------------------------------------------------------------------------------
def _rule_genomes(rng, n, nodes, bias, rule, m=None):
    """Random hidden layers; the action layer rewritten so that `rule` decides every row."""
    b = 1 if bias else 0
    genomes = _genomes(rng, n, nodes, bias).astype(np.float64)
    ni, no = nodes[-2], nodes[-1]
    last = genomes[:, genomes.shape[1] - (ni + b) * no:].reshape(n, no, ni + b)
    base = rng.standard_normal((n, ni + b)) * 0.5 / np.sqrt(ni + b)
    if rule == "tie":                 # rows 0 and 1 identical, every other row lower by the (positive) sum of its inputs
        last[:] = base[:, None, :] - 1.0
        last[:, 0] = last[:, 1] = base
    elif rule == "saturated":         # every output's sigmoid is 1.0 in FP64, the pre-activations grow with the index
        for o in range(no):
            if bias:
                last[:, o, :ni] = 0.0
                last[:, o, ni] = 50.0 + 10.0 * o
            else:
                last[:, o, :] = 1000.0 + 200.0 * o
    elif rule == "late_max":          # the maximum at output m >= 2, outputs 0 and 1 tied below it
        last[:] = base[:, None, :] - 1.0
        last[:, m] = base
    genomes[:, genomes.shape[1] - (ni + b) * no:] = last.reshape(n, -1)
    return genomes.astype(np.float32)


def _rules(no):
    if no == 1:
        return [("single", None, UP)]
    rules = [("tie", None, UP), ("saturated", None, UP)]
    if no >= 3:
        rules += [("late_max", m, DOWN) for m in sorted({2, no - 1})]
    return rules


@pytest.mark.parametrize("bias", [True, False])
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_mlp_argmax_rules(ngp, case, bias):
    name, nodes, envs, _ = case
    eng = ngp.Engine(ngp.Config(NETWORK_SHAPE=nodes, BIAS=bias), device=0)
    rng = np.random.RandomState(7 * sum(nodes) + envs + bias)
    n = 2
    x = (0.25 + 0.75 * rng.random_sample((n, envs, 6))).astype(np.float32)
    xd = torch.from_numpy(x).cuda()
    for rule, m, expect in _rules(nodes[-1]):
        genomes = _rule_genomes(rng, n, nodes, bias, rule, m)
        ref_out, ref_act = _oracle_rows(nodes, genomes, x, bias)
        assert np.all(ref_act == expect), (name, rule, m)
        if rule == "saturated":
            assert np.all(ref_out == 1.0), (name, "the action layer must saturate")
        g = torch.from_numpy(genomes).cuda()
        for route in ROUTES:
            act, out = _run_route(eng, route, g, xd)
            assert np.all(act.cpu().numpy() == expect), (name, rule, m, route, act.cpu().numpy())
            np.testing.assert_allclose(out.cpu().numpy(), ref_out, rtol=RTOL, atol=ATOL, err_msg=f"{name} {rule} {route}")
    eng.close()


# ---------------------------------------------------------------------------------------------------------------------------
# 1c. the fused rollout's generic MLP loop, bit for bit
# ---------------------------------------------------------------------------------------------------------------------------
SMALL_SHAPES = [(6, 2, 2), (6, 4, 3), (6, 32, 32, 2), (6, 1), (6, 8, 8, 8, 8, 8, 8, 5), (6, 3, 5)]


def _oracle_evaluate(args):
    import oracle
    nodes, genome, hof, hof_fit, pick, seed, gid, bias = args
    return oracle.evaluate(list(nodes), genome, hof, hof_fit, pick, seed=seed, genome_id=gid, bias=bias)


def _oracle_selfplay(args):
    import oracle
    nodes, right, left, seed, env_id, bias = args
    r = oracle.selfplay_game(list(nodes), right, left, seed=seed, env_id=env_id, bias=bias)
    return r.reward, r.frames


def _oracle_trace(args):
    """(reward, frames, left actions, right actions) of one self-play game from Start.2P, traced frame by frame"""
    import oracle
    nodes, right, left, seed, env_id, bias, cap = args
    env = oracle.Atari()
    env.reset_to_state(oracle.STATE_START_2P)
    res, tr = env.episode(oracle.Shape.make(list(nodes), bias), ("mlp", left), ("mlp", right), 1.0, seed, env_id=env_id, trace_cap=cap)
    return res.reward, res.frames, tr[:, 128].copy(), tr[:, 129].copy()


@pytest.mark.parametrize("bias", [True, False])
@pytest.mark.parametrize("nodes", SMALL_SHAPES, ids=["x".join(map(str, s)) for s in SMALL_SHAPES])
def test_fused_rollout_small_shapes(ngp, pool, nodes, bias):
    rng = np.random.RandomState(3 * sum(nodes) + bias)
    # reference schedule with a hall of fame: bots, the 1-player game and gathered opponents
    eng = ngp.Engine(ngp.Config(NETWORK_SHAPE=nodes, BIAS=bias), device=0)
    n = 2
    genomes = _genomes(rng, n, nodes, bias)
    hof = _genomes(rng, 3, nodes, bias); hof_fit = np.array([1.25, 0.5, -0.125])
    pick = rng.randint(0, 3, size=(n, 3)).astype(np.int32)
    ref_eval = pool.map(_oracle_evaluate, [(nodes, genomes[g], hof, hof_fit, pick[g], 4, g, bias) for g in range(n)])
    out = eng.evaluate(torch.from_numpy(genomes).cuda(), torch.from_numpy(hof).cuda(), torch.from_numpy(hof_fit).cuda(),
                       torch.from_numpy(pick).cuda(), seed=4, want_detail=True)
    for g, (fit, r, f) in enumerate(ref_eval):
        assert np.array_equal(out["frames"][g].cpu().numpy(), f), (g, out["frames"][g], f)
        assert np.array_equal(out["rewards"][g].cpu().numpy(), r), g
        assert out["fitness"][g].item() == fit
    eng.close()
    # round robin, and the same games as a recorded match list (key = the round-robin environment)
    n, games, seed, cap = 3, 2, 9, 12000
    eng = ngp.Engine(ngp.Config(NETWORK_SHAPE=nodes, BIAS=bias, SCHEDULE=ngp.SCHEDULE_ROUND_ROBIN, GAMES_TO_PLAY=games,
                                POPULATION_SIZE=n), device=0)
    genomes = _genomes(rng, n, nodes, bias)
    pairs = [(g, (g + k + 1) % n, g * games + k) for g in range(n) for k in range(games)]
    ref_sp = pool.map(_oracle_selfplay, [(nodes, genomes[r], genomes[l], seed, e, bias) for r, l, e in pairs])
    ref_tr = pool.map(_oracle_trace, [(nodes, genomes[r], genomes[l], seed, e, bias, cap) for r, l, e in pairs])
    gd = torch.from_numpy(genomes).cuda()
    out = eng.evaluate(gd, seed=seed, want_detail=True)
    ref_sp = list(ref_sp)
    assert np.array_equal(out["frames"].cpu().numpy().reshape(-1), [f for _, f in ref_sp])
    assert np.array_equal(out["rewards"].cpu().numpy().reshape(-1), [r for r, _ in ref_sp])
    right, left, key = (torch.tensor(c, dtype=torch.int32, device="cuda") for c in zip(*pairs))
    rm = eng.record_matches(gd, right, left, key=key, max_record=cap, seed=seed)
    frames = rm["frames"].cpu().numpy(); rewards = rm["rewards"].cpu().numpy(); act = rm["record"]["act"].cpu().numpy()
    for m, (rw, fr, la, ra) in enumerate(ref_tr):
        assert (rewards[m], frames[m]) == (rw, fr), m
        assert 0 < fr <= cap
        assert np.array_equal(act[m, :fr] & 3, la) and np.array_equal(act[m, :fr] >> 2, ra), m
    eng.close()


# ---------------------------------------------------------------------------------------------------------------------------
# 1d. the stepwise driver's tensor-core layers in whole episodes
# ---------------------------------------------------------------------------------------------------------------------------
def _oracle_episode(args):
    import oracle
    nodes, bias, right, left, seed, env_id, max_frames = args
    env = oracle.Atari()
    env.reset_to_state(oracle.STATE_START_2P)
    res, _ = env.episode(oracle.Shape.make(list(nodes), bias), ("mlp", left), ("mlp", right), 1.0, seed, env_id=env_id,
                         max_frames=max_frames)
    return res.reward, res.frames


# rows per genome and frame = 2 * games: 16 -> tmem<64>, 128 (BASELINE config 4) -> tmem<128>, 80 -> a ragged tmem<128> tile
@pytest.mark.parametrize("nodes,bias,n,games,kernel", [((6, 512, 512, 2), True, 3, 8, TM64), ((6, 512, 512, 2), True, 2, 64, TM128),
                                                       ((6, 128, 192, 2), False, 2, 40, TM128)])
def test_stepwise_tensor_core_episodes(ngp, pool, nodes, bias, n, games, kernel):
    seed, max_frames = 13, 300
    eng = ngp.Engine(ngp.Config(NETWORK_SHAPE=nodes, BIAS=bias, SCHEDULE=ngp.SCHEDULE_ROUND_ROBIN, GAMES_TO_PLAY=games,
                                POPULATION_SIZE=n, MAX_FRAMES=max_frames), device=0)
    rng = np.random.RandomState(sum(nodes) + games)
    genomes = _genomes(rng, n, nodes, bias)
    jobs = [(nodes, bias, genomes[g], genomes[(g + k + 1) % n], seed, g * games + k, max_frames) for g in range(n) for k in range(games)]
    ref = pool.map(_oracle_episode, jobs)
    out, names = _profiled(lambda: eng.evaluate(torch.from_numpy(genomes).cuda(), seed=seed, want_detail=True))
    assert any(alt in nm for alt in kernel for nm in names), (kernel[0], sorted(names))
    ref = list(ref)
    assert np.array_equal(out["frames"].cpu().numpy().reshape(-1), [f for _, f in ref]), (out["frames"], ref)
    assert np.array_equal(out["rewards"].cpu().numpy().reshape(-1), [r for r, _ in ref])
    eng.close()


# ---------------------------------------------------------------------------------------------------------------------------
# 1e. more than 65 535 genomes
# ---------------------------------------------------------------------------------------------------------------------------
BIG = 65537


def _device_genomes(n, nodes, seed):
    """n distinct genomes drawn on the device (no period that could line up with a 65 535-genome slice)"""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    parts = [torch.randn((n, (a + 1) * c), generator=gen, device="cuda") * (3.0 / np.sqrt(a + 1)) for a, c in zip(nodes[:-1], nodes[1:])]
    return torch.cat(parts, dim=1).contiguous()


def _np_forward(nodes, genomes, x):
    """vectorised FP64 restatement of the network with bias: genomes f32[n, G], x f32[n, envs, 6] -> sigmoid outputs f64"""
    h = x.astype(np.float64)
    off = 0
    for a, c in zip(nodes[:-1], nodes[1:]):
        W = genomes[:, off:off + (a + 1) * c].astype(np.float64).reshape(-1, c, a + 1)
        h = 1.0 / (1.0 + np.exp(-(np.matmul(h, W[:, :, :a].transpose(0, 2, 1)) + W[:, None, :, a])))
        off += (a + 1) * c
    return h


def _check_big(nodes, genomes, x, results, chunk=4096):
    """results: (act, out) pairs of one call each on all genomes, checked against the FP64 restatement and, on both sides of the
    first slice boundary, against the oracle"""
    import oracle
    n = genomes.shape[0]
    near = 0
    for g0 in range(0, n, chunk):
        ref = _np_forward(nodes, genomes[g0:g0 + chunk], x[g0:g0 + chunk])
        ref_act = np.where(np.argmax(ref, axis=-1) == 0, UP, DOWN)
        srt = np.sort(ref, axis=-1)
        clear = srt[..., -1] - srt[..., -2] > 1e-6      # decisions closer than that in FP64 are left to the oracle rows below
        near += int((~clear).sum())
        for act, out in results:
            np.testing.assert_allclose(out[g0:g0 + chunk], ref, rtol=RTOL, atol=ATOL, err_msg=f"genomes from {g0}")
            assert np.array_equal(act[g0:g0 + chunk][clear], ref_act[clear]), f"genomes from {g0}"
    assert near <= max(1, x.shape[0] * x.shape[1] // 10000), near
    for g in (0, 65533, 65534, 65535, 65536, n - 1):
        for e in range(x.shape[1]):
            o, a = oracle.mlp_forward(list(nodes), genomes[g], x[g, e].astype(np.float64))
            for act, out in results:
                np.testing.assert_allclose(out[g, e], o, rtol=RTOL, atol=ATOL, err_msg=f"genome {g} env {e}")
                assert act[g, e] == a, (g, e)


def test_mlp_forward_beyond_65535_genomes_one_env(ngp):
    nodes = (6, 40, 2)
    eng = ngp.Engine(ngp.Config(NETWORK_SHAPE=nodes), device=0)
    g = _device_genomes(BIG, nodes, 1)
    x = torch.rand((BIG, 1, 6), generator=torch.Generator(device="cuda").manual_seed(2), device="cuda")
    act, out = eng.mlp_forward(g, x)
    _check_big(nodes, g.cpu().numpy(), x.cpu().numpy(), [(act.cpu().numpy(), out.cpu().numpy())])
    eng.close()


def test_mlp_forward_beyond_65535_genomes_tensor_cores(ngp):
    """16 environments per genome: tcgen05 layers (plain and prepared), 65 537 genomes of [6,64,64,2] (about 1.3 GB)"""
    nodes = (6, 64, 64, 2)
    eng = ngp.Engine(ngp.Config(NETWORK_SHAPE=nodes), device=0)
    g = _device_genomes(BIG, nodes, 3)
    x = torch.rand((BIG, 16, 6), generator=torch.Generator(device="cuda").manual_seed(4), device="cuda")
    act, out = eng.mlp_forward(g, x)
    eng.mlp_prepare(g)
    act_p, out_p = eng.mlp_forward_prepared(g, x)
    _check_big(nodes, g.cpu().numpy(), x.cpu().numpy(), [(a.cpu().numpy(), o.cpu().numpy()) for a, o in ((act, out), (act_p, out_p))])
    eng.close()


def _oracle_reference_schedule(args):
    """ngp_evaluate's reference schedule for one genome, restated with a frame cap: game 1 is the 1-player cartridge-robot game,
    game 2 is against the score bot, games 3..5 against hall-of-fame members hof_pick with their fitness as multiplier"""
    import oracle
    nodes, genome, hof, hof_fit, pick, seed, gid, max_frames = args
    shape = oracle.Shape.make(list(nodes))
    env = oracle.Atari()
    out = []
    for i in range(6):
        left, mult = ("hardcoded", None), 1.0
        if i == 2:
            left = ("score", None)
        elif i >= 3:
            left, mult = ("mlp", hof[pick[i - 3]]), float(hof_fit[pick[i - 3]])
        env.reset_to_state(oracle.STATE_START_1P if i == 1 else oracle.STATE_START_2P)
        res, _ = env.episode(shape, left, ("mlp", genome), mult, seed, env_id=gid * 6 + i, max_frames=max_frames)
        out.append((res.reward, res.frames))
    return out


def test_evaluate_hall_of_fame_beyond_65535_opponent_rows(ngp, pool):
    """n = 21 846 genomes: 3n = 65 538 hall-of-fame rows, one batched MLP call per frame.  The first points fall before frame
    200, so the capped games' rewards depend on the decisions."""
    nodes, n, seed, max_frames = (6, 40, 2), 21846, 5, 200
    eng = ngp.Engine(ngp.Config(NETWORK_SHAPE=nodes, MAX_FRAMES=max_frames), device=0)
    rng = np.random.RandomState(11)
    genomes = _genomes(rng, n, nodes, True)
    hof = _genomes(rng, 3, nodes, True); hof_fit = np.array([0.75, 2.0, -0.5])
    pick = rng.randint(0, 3, size=(n, 3)).astype(np.int32)
    check = (0, n - 2, n - 1)           # genome n - 1's opponents are rows 65 535..65 537, across the first slice boundary
    ref = pool.map(_oracle_reference_schedule, [(nodes, genomes[g], hof, hof_fit, pick[g], seed, g, max_frames) for g in check])
    out = eng.evaluate(torch.from_numpy(genomes).cuda(), torch.from_numpy(hof).cuda(), torch.from_numpy(hof_fit).cuda(),
                       torch.from_numpy(pick).cuda(), seed=seed, want_detail=True)
    rewards, frames = out["rewards"].cpu().numpy(), out["frames"].cpu().numpy()
    assert frames.max() <= max_frames
    for g, r in zip(check, ref):
        assert np.array_equal(frames[g], [f for _, f in r]), (g, frames[g], r)
        assert np.array_equal(rewards[g], [w for w, _ in r]), g
    eng.close()
