"""Per-handle scratch memory: a refused allocation leaves the handle usable, and buffers that grew or are reused for a smaller
request give the same bits as a freshly created handle."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

SNAPSHOT_BYTES = 352            # sizeof(a26::Snapshot): one stepwise environment's state


@pytest.fixture(scope="module")
def ngp():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import neuro_genetic_pong_self_play_b200 as m
    return m


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _fresh(ngp, cfg, call, options=()):
    """`call` on a newly created handle."""
    eng = ngp.Engine(cfg, device=0)
    try:
        for name, value in options:
            eng.set_option(name, value)
        return call(eng)
    finally:
        eng.close()


def test_refused_allocation_leaves_handle_usable(ngp):
    """A request the runtime refuses (twice the device's memory) is an ordinary error return; the runtime's error state does not
    leak into the next call, and the handle keeps working."""
    cfg = ngp.Config()
    eng = ngp.Engine(cfg, device=0)
    n = 2 * torch.cuda.get_device_properties(0).total_memory // SNAPSHOT_BYTES + 1
    assert n < 2 ** 31
    with pytest.raises(ngp.NgpError):
        eng.env_reset(n)
    actions = torch.tensor([cfg.blank_action()] * 64, dtype=torch.uint8, device="cuda")

    def step(e):
        e.env_reset(64)
        return e.env_step(actions)["ram"].cpu()

    genomes = _cuda((np.random.RandomState(1).random_sample((4, eng.gene_size)) * 4 - 2).astype(np.float32))

    def evaluate(e):
        return e.evaluate(genomes, seed=3)["fitness"].cpu()

    assert torch.equal(step(eng), _fresh(ngp, cfg, step))
    assert torch.equal(evaluate(eng), _fresh(ngp, cfg, evaluate))
    eng.close()


def test_grown_and_reused_buffers_match_a_fresh_handle(ngp):
    rng = np.random.RandomState(7)

    # ngp_mlp_forward on a wide net: activation buffers grow with the environments per genome, then serve a smaller call
    cfg = ngp.Config(NETWORK_SHAPE=(6, 512, 512, 2))
    eng = ngp.Engine(cfg, device=0)
    genomes = _cuda((rng.standard_normal((3, eng.gene_size)) * 0.05).astype(np.float32))
    for envs in (16, 64, 16):
        x = _cuda(rng.random_sample((3, envs, 6)).astype(np.float32))
        act, out = eng.mlp_forward(genomes, x)
        act_f, out_f = _fresh(ngp, cfg, lambda e: e.mlp_forward(genomes, x))
        assert torch.equal(act, act_f) and torch.equal(out, out_f), envs
    eng.close()

    # ngp_evaluate with the handle's own reward and frame buffers
    cfg = ngp.Config()
    eng = ngp.Engine(cfg, device=0)
    for n in (8, 64, 8):
        g = _cuda((rng.random_sample((n, eng.gene_size)) * 4 - 2).astype(np.float32))
        a = eng.evaluate(g, seed=n)
        b = _fresh(ngp, cfg, lambda e: e.evaluate(g, seed=n))
        assert torch.equal(a["fitness"], b["fitness"]) and a["frames_total"] == b["frames_total"], n
    eng.close()

    # ngp_hof_update: the hall grows from 4 to 32 members, its members carried over
    cfg = ngp.Config()
    eng = ngp.Engine(cfg, device=0)
    G = eng.gene_size
    members, n_hof = np.zeros((0, G), np.float32), 0
    member_fit = np.zeros(0)
    for maxsize in (4, 16, 32):
        hg = np.zeros((maxsize, G), np.float32); hf = np.zeros(maxsize)
        hg[:n_hof] = members; hf[:n_hof] = member_fit
        pop = _cuda(rng.random_sample((48, G)).astype(np.float32))
        fit = _cuda(np.round(rng.standard_normal(48), 1))

        def update(e):
            hg_d, hf_d = _cuda(hg), _cuda(hf)
            count = e.hof_update(hg_d, hf_d, n_hof, pop, fit)
            return count, hg_d.cpu(), hf_d.cpu()

        (count, hg_a, hf_a), (count_f, hg_f, hf_f) = update(eng), _fresh(ngp, cfg, update)
        assert count == count_f and torch.equal(hg_a, hg_f) and torch.equal(hf_a, hf_f), maxsize
        members, member_fit, n_hof = hg_a[:count].numpy(), hf_a[:count].numpy(), count
    assert n_hof == 32
    eng.close()

    # ngp_ga_step through the order-statistics selection; its ranking buffers hold max(2048, next power of two >= n) entries,
    # so 4096 is where they grow
    cfg = ngp.Config(POPULATION_SIZE=1024)
    options = (("select_os_min_t", 16),)
    eng = ngp.Engine(cfg, device=0)
    for name, value in options:
        eng.set_option(name, value)
    for n in (64, 1024, 4096, 64):
        g = _cuda(rng.random_sample((n, eng.gene_size)).astype(np.float32))
        fit = _cuda(np.round(rng.standard_normal(n), 1))
        a = eng.ga_step(g, fit, seed=5, generation=n)
        b = _fresh(ngp, cfg, lambda e: e.ga_step(g, fit, seed=5, generation=n), options)
        for k in ("genomes", "parent_idx", "invalid", "stats"):
            assert torch.equal(a[k], b[k]), (n, k)
    eng.close()
