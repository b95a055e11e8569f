#!/usr/bin/env python3
"""bench.py -- headline benchmark: Pong self-play env-frames/s including both players' NN forward.

  python bench.py --gpus N --steps K --warmup W [--config {1,2,3,4,5}]      (N>1: launched under torch.distributed.run)
  python bench.py --impl reference --gpus N --steps K --warmup W [--config ..]
  python bench.py ... --dump-outputs DIR       (configs 1-4: also write what the last timed step computed as DIR/<name>.npy)

A "step" is one generation of the rank's population shard: the fused evaluation (emulator + observation + both players'
MLP + episode control for every game), the per-generation exchange (one record all-gather, issued asynchronously and
consumed a generation later; only when N>1) and the GA step that breeds the next generation's genomes.

--config selects the BASELINE.json workload (default 2, the one the metric is quoted on):
  1  main.py defaults from config.py: population 64, reference opponent schedule (bot, cartridge robot, score bot,
     3 x hall of fame), [6,2,2], hall-of-fame update every generation
  2  population 1024 per GPU, round-robin self-play (genome i vs i+1..i+6 inside the shard), [6,2,2]       (weak scaling)
  3  population 16384 sharded over the N GPUs (2048 per GPU at N=8), round-robin, exchange every generation (strong scaling)
  4  [6,512,512,2] with 64 environments per genome (round-robin against 64 opponents): per-frame stepwise driver, wide layers
     on the tcgen05 path
  5  NN forward + GA only on synthetic obs.npy-shaped inputs, population sweep 2^10 .. 2^20
The default run (config 2) also attaches short measurements of the other configurations under "configs".
Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GAMES = 6
FRAME_6507_INSTR = 6740          # 6507 instructions per emulated frame of this cartridge (oracle count)
METRIC = "pong_selfplay_env_frames_per_sec_incl_nn_forward"
SEED_POP, SEED_RUN = 1234, 99


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ngp", choices=["ngp", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[1, 2, 3, 4, 5])
    ap.add_argument("--population", type=int, default=0, help="genomes per GPU (configs 2, 4) / in total (configs 1, 3); 0 = the config's own")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of each cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the saturated-GPU context run and the other configs' short runs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the arrays the last timed generation returned (rank 0's shard) as "
                    "DIR/<name>.npy, at most 64 MB in all, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.impl == "reference" or args.config == 5):
        ap.error("--dump-outputs needs the generation loop of configs 1-4 on the GPU")
    return args


def workload(config: int, world: int, population: int):
    """(description, nodes, schedule name, games per genome, genomes per GPU, genomes in total, scaling)"""
    if config == 1:
        n = population or 64
        return dict(name=f"config 1: main.py defaults, population {n}, reference schedule (bot, robot, score bot, 3 x hall of fame), [6,2,2]",
                    nodes=(6, 2, 2), schedule="reference", games=6, n_total=n, scaling="strong")
    if config == 3:
        n = population or 16384
        return dict(name=f"config 3: population {n} sharded over {world} GPU(s), round-robin self-play, [6,2,2], 6 games/genome",
                    nodes=(6, 2, 2), schedule="round_robin", games=6, n_total=n, scaling="strong")
    if config == 4:
        n = population or 256
        return dict(name=f"config 4: [6,512,512,2] MLP, 64 environments per genome (round-robin vs 64 opponents), population {n}/GPU",
                    nodes=(6, 512, 512, 2), schedule="round_robin", games=64, n_total=n * world, scaling="weak")
    n = population or 1024
    return dict(name=f"population {n}/GPU round-robin self-play, [6,2,2] sigmoid MLP, {GAMES} games/genome = {n * GAMES} envs/GPU",
                nodes=(6, 2, 2), schedule="round_robin", games=6, n_total=n * world, scaling="weak")


# ---------------------------------------------------------------------------------------------------
# CPU arms: (a) the C oracle port of the whole path, (b) the reference's numpy path on the port's emulator
# ---------------------------------------------------------------------------------------------------
def _cpu_port_worker(args):
    import numpy as np
    import oracle
    worker, workers, budget_s, wl = args
    nodes, games, n = list(wl["nodes"]), wl["games"], wl["n_shard"]
    G = sum((a + 1) * b for a, b in zip(nodes[:-1], nodes[1:]))
    pop = oracle.init_population_philox(n, G, SEED_POP)              # generation 0 of the GPU arm's rank 0, same genomes
    frames = played = 0
    t0 = time.perf_counter()
    e = worker
    while time.perf_counter() - t0 < budget_s and e < n * games:
        g, k = divmod(e, games)
        if wl["schedule"] == "round_robin":
            res = oracle.selfplay_game(nodes, pop[g], pop[(g + k + 1) % n], seed=SEED_RUN, env_id=e, generation=0)
            frames += res.frames
        else:                                                        # generation 0 of the reference schedule: no hall of fame yet
            _, _, fr = oracle.evaluate(nodes, pop[g], None, None, (0, 0, 0), seed=SEED_RUN, genome_id=g, generation=0)
            frames += int(fr.sum()); e += games - 1
        played += 1
        e += workers
    return frames, played, time.perf_counter() - t0


def _cpu_numpy_worker(args):
    import numpy as np
    import oracle
    from oracle import numpy_path as npp
    worker, workers, budget_s, wl = args
    nodes, games, n = list(wl["nodes"]), wl["games"], wl["n_shard"]
    G = sum((a + 1) * b for a, b in zip(nodes[:-1], nodes[1:]))
    pop = oracle.init_population_philox(n, G, SEED_POP)
    frames = played = 0
    t0 = time.perf_counter()
    e = worker
    emu = oracle.Atari()
    while time.perf_counter() - t0 < budget_s and e < n * games:
        g, k = divmod(e, games)
        emu.reset_to_state(oracle.STATE_START_2P)
        left = npp.NeuralNetwork(nodes, pop[(g + k + 1) % n].tolist()) if wl["schedule"] == "round_robin" else npp.HardcodedAi()
        right = npp.NeuralNetwork(nodes, pop[g].tolist())
        left_budget = max(1, int(3000 * (budget_s - (time.perf_counter() - t0)) / 10))
        steps, _ = npp.perform_episode(emu, left, right, max_frames=left_budget)
        frames += steps; played += 1
        e += workers
    return frames, played, time.perf_counter() - t0


def cpu_baseline(budget_s: float, wl: dict, kind: str = "port"):
    import concurrent.futures as cf
    import oracle
    oracle.build()
    cores = os.cpu_count() or 1
    fn = _cpu_port_worker if kind == "port" else _cpu_numpy_worker
    t0 = time.perf_counter()
    with cf.ProcessPoolExecutor(max_workers=cores) as ex:
        res = list(ex.map(fn, [(i, cores, budget_s, wl) for i in range(cores)]))
    wall = time.perf_counter() - t0
    frames = sum(r[0] for r in res); games = sum(r[1] for r in res); longest = max(r[2] for r in res)
    what = ("C oracle port of the whole path (per-colour-clock TIA emulator, find_stuff, MLP, episode control)" if kind == "port" else
            "the reference's numpy path (utils.find_stuff: full-frame compare + argwhere + average per colour; numpy_nn.run; get_actions; "
            "perform_episode) restated call for call in oracle/numpy_path.py, on frames from the C oracle emulator standing in for gym-retro's env.step")
    return {"value": frames / longest, "unit": "env-frames/s", "cores": cores, "kind": "port" if kind == "port" else "reference-numpy+port-emulator",
            "sample": f"{games} games ({frames} frames) of generation 0 of this workload (same Philox genomes and pairings as the GPU arm's rank 0) "
                      f"on {cores} processes, {wall:.1f}s wall; {what}; gym-retro/Stella, DEAP and SCOOP cannot be installed here (no network)"}


def run_reference(args):
    """Reference arm: the reference's CPU implementation of the path on the box's host cores = the oracle port (gym-retro,
    DEAP and SCOOP are absent from the image and cannot be installed offline), all host cores, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cfg_id = 2 if args.config in (4, 5) else args.config             # the port's MLP is the small-net path; 4/5 have no CPU arm of their own
    wl = workload(cfg_id, world, args.population)
    wl["n_shard"] = max(1, wl["n_total"] // world)
    per_step = max(2.0, min(20.0, 60.0 / max(1, args.steps + args.warmup)))
    vals, last = [], None
    for i in range(args.warmup + args.steps):
        last = cpu_baseline(per_step, wl)
        if i >= args.warmup:
            vals.append(last["value"])
    value = sum(vals) / len(vals)
    last["value"] = value
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "env-frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_step * 1e3, "higher_is_better": True,
        "scaling": wl["scaling"], "vs_baseline": None, "dtype": "u8+f64", "data": "synthetic",
        "config": {"workload": wl["name"] + " (bounded sample per step)"},
        "cpu_baseline": last, "e2e": {"value": value, "unit": "env-frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._halt = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                parts = [p.strip() for p in out.split(",")]
                self.samples.append(float(parts[0])); self.max_mhz = float(parts[1])
                for n, v in zip(names, parts[2:]):
                    if v.lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=3)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


# ---------------------------------------------------------------------------------------------------
# the generation loop both the device-timed and the end-to-end measurements walk
# ---------------------------------------------------------------------------------------------------
class Generation:
    """One rank's population shard + everything a generation needs (engine, hall of fame, exchange)."""

    def __init__(self, ngp, wl, world, rank, local):
        import torch
        from neuro_genetic_pong_self_play_b200 import parallel
        from neuro_genetic_pong_self_play_b200.reference_api import HallOfFame
        self.torch, self.wl, self.world, self.rank = torch, wl, world, rank
        n_total = wl["n_total"]
        self.lo, self.hi = parallel.shard_bounds(n_total, world, rank)
        self.n = self.hi - self.lo
        schedule = ngp.SCHEDULE_ROUND_ROBIN if wl["schedule"] == "round_robin" else ngp.SCHEDULE_REFERENCE
        # TOURNAMENT_SIZE = POPULATION_SIZE // 4 of the population selection runs over = the shard (island model, DESIGN.md section 6)
        self.cfg = ngp.Config(SCHEDULE=schedule, POPULATION_SIZE=self.n, GAMES_TO_PLAY=wl["games"], NETWORK_SHAPE=tuple(wl["nodes"]))
        self.eng = ngp.Engine(self.cfg, device=local)
        self.G = self.eng.gene_size
        self.hof = HallOfFame(max(1, n_total // 4) if wl["schedule"] == "reference" else 0, self.eng)
        # multi-GPU: the hall of fame is fed the merged elites of all ranks (k_total of them per generation)
        self.k_total = min(n_total // 4, 64 * world) if world > 1 else 0
        self.exchange = parallel.Exchange(self.eng, n_total, self.k_total) if world > 1 else None
        if world > 1 and self.hof.maxsize == 0:
            self.hof = HallOfFame(self.k_total, self.eng)            # global elites (round-robin runs do not play against them)
        self.reset()

    def reset(self):
        # every rank draws ITS shard from the one population stream: identically distributed shards, the global population
        # does not depend on the number of ranks (rank r = rows lo..hi of the population Philox(SEED_POP) generates)
        self.genomes = self.eng.init_population(self.hi, seed=SEED_POP)[self.lo:].contiguous() if self.world > 1 else \
            self.eng.init_population(self.n, seed=SEED_POP)
        self.gen = 0
        self.hof.clear()
        if self.exchange is not None and self.exchange.pending:
            self.exchange.finish()

    def step(self, genomes=None):
        """evaluate -> (exchange | hall of fame) -> breed.  Returns the device tensor of per-game frame counts."""
        eng, gen = self.eng, self.gen
        g = self.genomes if genomes is None else genomes
        hg, hf = self.hof.tensors() if self.wl["schedule"] == "reference" else (None, None)
        out = eng.evaluate(g, hg, hf, seed=SEED_RUN, generation=gen, sync=False, want_detail=True)
        fitness = out["fitness"]
        if self.exchange is not None:
            if self.exchange.pending:                                # generation gen-1's record: merged elites -> hall of fame
                _, eg, ef = self.exchange.finish()
                self.hof.update(eg, ef)
            self.exchange.start(g, fitness)
        elif self.hof.maxsize:
            self.hof.update(g, fitness)
        nxt = eng.ga_step(g, fitness, seed=SEED_RUN, generation=gen)
        self.genomes = nxt["genomes"]
        self.fitness = fitness
        self.last = (out, nxt)
        self.gen += 1
        return out["frames"]

    def close(self):
        if self.exchange is not None and self.exchange.pending:
            self.exchange.finish()
        self.eng.close()


def timed_generations(gen: Generation, steps: int, warmup: int, dist, sampler=None):
    """Device-timed K generations after W warm-up generations.  Returns (ms, frames, rollout_ms, launches) of this rank."""
    torch = gen.torch
    gen.reset()
    for _ in range(warmup):
        gen.step()
    torch.cuda.synchronize()
    gen.eng.profile_enable(True)
    gen.eng.profile_read()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    if sampler:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches_before = gen.eng.launches
    ev0.record()
    frames_steps = [gen.step() for _ in range(steps)]
    ev1.record()
    launches = gen.eng.launches - launches_before
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    ms = ev0.elapsed_time(ev1)
    frames = int(sum(int(t.sum().item()) for t in frames_steps))     # summed after the timed region
    rollout_ms, _ = gen.eng.profile_read()                           # CUDA-event time of the dominant kernel inside the timed region
    gen.eng.profile_enable(False)
    return ms, frames, rollout_ms, launches


DUMP_POPULATION_BYTES, DUMP_HOF_BYTES = 40 << 20, 16 << 20          # with the .npy headers well under 64 MB in all


def _dump_rows(n: int, row_bytes: int, budget: int):
    """All n rows, or a fixed seeded sample of them (ascending) when they do not fit in `budget` bytes."""
    import numpy as np
    k = min(n, max(1, budget // row_bytes))
    return np.arange(n) if k == n else np.sort(np.random.RandomState(0).choice(n, k, replace=False))


def dump_outputs(gen: Generation, directory: str):
    """What the last generation handed back -- evaluate (fitness, per-game rewards and frame counts), the GA step (next
    genomes, parents, invalid flags, fitness statistics) and the hall of fame it updated -- as DIR/<name>.npy: genomes in
    float32, everything else in float64 (integers exactly).  Per-genome arrays keep the rows in population_rows.npy (all of
    them unless a wide net's genomes would pass the size budget), hall-of-fame arrays those in hof_rows.npy."""
    import numpy as np
    torch = gen.torch
    out, nxt = gen.last
    groups = [("population", DUMP_POPULATION_BYTES, {"fitness": out["fitness"], "rewards": out["rewards"], "frames": out["frames"],
                                                     "genomes": nxt["genomes"], "parent_idx": nxt["parent_idx"], "invalid": nxt["invalid"]})]
    hg, hf = gen.hof.tensors()
    if hf is not None:
        groups.append(("hof", DUMP_HOF_BYTES, {"hof_fitness": hf, "hof_genomes": hg}))
    arrays = {"ga_stats": nxt["stats"]}
    for name, budget, group in groups:
        n = next(iter(group.values())).shape[0]
        row_bytes = 8 + sum((4 if t.dtype == torch.float32 else 8) * (t.numel() // n) for t in group.values())
        rows = _dump_rows(n, row_bytes, budget)
        idx = torch.from_numpy(rows).to(gen.eng.device)
        arrays[name + "_rows"] = rows
        arrays.update({k: t.index_select(0, idx) for k, t in group.items()})
    os.makedirs(directory, exist_ok=True)
    for k, a in arrays.items():
        a = a.cpu().numpy() if isinstance(a, torch.Tensor) else a
        np.save(os.path.join(directory, k + ".npy"), a.astype(np.float32 if a.dtype == np.float32 else np.float64))


def e2e_generations(gen: Generation, steps: int, warmup: int, dist):
    """The same generations (same initial population, same seeds => the same games as the device-timed run) through HOST
    buffers: every step copies the genomes host->device from pinned memory, evaluates, breeds, and reads fitness and the next
    generation's genomes back to the host.  Wall clock around the K steps."""
    torch = gen.torch
    gen.reset()
    host = torch.empty((gen.n, gen.G), dtype=torch.float32).pin_memory()
    host_fit = torch.empty(gen.n, dtype=torch.float64).pin_memory()
    host_frames = torch.empty((gen.n, gen.wl["games"]), dtype=torch.int32).pin_memory()
    host.copy_(gen.genomes)
    dev = torch.empty_like(gen.genomes)
    frames = 0

    def one():
        dev.copy_(host, non_blocking=True)                           # H2D: this generation's genomes
        fr = gen.step(dev)
        host.copy_(gen.genomes, non_blocking=True)                   # D2H: next generation
        host_fit.copy_(gen.fitness, non_blocking=True)               # D2H: fitness
        host_frames.copy_(fr, non_blocking=True)
        # the step's results are on the host once THIS stream is done; the record exchange of the generation runs on its side
        # stream and is consumed a generation later (a device-wide synchronize here would make every rank wait for the slowest
        # rank's generation in every step, which the exchange was made asynchronous to avoid)
        torch.cuda.current_stream().synchronize()
        return int(host_frames.sum().item())

    for _ in range(warmup):
        one()
    if dist is not None:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        frames += one()
    s = time.perf_counter() - t0
    h2d = gen.n * gen.G * 4
    d2h = gen.n * gen.G * 4 + gen.n * 8 + gen.n * gen.wl["games"] * 4
    return s, frames, h2d, d2h


def reduce_ranks(torch, dist, world, maxed, summed):
    if world == 1:
        return maxed, summed
    a = torch.tensor(maxed, dtype=torch.float64, device="cuda"); dist.all_reduce(a, op=dist.ReduceOp.MAX)
    b = torch.tensor(summed, dtype=torch.float64, device="cuda"); dist.all_reduce(b, op=dist.ReduceOp.SUM)
    return a.tolist(), b.tolist()


# ---------------------------------------------------------------------------------------------------
# config 5: NN forward + GA only
# ---------------------------------------------------------------------------------------------------
def config5_sweep(ngp, local, world, dist, sizes=None, envs=6, reps=5, warmup=2):
    """Policy forward on synthetic obs.npy-shaped inputs (6 observation values per environment, `envs` environments per
    genome) + one GA step (fitness statistics, tournament selection, blend crossover, Gaussian mutation), per population
    size; the population is sharded over the ranks like every other config.  Device-timed (CUDA events), max over ranks."""
    import torch
    rows = []
    sizes = sizes or [2 ** k for k in range(10, 21, 2)]
    for n_total in sizes:
        n = n_total // world
        cfg = ngp.Config(SCHEDULE=ngp.SCHEDULE_ROUND_ROBIN, POPULATION_SIZE=n)
        eng = ngp.Engine(cfg, device=local)
        genomes = eng.init_population(n, seed=5)
        x = torch.rand((n, envs, 6), dtype=torch.float32, device=eng.device)
        fitness = torch.rand(n, dtype=torch.float64, device=eng.device)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        t_f = t_g = 0.0
        for r in range(reps + warmup):
            ev[0].record()
            eng.mlp_forward(genomes, x, want_out=False)
            ev[1].record()
            nxt = eng.ga_step(genomes, fitness, seed=7, generation=r)
            ev[2].record()
            torch.cuda.synchronize()
            if r >= warmup:
                t_f += ev[0].elapsed_time(ev[1]); t_g += ev[1].elapsed_time(ev[2])
            genomes = nxt["genomes"]
        (mf, mg), _ = reduce_ranks(torch, dist, world, [t_f / reps, t_g / reps], [0.0])
        rows.append({"population": n_total, "forward_ms": mf, "ga_step_ms": mg, "policy_forwards_per_s": n_total * envs / (mf * 1e-3),
                     "ga_genomes_per_s": n_total / (mg * 1e-3)})
        eng.close()
        del genomes, x, fitness, nxt
    return rows


# ---------------------------------------------------------------------------------------------------
# main arm
# ---------------------------------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    import torch
    import torch.distributed as dist

    import neuro_genetic_pong_self_play_b200 as ngp

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    D = dist if world > 1 else None
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass

    if args.config == 5:
        rows = config5_sweep(ngp, local, world, D, reps=args.steps, warmup=args.warmup)
        if rank == 0:
            top = rows[-1]
            print(json.dumps({"metric": "policy_forwards_per_sec_plus_ga", "value": top["policy_forwards_per_s"], "unit": "forwards/s", "n_gpus": world,
                              "steps": args.steps, "warmup": args.warmup, "ms_per_step": top["forward_ms"] + top["ga_step_ms"], "higher_is_better": True, "scaling": "strong",
                              "vs_baseline": None, "dtype": "f32 (hidden layers) + f64 (action layer)", "data": "synthetic",
                              "config": {"workload": "config 5: NN forward + GA only on synthetic obs.npy-shaped inputs, population sweep"}, "sweep": rows}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    wl = workload(args.config, world, args.population)
    gen = Generation(ngp, wl, world, rank, local)
    n, G, games = gen.n, gen.G, wl["games"]
    sampler = ClockSampler(local) if rank == 0 else None
    ms, frames, rollout_ms, launches = timed_generations(gen, args.steps, args.warmup, D, sampler)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(gen, args.dump_outputs)
    (ms, rollout_ms), (frames,) = reduce_ranks(torch, dist, world, [ms, rollout_ms], [float(frames)])
    e2e_s, e2e_frames, h2d, d2h = e2e_generations(gen, args.steps, args.warmup, D)
    (e2e_s,), (e2e_frames,) = reduce_ranks(torch, dist, world, [e2e_s], [float(e2e_frames)])
    line = None
    if rank == 0:
        value = frames / (ms * 1e-3)
        sm_mhz = (clocks or {}).get("sm_mhz") or peaks.get("sm_max_mhz", 1965.0)
        sm_count = torch.cuda.get_device_properties(local).multi_processor_count
        # issue roofline of the dominant kernel: thread-instructions the emulated frames need at full lane convergence
        # (ncu-measured per frame) against what the chip can issue
        prof = {}
        try:
            prof = json.load(open(os.path.join(ROOT, "profiles", "rollout_issue_model.json")))
        except Exception:
            pass
        frames_rank0 = frames / world
        kernel_s = rollout_ms * 1e-3
        tipf = prof.get("thread_inst_per_env_frame")
        issue_peak = sm_count * 4 * 32 * sm_mhz * 1e6
        achieved = frames_rank0 * tipf / kernel_s if (tipf and kernel_s > 0) else None
        hbm_alg = n * G * 4 + n * games * 12 + n * 8                                # genomes in, rewards/frames/fitness out
        roofline = {
            "bound": "issue",          # neither "hbm" nor "tensor" binds: per-env state is on-chip, no GEMM in the 6507/TIA core
            "kernel": "rollout_kernel<1> (fused emulator + observation + policy + episode control)",
            "achieved": achieved / 1e9 if achieved else None, "peak": issue_peak / 1e9, "unit": "G thread-inst/s",
            "frac": achieved / issue_peak if achieved else None,
            "traffic": prof.get("dram_bytes_per_launch"),
            "algorithmic_unit": "thread-instructions per env-frame at full lane convergence, from ncu: %s" % prof.get("source"),
            "thread_inst_per_env_frame": tipf, "emulated_6507_inst_per_s": frames_rank0 * FRAME_6507_INSTR / kernel_s if kernel_s > 0 else None,
            "kernel_ms_per_launch": rollout_ms / max(1, args.steps),
            "hbm": {"algorithmic_bytes_per_launch": hbm_alg, "achieved_gbs": hbm_alg * args.steps / kernel_s / 1e9 if kernel_s > 0 else None,
                    "peak_gbs": peaks.get("hbm_gbs", 6650.0), "peak_source": "measured" if peaks else "fallback"},
            "sm_clock_mhz_used": sm_mhz,
        }
        line = {
            "metric": METRIC, "value": value, "unit": "env-frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": wl["scaling"],
            "vs_baseline": None, "dtype": "u8 (6507/TIA integer) + f64 (policy MLP, reward)", "data": "synthetic",
            "config": {"workload": wl["name"], "parallelism": f"population sharded over {world} GPU(s), intra-shard pairings, "
                       "one asynchronous record all-gather per generation" if world > 1 else "1 GPU",
                       "l2": "per-env state on-chip; inputs (genomes) %d KB" % (n * G * 4 // 1024)},
            "frames_per_step": frames / args.steps, "generations_per_hour": 3600.0 / (ms * 1e-3 / args.steps),
            "e2e": {"value": e2e_frames / e2e_s, "unit": "env-frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "what": "the same generations (same population, seeds, games) with genomes copied H2D from pinned memory and fitness + next "
                            "generation + frame counts copied D2H every step; wall clock"},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
        }
    gen.close()
    extras = args.config == 2 and not args.no_extras
    if rank == 0 and not args.no_cpu_baseline and world == 1 and wl["nodes"] == (6, 2, 2):
        wlc = dict(wl, n_shard=n)
        line["cpu_baseline"] = cpu_baseline(args.cpu_seconds, wlc)
        if extras:
            line["cpu_baseline_numpy"] = cpu_baseline(args.cpu_seconds, wlc, kind="numpy")
    if extras:
        configs = {}

        def short(config, steps, warmup, population=0):
            w = workload(config, world, population)
            g2 = Generation(ngp, w, world, rank, local)
            m, f, r, _ = timed_generations(g2, steps, warmup, D)
            (m, r), (f,) = reduce_ranks(torch, dist, world, [m, r], [float(f)])
            g2.close()
            # per-generation breakdown (SURVEY 8d, config 3): the rollout kernel on its own CUDA events; what is left of the step is
            # the GA step, the hall-of-fame update and whatever the rank waits for the record exchange (NCCL, asynchronous)
            return {"workload": w["name"], "env_frames_per_s": f / (m * 1e-3), "ms_per_step": m / steps, "rollout_ms_per_step": r / steps,
                    "ga_hof_exchange_ms_per_step": max(0.0, (m - r) / steps) if r > 0 else None,       # None: the per-frame driver has no single rollout kernel
                    "frames_per_step": f / steps, "steps": steps, "warmup": warmup, "scaling": w["scaling"]}

        def lockstep():
            """Throughput capability of the fused kernel with every lane busy: 32 768 genomes per GPU (196 608 environments), every
            episode capped at 300 frames (MAX_FRAMES), so no lane waits for a marathon rally.  NOT the GA workload (episodes are
            cut short): context for north_star's >= 1e9 frames/s target."""
            n2 = 32768
            cfg2 = ngp.Config(SCHEDULE=ngp.SCHEDULE_ROUND_ROBIN, POPULATION_SIZE=n2, GAMES_TO_PLAY=GAMES, MAX_FRAMES=300)
            e2 = ngp.Engine(cfg2, device=local)
            g2 = e2.init_population(n2, seed=SEED_POP + rank)
            e2.evaluate(g2, seed=5)
            e2.profile_enable(True); e2.profile_read()
            total = 0
            for rep in range(2):
                total += e2.evaluate(g2, seed=6 + rep)["frames_total"]
            ms2, _ = e2.profile_read()
            e2.close()
            (ms2,), (total,) = reduce_ranks(torch, dist, world, [ms2], [float(total)])
            return {"workload": f"{n2} genomes/GPU round-robin, {n2 * GAMES} envs/GPU, episodes capped at 300 frames (lock-step regime, not the GA workload)",
                    "env_frames_per_s": total / (ms2 * 1e-3), "kernel_ms": ms2 / 2, "n_gpus": world}

        for name, fn in (("config1", lambda: short(1, 3, 1)),
                         ("lockstep_capability", lockstep),
                         ("config3", lambda: short(3, 2, 1)),
                         # the GA workload with every resident lane busy from the first frame: 12 288 genomes x 6 games = 73 728
                         # environments per GPU, one wave of the 148 x 512 lanes of the CTA-synchronous flavour (full episodes, GA
                         # step and exchange included) -- north_star's >= 1e9 frames/s target on 8 GPUs without capping episodes
                         ("ga_large_population", lambda: short(2, 2, 1, population=12288)),
                         ("config4", lambda: short(4, 1, 1)),
                         ("config5", lambda: config5_sweep(ngp, local, world, D))):
            try:
                configs[name] = fn()
            except Exception as e:      # never lose the headline line over a context measurement
                configs[name] = {"error": str(e)[:300]}
        if rank == 0:
            line["configs"] = configs
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
