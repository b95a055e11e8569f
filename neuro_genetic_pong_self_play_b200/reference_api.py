"""The reference's call surface, batched underneath (SURVEY section 8b).

Names and argument meaning follow the reference so its call sites read the same:
  NeuralNetwork(nodes, weights=..., bias=...).run(vec6)        numpy_nn.py:35-50, 120-137
  find_stuff(observation)                                      utils.py:14-19
  toolbox.evaluate(individual) -> (fitness,)                   main.py:28-66
  toolbox.map / select / mate / mutate / clone / population    ga.py:83-94
  HallOfFame(maxsize).update(population)                       ga.py:78 (DEAP tools.HallOfFame)
  run_generations(...)  (eaSimple-shaped loop + logbook)       main.py:157-173
  save_checkpoint / load_latest_population                     utils.py:116-125, ga.py:13-53
  replay(individual) / repeat_upsample                         pickle_inspector.py:1-12, main.py:115-125, utils.py:156-168
  cross_play(toolbox, a, b)                                    no counterpart: main.evaluate's schedule as any match list
  render_recorded / replay_selfplay                            main.evaluate(render=True) for recorded games
  play_policy / model_policy                                   perform_episode with any model object (main.py:69-112,
                                                               play_against_human.py): outside policies in a match list
Every call lands in libngp.so's CUDA kernels through Engine; nothing here computes on the CPU except argument
marshalling (individuals are rows of device tensors instead of Python lists)."""
from __future__ import annotations

import glob
import os
import time
import warnings
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from .config import Config
from .engine import Engine

_engines = {}


def get_engine(config: Config | None = None, device: int | None = None) -> Engine:
    config = config or Config()
    key = (config, torch.cuda.current_device() if device is None else device)
    if key not in _engines:
        _engines[key] = Engine(config, device)
    return _engines[key]


class NeuralNetwork:
    """numpy_nn.NeuralNetwork's inference surface (training is out of scope)."""

    def __init__(self, nodes: Sequence[int], learning_rate=0.1, bias=None, weights=None, engine: Engine | None = None):
        if weights is None:
            raise _lib.NgpError("random weight initialisation (numpy_nn.py:71-82) is outside the GA path; pass weights")
        self.nodes = list(nodes)
        self.bias = 1 if bias else 0
        cfg = Config(NETWORK_SHAPE=tuple(self.nodes), BIAS=bool(bias))
        self._eng = engine or get_engine(cfg)
        g = np.asarray(weights, np.float32)
        need = cfg.gene_size()
        if len(g) < need:
            raise ValueError(f"need {need} weights, got {len(g)}")
        if len(g) > need:                                   # populate_weights only warns (numpy_nn.py:66-67)
            warnings.warn("There are extra weights that were not used (numpy_nn.py:66-67)")
        self._genome = torch.from_numpy(np.ascontiguousarray(g[:need])).to(self._eng.device).reshape(1, need)

    def run(self, input_vector):
        if len(input_vector) != self.nodes[0]:
            raise Exception("input vector wrong shape")            # numpy_nn.py:121-122
        x = torch.tensor(np.asarray(input_vector, np.float32).reshape(1, 1, -1), device=self._eng.device)
        act, _ = self._eng.mlp_forward(self._genome, x, want_out=False)
        return [1, 0] if int(act.item()) == _lib.ACT_UP else [0, 1]


def find_stuff(observation: np.ndarray, engine: Engine | None = None):
    """(210,160,3) uint8 -> [ball, left, right], each (row, col) float array or None."""
    eng = engine or get_engine()
    f = torch.from_numpy(np.ascontiguousarray(observation, np.uint8)).to(eng.device).reshape(1, 210, 160, 3)
    loc, valid = eng.find_stuff(f)
    loc = loc.cpu().numpy()[0].astype(np.float64); valid = valid.cpu().numpy()[0]
    return [loc[t] if valid[t] else None for t in range(3)]


class HallOfFame:
    """deap.tools.HallOfFame(maxsize): the best distinct individuals ever seen, best first -- resident on the device
    (ngp_hof_update).  The reference's in-place random.shuffle of `items` (utils.py:93-95) is not reproduced: members stay
    sorted and an opponent is drawn by index."""

    def __init__(self, maxsize: int, engine: Engine):
        self.maxsize = int(maxsize)
        self.engine = engine
        self.genomes = torch.zeros((max(1, self.maxsize), engine.gene_size), dtype=torch.float32, device=engine.device)
        self.fitness = torch.zeros(max(1, self.maxsize), dtype=torch.float64, device=engine.device)
        self.n = 0

    def __len__(self):
        return self.n

    def clear(self):
        self.n = 0

    def update(self, genomes: torch.Tensor, fitness: torch.Tensor):
        if self.maxsize == 0 or genomes.shape[0] == 0:
            return
        self.n = self.engine.hof_update(self.genomes[: self.maxsize], self.fitness[: self.maxsize], self.n, genomes.contiguous(),
                                        fitness.contiguous())

    def tensors(self, device=None):
        """(genomes [n, G], fitness [n]) views of the members, or (None, None) when empty."""
        if self.n == 0:
            return None, None
        return self.genomes[: self.n], self.fitness[: self.n]

    @property
    def items(self):
        """Host copy of the members as lists of genes, best first (DEAP's HallOfFame.items)."""
        return [row.tolist() for row in self.genomes[: self.n].cpu()]

    @property
    def keys(self):
        """Member fitness values, best first (DEAP keeps them ascending; only inspection uses this)."""
        return self.fitness[: self.n].cpu().tolist()

    def load(self, genomes: np.ndarray, fitness: np.ndarray):
        n = min(len(fitness), self.maxsize)
        self.n = n
        if n:
            self.genomes[:n] = torch.from_numpy(np.ascontiguousarray(genomes[:n], np.float32)).to(self.engine.device)
            self.fitness[:n] = torch.from_numpy(np.ascontiguousarray(fitness[:n], np.float64)).to(self.engine.device)


class Toolbox:
    """The slice of the DEAP toolbox the reference registers (ga.py:83-94), on device tensors: an individual is a row
    f32[G], a population a tensor f32[N][G], fitness a tensor f64[N]."""

    def __init__(self, config: Config | None = None, engine: Engine | None = None, seed: int = 0):
        self.config = config or Config()
        self.engine = engine or get_engine(self.config)
        self.seed = seed
        self.generation = 0
        self.hall_of_fame = HallOfFame(self.config.HALL_OF_FAME_AMOUNT, self.engine)
        self.last_frames = 0

    # ---- toolbox.population / individual / clone (ga.py:85-87) ----
    def population(self, n: int, seed: int | None = None) -> torch.Tensor:
        return self.engine.init_population(n, seed=self.seed if seed is None else seed)

    def individual(self) -> torch.Tensor:
        return self.engine.init_population(1, seed=self.seed + 0x9E3779B9 * (self.generation + 1))[0]

    @staticmethod
    def clone(t: torch.Tensor) -> torch.Tensor:
        return t.clone()

    # ---- toolbox.evaluate / toolbox.map (main.py:28-66, ga.py:83) ----
    def evaluate(self, individual, render=False):
        """main.evaluate for ONE individual -> 1-tuple (main.py:66)."""
        if isinstance(individual, torch.Tensor):
            g = individual.to(self.engine.device, torch.float32).reshape(1, -1).contiguous()
        else:
            g = torch.tensor(np.asarray(individual, np.float32).reshape(1, -1), device=self.engine.device)
        return (float(self.map_evaluate(g)[0].item()),)

    def map(self, fn, individuals):
        """toolbox.map(toolbox.evaluate, individuals) is ONE fused launch; any other function maps as usual."""
        if getattr(fn, "__func__", None) is Toolbox.evaluate and getattr(fn, "__self__", None) is self:
            if isinstance(individuals, torch.Tensor):
                g = individuals
            else:
                g = torch.tensor(np.asarray(list(individuals), np.float32), device=self.engine.device)
            return [(float(f),) for f in self.map_evaluate(g.contiguous()).cpu().tolist()]
        return map(fn, individuals)

    def map_evaluate(self, genomes: torch.Tensor, sync: bool = True) -> torch.Tensor:
        """Fitness tensor f64[N] of a whole population (device in, device out)."""
        hg, hf = self.hall_of_fame.tensors()
        out = self.engine.evaluate(genomes, hg, hf, seed=self.seed, generation=self.generation, sync=sync)
        if sync:
            self.last_frames = out["frames_total"]
        return out["fitness"]

    # ---- toolbox.select / mate / mutate (ga.py:89-94) ----
    def select(self, genomes: torch.Tensor, fitness: torch.Tensor, k: int | None = None, draws: torch.Tensor | None = None):
        """selTournament(population, k, tournsize=TOURNAMENT_SIZE) -> (the k selected individuals (copies), their indices)."""
        k = genomes.shape[0] if k is None else k
        idx = self.engine.select(fitness, k, draws, seed=self.seed, generation=self.generation)
        return genomes.index_select(0, idx.long()), idx

    def mate(self, ind1: torch.Tensor, ind2: torch.Tensor, u: torch.Tensor | None = None, pair: int = 0):
        """cxBlend in place on two individuals (rows of a population tensor work: they are contiguous views)."""
        return self.engine.mate(ind1, ind2, u, pair, seed=self.seed, generation=self.generation)

    def mutate(self, ind: torch.Tensor, u: torch.Tensor | None = None, z: torch.Tensor | None = None, slot: int = 0):
        """mutGaussian in place on one individual; returns a 1-tuple like DEAP."""
        return self.engine.mutate(ind, u, z, slot, seed=self.seed, generation=self.generation)

    def vary(self, genomes: torch.Tensor, fitness: torch.Tensor, noise: dict | None = None):
        """toolbox.select + varAnd(mate, mutate) as one fused GA step."""
        return self.engine.ga_step(genomes, fitness, seed=self.seed, generation=self.generation, noise=noise)


def cross_play(toolbox: Toolbox, a: torch.Tensor, b: torch.Tensor):
    """Every row of `a` on the right against every row of `b` on the left, as one match list (Engine.play_matches over
    cat([a, b]), the toolbox's seed and generation): one fused launch when the network fits the fused rollout, the per-frame
    driver (ngp_play_matches_stepwise) for wider networks.  A cross table such as this generation's champions against earlier
    generations' champions.  Returns dict(reward f64[A][B] of the right player, score i32[A][B][2] = (left, right) points,
    frames i32[A][B]); match (i, j) is list entry i * B + j."""
    eng = toolbox.engine
    genomes = torch.cat([a, b]).to(eng.device, torch.float32).contiguous()
    A, B = a.shape[0], b.shape[0]
    rows = torch.arange(A + B, dtype=torch.int32, device=eng.device)
    right = rows[:A].repeat_interleave(B)
    left = rows[A:].repeat(A)
    out = eng.play_matches(genomes, right, left, seed=toolbox.seed, generation=toolbox.generation)
    return {"reward": out["rewards"].view(A, B), "score": out["scores"].view(A, B, 2), "frames": out["frames"].view(A, B)}


def _stats_row(gen, nevals, fit, frames, t0):
    f = fit.double()
    return dict(gen=gen, nevals=int(nevals), avg=f.mean().item(), std=f.std(unbiased=False).item(), min=f.min().item(),
                max=f.max().item(), frames=int(frames), seconds=time.time() - t0)


def run_generations(toolbox: Toolbox, genomes: torch.Tensor, ngen: int, fitness: Optional[torch.Tensor] = None, verbose: bool = True,
                    exchange=None, noise_fn=None):
    """deap.algorithms.eaSimple as the reference drives it (main.py:165-170): evaluate the invalid individuals, update the
    hall of fame, then ngen x (select, varAnd, evaluate the invalid offspring, update the hall of fame, log
    gen/nevals/avg/std/min/max).

    fitness: None = nobody evaluated yet; otherwise f64[N] with NaN marking invalid individuals (a topped-up checkpoint).
    exchange: a parallel.Exchange when the population is sharded over several ranks (`genomes` is then this rank's shard):
    selection and variation stay inside the shard; the hall of fame is fed the merged elites of all ranks and the logbook
    rows describe the whole population, both one generation late (the all-gather of generation g is consumed while
    generation g+1 is being played, so no rank waits for another inside a generation).
    noise_fn(generation) -> dict: injected GA noise (parity tests)."""
    log = []
    sharded = exchange is not None and exchange.world > 1
    pending = None          # (gen, nevals, frames, t0) of the generation whose exchange is in flight

    def emit(row):
        log.append(row)
        if verbose:
            print("{gen}\t{nevals}\t{avg:.6g}\t{std:.6g}\t{min:.6g}\t{max:.6g}".format(**row), flush=True)

    def consume():
        nonlocal pending
        if pending is None:
            return
        fit_all, eg, ef = exchange.finish()
        toolbox.hall_of_fame.update(eg, ef)
        gen, nevals, frames, t0 = pending
        pending = None
        emit(_stats_row(gen, nevals, fit_all, frames, t0))

    def after_evaluate(gen, nevals, t0):
        nonlocal pending
        if sharded:
            consume()                                    # generation gen-1's exchange: hall of fame + logbook row
            exchange.start(genomes, fitness)
            pending = (gen, nevals, toolbox.last_frames, t0)
        else:
            toolbox.hall_of_fame.update(genomes, fitness)
            emit(_stats_row(gen, nevals, fitness, toolbox.last_frames, t0))

    t0 = time.time()
    if fitness is None or bool(torch.isnan(fitness).any()):
        evaluated = toolbox.map_evaluate(genomes)
        if fitness is None:
            nevals, fitness = genomes.shape[0], evaluated
        else:
            invalid = torch.isnan(fitness)
            nevals, fitness = int(invalid.sum().item()), torch.where(invalid, evaluated, fitness)
        after_evaluate(toolbox.generation, nevals, t0)
    for _ in range(ngen):
        toolbox.generation += 1
        t0 = time.time()
        nxt = toolbox.vary(genomes, fitness, noise_fn(toolbox.generation) if noise_fn else None)
        children, invalid, parents = nxt["genomes"], nxt["invalid"].bool(), nxt["parent_idx"].long()
        evaluated = toolbox.map_evaluate(children)
        # eaSimple re-evaluates only individuals whose fitness was invalidated; clones keep their parent's
        fitness = torch.where(invalid, evaluated, fitness.index_select(0, parents))
        genomes = children
        after_evaluate(toolbox.generation, int(invalid.sum().item()), t0)
    if sharded:
        consume()
    return genomes, fitness, log


# ---- replay of one individual with frames (pickle_inspector.py:1-12 -> main.evaluate(individual, render=True), main.py:115-125) ----
def repeat_upsample(rgb: torch.Tensor, k: int = 1, l: int = 1) -> torch.Tensor:
    """utils.repeat_upsample (utils.py:156-168): every pixel repeated k times along y and l times along x; k or l <= 0 returns
    the input unchanged (the reference logs an error once and does the same)."""
    if k <= 0 or l <= 0:
        return rgb
    return rgb.repeat_interleave(k, dim=-3).repeat_interleave(l, dim=-2)


def replay(toolbox: Toolbox, individual, game: int = 0, upsample=(4, 4), max_frames: int = 0):
    """One game of main.evaluate's schedule for ONE individual, frame by frame through the explicit-action API (ngp_env_step),
    keeping what the reference's viewer would show: returns dict(frames u8[T, 210*k, 160*l, 3] on the device -- render_game's
    upscaled rgb_array per env.step --, reward, steps, score).  game: 0 HardcodedAi, 1 the cartridge robot (players=1),
    2 ScoreHardcodedAi, 3..5 a hall-of-fame opponent when the toolbox has one (else HardcodedAi), as main.py:33-58.
    The decisions use the same kernels as the batched path (ngp_mlp_forward for the networks); there is no window and no
    sleeping to 60 fps -- showing the frames is the caller's business."""
    eng, cfg = toolbox.engine, toolbox.config
    dev = eng.device
    g = (individual if isinstance(individual, torch.Tensor) else torch.tensor(np.asarray(individual, np.float32))).to(dev, torch.float32).reshape(1, -1).contiguous()
    state = _lib.STATE_START_1P if game == 1 else _lib.STATE_START_2P
    left_genome, mult, left_kind = None, 1.0, "score" if game == 2 else "hardcoded"
    if game >= 3 and len(toolbox.hall_of_fame):
        hg, hf = toolbox.hall_of_fame.tensors()
        pick = int(torch.randint(len(toolbox.hall_of_fame), (1,)).item())
        left_genome, mult, left_kind = hg[pick:pick + 1].contiguous(), float(hf[pick].item()), "mlp"
    eng.env_reset(1, state)
    action = torch.tensor([cfg.blank_action()], dtype=torch.uint8, device=dev)
    frames, last_score, timeout, total, last_ball, steps = [], None, 0.0, 0.0, None, 0
    W, H, PH = float(cfg.GAME_WIDTH), float(cfg.GAME_PLAYABLE_HEIGHT), cfg.SCALED_PADDLE_HEIGHT

    def run(model, vec):
        act, _ = eng.mlp_forward(model, torch.tensor([[vec]], dtype=torch.float32, device=dev), want_out=False)
        return [1, 0] if int(act.item()) == _lib.ACT_UP else [0, 1]

    def bot(vec, s1, s2):
        if left_kind == "score" and s1 > s2:                           # dumb_ais.py:11-25
            return [0, 0]
        return [1, 0] if vec[1] < vec[4] else ([0, 1] if vec[1] > vec[4] else [0, 0])      # dumb_ais.py:1-8

    def clamp(valid, row, act):                                       # utils.keep_within_game_bounds_please, utils.py:71-77
        if valid:
            if row < PH:
                return [0, 1]
            if row > H - PH:
                return [1, 0]
        return act

    while True:
        out = eng.env_step(action)
        frames.append(repeat_upsample(out["frames"][0], *upsample))
        ram = out["ram"][0].cpu().numpy()
        s1, s2 = int(ram[13]), int(ram[14])
        loc = out["loc"][0].double().cpu().numpy(); valid = out["valid"][0].cpu().numpy()
        steps += 1
        la, ra = [0, 0], [0, 0]
        if valid[0]:                                                  # main.get_actions, main.py:138-154
            ball = loc[0]; last = ball if last_ball is None else last_ball
            if valid[1] and valid[2]:
                rv = [ball[1] / W, ball[0] / H, last[1] / W, last[0] / H, loc[2][0] / H, loc[1][0] / H]
                lv = [(W - ball[1]) / W, ball[0] / H, (W - last[1]) / W, last[0] / H, loc[1][0] / H, loc[2][0] / H]
                ra = run(g, rv)
                la = run(left_genome, lv) if left_kind == "mlp" else bot(lv, s1, s2)
            else:
                la, ra = ([1, 0] if torch.rand(1).item() < 0.5 else [0, 1]), ([1, 0] if torch.rand(1).item() < 0.5 else [0, 1])
        last_ball = loc[0].copy() if valid[0] else None
        ra, la = clamp(valid[2], loc[2][0], ra), clamp(valid[1], loc[1][0], la)
        a = cfg.blank_action()
        a[cfg.RIGHT_ACTION_START:cfg.RIGHT_ACTION_END] = ra; a[cfg.RIGHT_ACTION_END:cfg.LEFT_ACTION_END] = la
        action = torch.tensor([a], dtype=torch.uint8, device=dev)
        if last_score is not None:                                    # calculate_timeout_and_frames, main.py:128-135
            if last_score == (s1, s2):
                timeout += 1.0
            else:
                total += timeout; timeout = 0.0
        last_score = (s1, s2)
        if s1 >= cfg.WIN_SCORE or s2 >= cfg.WIN_SCORE or timeout > cfg.TIMEOUT_THRESH or (max_frames and steps >= max_frames):
            break
    reward = 0.0 if s1 == s2 else ((s2 - s1) + s2 * mult) / (total / cfg.TIME_SCALER)       # utils.calculate_reward, utils.py:104-109
    return {"frames": torch.stack(frames), "reward": reward, "steps": steps, "score": (s1, s2)}


def render_recorded(toolbox: Toolbox, rec: dict, matches, upsample=(1, 1), core: int | None = None, want_ram: bool = False,
                    start_states=None):
    """Re-renders recorded games (Engine.record_matches' result) pixel for pixel: the emulator is deterministic, so the
    recorded decisions are all it needs.  Each match m in `matches` is played again through env_reset + env_step (verify
    mode, every pixel), one batch per start state ('Start' with players = 1 for ROBOT matches, 'Start.2P' for the rest):
    step 0 gets BLANK_ACTION, step t gets BLANK_ACTION with record t-1's decisions written to [4:6] (right) and [6:8] (left),
    as perform_episode does (main.py:91-92).  Returns one u8[T_m, 210*k, 160*l, 3] device tensor per match, T_m =
    min(frames[m], max_record); with want_ram, (frames, ram u8[T_m, 128]) pairs.  core: the 6507 core of env_step (None =
    the toolbox config's CORE).  Resets the engine's stepwise environments (env_reset).
    start_states = (states, t): renders matches that were resumed from save states (Engine.play_matches_states) from there:
    states u8[M, NGP_GAME_STATE_BYTES] holds the state match m started from in row m, captured after t[m] env.steps (t an
    int or a sequence per match); the environments start with env_set_state and step t[m] gets record t[m]-1's decisions, so
    that entry must hold the captured frame's (branch() copies the entries below t from the original game).  Frames
    t[m]..T_m-1 are returned."""
    eng, cfg = toolbox.engine, toolbox.config
    dev = eng.device
    core = cfg.CORE if core is None else int(core)
    matches = [int(m) for m in matches]
    frames_n = rec["frames"].cpu().tolist()
    left = rec["left"].cpu().tolist()
    act = rec["record"]["act"]
    T_max = act.shape[1]
    if start_states is None:
        starts = [0] * len(frames_n)
    else:
        states, t = start_states
        starts = [int(t)] * len(frames_n) if np.ndim(t) == 0 else [int(v) for v in t]
    out = {}
    blank = torch.tensor(cfg.blank_action(), dtype=torch.uint8, device=dev)
    for state in (_lib.STATE_START_1P, _lib.STATE_START_2P):
        group = [m for m in dict.fromkeys(matches) if (left[m] == _lib.OPP_ROBOT) == (state == _lib.STATE_START_1P)]
        if not group:
            continue
        lens = [max(min(frames_n[m], T_max) - starts[m], 0) for m in group]
        T = max(lens)
        # env.step k0[i] + j of match i gets the decisions of record entry k0[i] + j - 1 (BLANK_ACTION alone for step 0)
        k = torch.tensor([starts[m] for m in group], device=dev)[:, None] + torch.arange(T, device=dev)[None, :]      # [n, T]
        a = act[torch.tensor(group, device=dev)[:, None], (k - 1).clamp(0, T_max - 1)].long()
        first = k == 0
        ra, la = torch.where(first, _lib.ACT_NONE, a >> 2).t(), torch.where(first, _lib.ACT_NONE, a & 3).t()
        actions = blank.repeat(T, len(group), 1)                                      # [T, n, 16]: input of env.step k
        actions[:, :, cfg.RIGHT_ACTION_START] = (ra == _lib.ACT_UP).to(torch.uint8)
        actions[:, :, cfg.RIGHT_ACTION_START + 1] = (ra == _lib.ACT_DOWN).to(torch.uint8)
        actions[:, :, cfg.RIGHT_ACTION_END] = (la == _lib.ACT_UP).to(torch.uint8)
        actions[:, :, cfg.RIGHT_ACTION_END + 1] = (la == _lib.ACT_DOWN).to(torch.uint8)
        pix = [torch.empty((n, 210, 160, 3), dtype=torch.uint8, device=dev) for n in lens]
        ram = [torch.empty((n, 128), dtype=torch.uint8, device=dev) for n in lens]
        if start_states is None:
            eng.env_reset(len(group), state)
        else:
            eng.env_set_state(states[torch.tensor(group, device=dev)].contiguous())
        for t in range(T):
            step = eng.env_step(actions[t].contiguous(), want_frames=True, want_obs=False, core=core)
            for i, n in enumerate(lens):
                if t < n:
                    pix[i][t] = step["frames"][i]
                    ram[i][t] = step["ram"][i]
        for i, m in enumerate(group):
            out[m] = (repeat_upsample(pix[i], *upsample), ram[i])
    return [out[m] if want_ram else out[m][0] for m in matches]


def branch(toolbox: Toolbox, genomes: torch.Tensor, right, left, m: int, t: int, new_right: int | None = None,
           new_left: int | None = None, key: int | None = None, mult=None, max_record: int | None = None):
    """A counterfactual branch of list match m (right[m] vs left[m], a genome row or OPP_* code; lists as play_matches takes
    them): the game is played to env.step t and captured there (Engine.play_matches_states), then continued from that exact
    position with new_right / new_left (None = the same players; a robot match stays a robot match) under the same fall-back
    key (key = None: m, the match's index in the list) and the toolbox's seed and generation.  Both calls run on the driver
    Engine.play_matches_states picks (the fused rollout, or the per-frame driver for wide networks).  The first resumed env.step
    still uses the decisions the old players took on frame t.  Returns record_matches' dict for the one branched match:
    rewards, frames, scores (the whole episode's), frames_total (the frames emulated after t), left, record (entries below
    t are the original game's) -- plus `capture`, the state at t, and `start_states` = (capture, t) for render_recorded.
    Raises ValueError when the game ended before env.step t."""
    eng, cfg = toolbox.engine, toolbox.config
    dev = eng.device
    genomes = genomes.to(dev, torch.float32).contiguous()
    right = [int(v) for v in (right.tolist() if torch.is_tensor(right) else right)]
    left = [int(v) for v in (left.tolist() if torch.is_tensor(left) else left)]
    mult_m = 1.0 if mult is None else float(mult[m])

    def one(v, dtype=torch.int32):
        return torch.tensor([v], dtype=dtype, device=dev)

    bound = max_record or (cfg.MAX_FRAMES if cfg.MAX_FRAMES > 0 else 2 * cfg.WIN_SCORE * (cfg.TIMEOUT_THRESH + 2))
    k = one(m if key is None else int(key))
    common = dict(key=k, max_record=bound, seed=toolbox.seed, generation=toolbox.generation)
    orig = eng.play_matches_states(genomes, one(right[m]), one(left[m]), one(mult_m, torch.float64), capture_at=one(int(t)), **common)
    if int(orig["frames"].item()) <= t:
        raise ValueError(f"match {m} ended after {int(orig['frames'].item())} env.steps, before env.step {t}")
    nr = right[m] if new_right is None else int(new_right)
    nl = left[m] if new_left is None else int(new_left)
    out = eng.play_matches_states(genomes, one(nr), one(nl), one(mult_m, torch.float64), states=orig["capture"], start=one(0),
                                  **common)
    out["record"]["raw"][:, :t] = orig["record"]["raw"][:, :t]
    out["capture"] = orig["capture"]
    out["start_states"] = (orig["capture"], int(t))
    return out


def model_policy(model):
    """A policy for play_policy from a reference-style model object -- anything with .run(vec6) -> [up, down], as
    perform_episode takes it (main.py:69-112): numpy_nn.NeuralNetwork, a dumb_ais bot, a keyboard reader.  Each observation row
    is passed to model.run as a list of six floats; [1, 0] is NGP_ACT_UP, [0, 1] NGP_ACT_DOWN, anything else NGP_ACT_NONE
    (both buttons held cancel, FILTERED, main.py:23,55)."""
    def policy(obs: torch.Tensor) -> torch.Tensor:
        acts = []
        for vec in obs.detach().cpu().double().numpy():
            up, down = (bool(v) for v in model.run([float(v) for v in vec])[:2])
            acts.append(_lib.ACT_UP if up and not down else _lib.ACT_DOWN if down and not up else _lib.ACT_NONE)
        return torch.tensor(acts, dtype=torch.uint8, device=obs.device)
    return policy


def play_policy(toolbox: Toolbox, genomes: torch.Tensor | None, right, left, policy, mult=None, key=None, states=None, start=None,
                fresh: bool = False, max_record: int | None = None, check_every: int = 8):
    """Plays a match list in which every seat named PLAYER_EXTERNAL is driven by `policy` (play_against_human.py /
    main.run_against_human with any controller): policy(obs f32[K, 6]) -> K NGP_ACT_* decisions (a tensor or a sequence), called
    once per step on the external seats whose match needs a decision (Engine.session's NEED; utils.inference's vector, the left
    seat's x-mirrored), not called on a step without one.  right / left: lists as Engine.session takes them (sequences or int32
    tensors); genomes may be None when no seat names a row.  Runs on the toolbox's seed and generation and records every frame
    (max_record None = the longest possible game of the config), so that render_recorded re-renders any game of the result.
    check_every: steps between two reads of the running count (each read synchronises).  Returns MatchSession.result()."""
    eng, cfg = toolbox.engine, toolbox.config
    dev = eng.device

    def dev_i32(v):
        return (v if torch.is_tensor(v) else torch.tensor(list(v), dtype=torch.int32)).to(dev, torch.int32).contiguous()

    r, l = dev_i32(right), dev_i32(left)
    bound = max_record or (cfg.MAX_FRAMES if cfg.MAX_FRAMES > 0 else 2 * cfg.WIN_SCORE * (cfg.TIMEOUT_THRESH + 2))
    if genomes is not None:
        genomes = genomes.to(dev, torch.float32).contiguous()
    with eng.session(genomes, r, l, mult=mult, key=key, states=states, start=start, fresh=fresh, max_record=bound, seed=toolbox.seed,
                     generation=toolbox.generation) as s:
        external = torch.stack([l == _lib.PLAYER_EXTERNAL, r == _lib.PLAYER_EXTERNAL], dim=1)          # [M, 2] (left, right)
        actions = torch.zeros((r.shape[0], 2), dtype=torch.uint8, device=dev)
        step = 0
        while step % check_every or s.running():
            rows = external & s.need[:, None]
            if bool(rows.any()):
                act = policy(s.obs[rows])
                actions[rows] = torch.as_tensor(act, device=dev).to(torch.uint8)
            s.step(actions)
            step += 1
        return s.result()


def replay_selfplay(toolbox: Toolbox, genomes: torch.Tensor, g: int, k: int, upsample=(4, 4)):
    """Round-robin game k of genome g, played and rendered exactly as Engine.evaluate plays it under SCHEDULE_ROUND_ROBIN
    with the toolbox's seed and generation: one record_matches call (right = g, left = (g + k + 1) % n, key = g * games + k;
    the fused rollout, or the per-frame driver for wide networks), then render_recorded.  Returns replay's dict: frames u8[T, 210*k, 160*l, 3], reward, steps, score = (left, right)."""
    eng, cfg = toolbox.engine, toolbox.config
    dev = eng.device
    n, games = genomes.shape[0], cfg.GAMES_TO_PLAY
    genomes = genomes.to(dev, torch.float32).contiguous()

    def one(v):
        return torch.tensor([v], dtype=torch.int32, device=dev)

    # an episode ends at the latest when a point has not been scored for TIMEOUT_THRESH frames after the last of the
    # 2 * WIN_SCORE - 1 points that can be scored
    bound = cfg.MAX_FRAMES if cfg.MAX_FRAMES > 0 else 2 * cfg.WIN_SCORE * (cfg.TIMEOUT_THRESH + 2)
    args = (genomes, one(g), one((g + k + 1) % n))
    rec = eng.record_matches(*args, key=one(g * games + k), max_record=bound, seed=toolbox.seed, generation=toolbox.generation)
    steps = int(rec["frames"].item())
    if steps > bound:                                    # never expected; the replay is deterministic, so record it again
        rec = eng.record_matches(*args, key=one(g * games + k), max_record=steps, seed=toolbox.seed, generation=toolbox.generation)
    frames = render_recorded(toolbox, rec, [0], upsample=upsample)[0]
    s1, s2 = (int(v) for v in rec["scores"][0].tolist())
    return {"frames": frames, "reward": float(rec["rewards"].item()), "steps": steps, "score": (s1, s2)}


# ---- checkpoint / resume (utils.py:116-125, ga.py:13-53) -------------------------------------------
# Layout: one .npz per checkpoint (population, fitness, hall of fame, Philox seed + generation counter = the RNG state,
# network_shape, bias).  The reference pickles DEAP objects (deap.creator.Individual, tools.HallOfFame); its files are read
# one way by read_reference_checkpoint (stand-in classes, no DEAP needed), so a run of the reference can be continued here.
def save_checkpoint(toolbox: Toolbox, genomes: torch.Tensor, fitness: torch.Tensor, directory: str = "checkpoints/checkpoints") -> str:
    os.makedirs(directory, exist_ok=True)
    path = os.path.join(directory, "c_{}.npz".format(time.strftime("%H_%M_%S")))
    k = 1
    while os.path.exists(path):                          # two saves within one second (the reference would overwrite)
        path = os.path.join(directory, "c_{}_{}.npz".format(time.strftime("%H_%M_%S"), k)); k += 1
    hof = toolbox.hall_of_fame
    hg, hf = hof.tensors()
    np.savez(path, population=genomes.cpu().numpy(), fitness=fitness.cpu().numpy(),
             hof_genomes=hg.cpu().numpy() if hg is not None else np.zeros((0, genomes.shape[1]), np.float32),
             hof_fitness=hf.cpu().numpy() if hf is not None else np.zeros(0, np.float64), seed=np.uint64(toolbox.seed),
             generation=np.uint64(toolbox.generation), network_shape=np.asarray(toolbox.config.NETWORK_SHAPE, np.int32),
             bias=np.int32(1 if toolbox.config.BIAS else 0))
    return path


def read_reference_checkpoint(path: str):
    """One-way importer of the REFERENCE's checkpoints (utils.save_checkpoint, utils.py:116-125: a pickled dict with
    population = list of deap.creator.Individual, hall_of_fame = deap.tools.HallOfFame, rndstate, network_shape) without
    DEAP: the unpickler substitutes plain stand-ins for every class under `deap.` (an Individual is a list of genes whose
    `fitness.wvalues` holds the weighted fitness; weights are (1.0,), ga.py:80).  Returns a dict with population f32[N][G],
    fitness f64[N] (NaN = invalid), hof_genomes, hof_fitness (best first), network_shape.  `rndstate` (Python's Mersenne
    twister) has no counterpart here: the Philox seed/generation of the toolbox stay as they are."""
    import pickle

    class _Obj:
        def __setstate__(self, state):
            if isinstance(state, tuple) and len(state) == 2 and isinstance(state[1], dict):      # (dict, slots)
                state = {**(state[0] or {}), **state[1]}
            self.__dict__.update(state or {})

    class _Seq(list, _Obj):
        pass

    class _Unpickler(pickle.Unpickler):
        def find_class(self, module, name):
            if module.split(".")[0] in ("deap", "scoop"):
                return _Seq if name == "Individual" else type(name, (_Obj,), {})
            return super().find_class(module, name)

    with open(path, "rb") as f:
        cp = _Unpickler(f).load()

    def fit_of(ind):
        w = getattr(getattr(ind, "fitness", None), "wvalues", ())
        return float(w[0]) if len(w) else float("nan")

    pop = list(cp["population"])
    out = {"population": np.asarray([list(i) for i in pop], np.float32).reshape(len(pop), -1),
           "fitness": np.asarray([fit_of(i) for i in pop], np.float64),
           "network_shape": tuple(int(v) for v in cp.get("network_shape", ())) or None}
    hof = cp.get("hall_of_fame")
    items = list(getattr(hof, "items", [])) if hof is not None else []
    out["hof_genomes"] = np.asarray([list(i) for i in items], np.float32).reshape(len(items), -1)
    out["hof_fitness"] = np.asarray([fit_of(i) for i in items], np.float64)          # DEAP keeps items best first
    return out


def load_latest_population(toolbox: Toolbox, directory: str = "checkpoints/checkpoints"):
    """Newest checkpoint by ctime (ga.py:32-38), sorted by fitness descending (ga.py:45), truncated or topped up with fresh
    random individuals to POPULATION_SIZE (ga.py:13-29).  Returns (genomes, fitness); fitness is None without a checkpoint
    and holds NaN for topped-up (never evaluated) individuals -- loaded individuals keep their fitness, as in the reference."""
    files = glob.glob(os.path.join(directory, "*.npz")) + glob.glob(os.path.join(directory, "*.pkl"))
    n = toolbox.config.POPULATION_SIZE
    if not files:
        others = glob.glob(os.path.join(directory, "*"))
        if others:
            warnings.warn(f"{len(others)} file(s) in {directory} are neither .npz checkpoints of this package nor the reference's "
                          ".pkl checkpoints and are ignored")
        return toolbox.population(n), None
    newest = max(files, key=os.path.getctime)
    if newest.endswith(".pkl"):                          # a checkpoint written by the reference itself (utils.py:116-125)
        ref = read_reference_checkpoint(newest)
        if ref["population"].shape[1] != toolbox.engine.gene_size:
            raise _lib.NgpError("reference checkpoint gene size differs from the configured NETWORK_SHAPE; rebuild the Toolbox with it")
        valid = ~np.isnan(ref["hof_fitness"])            # utils.py:96-98 skips hall-of-fame members without a valid fitness
        cp = {"network_shape": np.asarray(ref["network_shape"] or toolbox.config.NETWORK_SHAPE, np.int32), "fitness": ref["fitness"],
              "population": ref["population"], "seed": toolbox.seed, "generation": toolbox.generation,
              "hof_genomes": ref["hof_genomes"][valid], "hof_fitness": ref["hof_fitness"][valid]}
        cp["fitness"] = np.where(np.isnan(cp["fitness"]), -np.inf, cp["fitness"])            # invalid individuals sort last ...
    else:
        cp = np.load(newest)
    if tuple(int(v) for v in cp["network_shape"]) != tuple(toolbox.config.NETWORK_SHAPE):
        raise _lib.NgpError("checkpoint network_shape differs from the configured NETWORK_SHAPE; rebuild the Toolbox with it")
    if "bias" in cp and bool(int(cp["bias"])) != bool(toolbox.config.BIAS):
        raise _lib.NgpError("checkpoint BIAS differs from the configured BIAS")
    order = np.argsort(-cp["fitness"], kind="stable")
    pop, fit = cp["population"][order][:n], cp["fitness"][order][:n]
    toolbox.seed = int(cp["seed"]); toolbox.generation = int(cp["generation"])
    toolbox.hall_of_fame.load(cp["hof_genomes"], cp["hof_fitness"])
    dev = toolbox.engine.device
    fit = np.where(np.isinf(fit), np.nan, fit)                                                # ... and are re-evaluated
    genomes = torch.from_numpy(np.ascontiguousarray(pop)).to(dev)
    fitness = torch.from_numpy(np.ascontiguousarray(fit)).to(dev)
    if len(pop) < n:
        fresh = toolbox.population(n - len(pop), seed=toolbox.seed + 1 + toolbox.generation)
        genomes = torch.cat([genomes, fresh])
        fitness = torch.cat([fitness, torch.full((n - len(pop),), float("nan"), dtype=torch.float64, device=dev)])
    return genomes, fitness
