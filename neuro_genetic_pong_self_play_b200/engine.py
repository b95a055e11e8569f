"""Engine: one ngp_handle per GPU.  PyTorch tensors are used only as device buffers (data_ptr()
goes straight into the C ABI); all computation happens in libngp.so's CUDA kernels."""
from __future__ import annotations

import ctypes
import os
from typing import Optional

import numpy as np
import torch

from . import _lib
from .config import Config

ROM_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data", "video_olympics.a26")


def load_rom() -> bytes:
    with open(ROM_PATH, "rb") as f:
        rom = f.read()
    if len(rom) != 2048:
        raise _lib.NgpError("bundled cartridge image must be 2048 bytes")
    return rom


def _p(t: Optional[torch.Tensor]):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream(device) -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def record_views(raw: torch.Tensor) -> dict:
    """Named views of an ngp_frame_record buffer u8[M, T, 32] (include/ngp.h): loc f32[M, T, 3, 2], valid u8[M, T],
    score u8[M, T, 2], act u8[M, T], timeout i32[M, T]; `raw` is the buffer itself."""
    m, t = raw.shape[0], raw.shape[1]
    return {"raw": raw, "loc": raw[..., 0:24].view(torch.float32).view(m, t, 3, 2), "valid": raw[..., 24],
            "score": raw[..., 25:27], "act": raw[..., 27], "timeout": raw[..., 28:32].view(torch.int32).view(m, t)}


class Engine:
    def __init__(self, config: Config | None = None, device: int | None = None, rom: bytes | None = None):
        if not torch.cuda.is_available():
            raise _lib.NgpError("no CUDA device: this package has no CPU fallback")
        self.config = config or Config()
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device("cuda", self.device_index)
        self._L = _lib.load()
        torch.cuda.init()
        with torch.cuda.device(self.device):
            torch.zeros(1, device=self.device)            # make sure the primary context exists
            h = ctypes.c_void_p()
            cfg = self.config.to_c()
            image = load_rom() if rom is None else bytes(rom)      # another 2 KiB cartridge: interpreter core only
            if len(image) != 2048:
                raise _lib.NgpError("cartridge image must be 2048 bytes")
            _lib.check(self._L.ngp_create(ctypes.byref(cfg), image, self.device_index, ctypes.byref(h)), "ngp_create")
        self._h = h
        self.gene_size = int(self._L.ngp_gene_size(self._h))
        self._n_envs = 0

    def close(self):
        if getattr(self, "_h", None):
            self._L.ngp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launches(self) -> int:
        return int(self._L.ngp_launch_count(self._h))

    def profile_enable(self, on: bool = True):
        _lib.check(self._L.ngp_profile_enable(self._h, 1 if on else 0), "ngp_profile_enable")

    def profile_read(self):
        """(milliseconds, launches) of the fused rollout kernel since the last read (CUDA events on its stream)."""
        ms, n = ctypes.c_double(0.0), ctypes.c_int32(0)
        _lib.check(self._L.ngp_profile_read(self._h, ctypes.byref(ms), ctypes.byref(n)), "ngp_profile_read")
        return ms.value, n.value

    def set_option(self, name: str, value: int):
        """Tuning switch (include/ngp.h: ngp_set_option); 0 restores the automatic choice."""
        _lib.check(self._L.ngp_set_option(self._h, name.encode(), int(value)), "ngp_set_option")

    def _check_tensor(self, t: torch.Tensor, dtype, name: str):
        if not (t.is_cuda and t.device == self.device and t.dtype == dtype and t.is_contiguous()):
            raise ValueError(f"{name}: expected a contiguous {dtype} tensor on {self.device}")

    # ---- K1: explicit-action stepping (retro env.reset / env.step stand-in) -----------------
    def env_reset(self, n_envs: int, state: int = _lib.STATE_START_2P):
        _lib.check(self._L.ngp_env_reset(self._h, n_envs, state, _stream(self.device)), "ngp_env_reset")
        self._n_envs = n_envs

    def env_step(self, actions: torch.Tensor, want_frames: bool = True, want_obs: bool = True, core: int = _lib.CORE_INTERPRETER):
        """actions: u8[n_envs,16] gym-retro buttons.  Returns dict(ram, frames, loc, valid, regs)."""
        n = self._n_envs
        self._check_tensor(actions, torch.uint8, "actions")
        assert tuple(actions.shape) == (n, 16)
        out = {
            "ram": torch.empty((n, 128), dtype=torch.uint8, device=self.device),
            "regs": torch.empty((n, 8), dtype=torch.uint8, device=self.device),
            "frames": torch.empty((n, 210, 160, 3), dtype=torch.uint8, device=self.device) if want_frames else None,
            "loc": torch.empty((n, 3, 2), dtype=torch.float32, device=self.device) if want_obs else None,
            "valid": torch.empty((n, 3), dtype=torch.uint8, device=self.device) if want_obs else None,
        }
        _lib.check(self._L.ngp_env_step_core(self._h, core, _p(actions), _p(out["ram"]), _p(out["frames"]), _p(out["loc"]),
                                             _p(out["valid"]), _p(out["regs"]), _stream(self.device)), "ngp_env_step")
        return out

    def env_get_state(self) -> torch.Tensor:
        """Save states of the stepwise environments as env_reset / env_step / env_set_state left them (gym-retro
        env.em.get_state()): u8[n_envs, NGP_GAME_STATE_BYTES], without an episode."""
        out = torch.empty((self._n_envs, _lib.NGP_GAME_STATE_BYTES), dtype=torch.uint8, device=self.device)
        _lib.check(self._L.ngp_env_get_state(self._h, _p(out), _stream(self.device)), "ngp_env_get_state")
        return out

    def env_set_state(self, states: torch.Tensor):
        """The counterpart of env_reset (gym-retro env.em.set_state()): the stepwise environments become the consoles of
        `states` u8[n, NGP_GAME_STATE_BYTES] (one players value for all; any episode part is ignored).  A state that fails
        validation raises NgpError and leaves the environments as they were."""
        self._check_tensor(states, torch.uint8, "states")
        assert states.dim() == 2 and states.shape[1] == _lib.NGP_GAME_STATE_BYTES
        _lib.check(self._L.ngp_env_set_state(self._h, _p(states), states.shape[0], _stream(self.device)), "ngp_env_set_state")
        self._n_envs = states.shape[0]

    def env_digest(self) -> torch.Tensor:
        d = torch.empty((self._n_envs, 8), dtype=torch.int32, device=self.device)
        _lib.check(self._L.ngp_env_digest(self._h, _p(d), _stream(self.device)), "ngp_env_digest")
        return d

    # ---- K2 ----------------------------------------------------------------------------------
    def find_stuff(self, frames: torch.Tensor):
        self._check_tensor(frames, torch.uint8, "frames")
        n = frames.shape[0]
        assert tuple(frames.shape[1:]) == (210, 160, 3)
        loc = torch.empty((n, 3, 2), dtype=torch.float32, device=self.device)
        valid = torch.empty((n, 3), dtype=torch.uint8, device=self.device)
        _lib.check(self._L.ngp_find_stuff(self._h, _p(frames), n, _p(loc), _p(valid), _stream(self.device)), "ngp_find_stuff")
        return loc, valid

    # ---- K3 ----------------------------------------------------------------------------------
    def mlp_forward(self, genomes: torch.Tensor, x: torch.Tensor, want_out: bool = True):
        self._check_tensor(genomes, torch.float32, "genomes")
        self._check_tensor(x, torch.float32, "x")
        n, envs = x.shape[0], x.shape[1]
        assert tuple(genomes.shape) == (n, self.gene_size) and x.shape[2] == self.config.NETWORK_SHAPE[0]
        act = torch.empty((n, envs), dtype=torch.uint8, device=self.device)
        out = torch.empty((n, envs, self.config.NETWORK_SHAPE[-1]), dtype=torch.float32, device=self.device) if want_out else None
        _lib.check(self._L.ngp_mlp_forward(self._h, _p(genomes), _p(x), n, envs, _p(act), _p(out), _stream(self.device)), "ngp_mlp_forward")
        return act, out

    def mlp_prepare(self, genomes: torch.Tensor):
        """NeuralNetwork.__init__/populate_weights for a whole genome set: packs the wide layers once (ngp_mlp_prepare)."""
        self._check_tensor(genomes, torch.float32, "genomes")
        assert genomes.shape[1] == self.gene_size
        _lib.check(self._L.ngp_mlp_prepare(self._h, _p(genomes), genomes.shape[0], _stream(self.device)), "ngp_mlp_prepare")

    def mlp_forward_prepared(self, genomes: torch.Tensor, x: torch.Tensor, want_out: bool = True):
        """mlp_forward on the genome set last passed to mlp_prepare (weights streamed from the packed copy)."""
        self._check_tensor(genomes, torch.float32, "genomes")
        self._check_tensor(x, torch.float32, "x")
        n, envs = x.shape[0], x.shape[1]
        act = torch.empty((n, envs), dtype=torch.uint8, device=self.device)
        out = torch.empty((n, envs, self.config.NETWORK_SHAPE[-1]), dtype=torch.float32, device=self.device) if want_out else None
        _lib.check(self._L.ngp_mlp_forward_prepared(self._h, _p(genomes), _p(x), n, envs, _p(act), _p(out), _stream(self.device)),
                   "ngp_mlp_forward_prepared")
        return act, out

    # ---- fused hot path ----------------------------------------------------------------------
    def evaluate(self, genomes: torch.Tensor, hof_genomes: torch.Tensor | None = None, hof_fitness: torch.Tensor | None = None,
                 hof_pick: torch.Tensor | None = None, seed: int = 0, generation: int = 0, want_detail: bool = False,
                 sync: bool = True):
        """population genomes in -> fitness out (toolbox.map(toolbox.evaluate, population))."""
        self._check_tensor(genomes, torch.float32, "genomes")
        n = genomes.shape[0]
        assert genomes.shape[1] == self.gene_size
        n_hof = 0 if hof_genomes is None else hof_genomes.shape[0]
        if n_hof:
            self._check_tensor(hof_genomes, torch.float32, "hof_genomes")
            self._check_tensor(hof_fitness, torch.float64, "hof_fitness")
        if hof_pick is not None:
            self._check_tensor(hof_pick, torch.int32, "hof_pick")
        games = self.config.GAMES_TO_PLAY
        fitness = torch.empty(n, dtype=torch.float64, device=self.device)
        rewards = torch.empty((n, games), dtype=torch.float64, device=self.device) if want_detail else None
        frames = torch.empty((n, games), dtype=torch.int32, device=self.device) if want_detail else None
        total = ctypes.c_uint64(0)
        _lib.check(self._L.ngp_evaluate(self._h, _p(genomes), n, _p(hof_genomes) if n_hof else None, _p(hof_fitness) if n_hof else None,
                                        n_hof, _p(hof_pick), seed, generation, _p(fitness), _p(rewards), _p(frames),
                                        ctypes.byref(total) if sync else None, _stream(self.device)), "ngp_evaluate")
        return {"fitness": fitness, "rewards": rewards, "frames": frames, "frames_total": int(total.value) if sync else None}

    def _match_list(self, genomes, right, left, **per_match):
        """The argument check and the outputs the match-list methods share: genomes f32[N, gene_size], right and left i32[M],
        and per_match name=(tensor or None, dtype) of shape [M].  Returns dict(rewards f64[M], frames i32[M], scores i32[M, 2])."""
        self._check_tensor(genomes, torch.float32, "genomes")
        self._check_tensor(right, torch.int32, "right")
        self._check_tensor(left, torch.int32, "left")
        assert genomes.dim() == 2 and genomes.shape[1] == self.gene_size
        m = right.shape[0]
        assert right.dim() == 1 and tuple(left.shape) == (m,)
        for name, (t, dtype) in per_match.items():
            if t is not None:
                self._check_tensor(t, dtype, name)
                assert tuple(t.shape) == (m,), name
        return {"rewards": torch.empty(m, dtype=torch.float64, device=self.device),
                "frames": torch.empty(m, dtype=torch.int32, device=self.device),
                "scores": torch.empty((m, 2), dtype=torch.int32, device=self.device)}

    def play_matches(self, genomes: torch.Tensor, right: torch.Tensor, left: torch.Tensor, mult: torch.Tensor | None = None,
                     seed: int = 0, generation: int = 0, sync: bool = True):
        """An explicit match list in one fused launch (ngp_play_matches): match m puts genome row right[m] on the right against
        genome row left[m] (x-mirrored, as in self-play) or an OPP_* code; mult[m] is the hall-of-fame multiplier of the right
        player's score bonus (None = 1.0).  Returns dict(rewards f64[M] of the right player, frames i32[M], scores i32[M, 2]
        = (left, right) points, frames_total).  The lists are checked on the device; a bad entry raises NgpError and nothing
        is played."""
        out = self._match_list(genomes, right, left, mult=(mult, torch.float64))
        total = ctypes.c_uint64(0)
        _lib.check(self._L.ngp_play_matches(self._h, _p(genomes), genomes.shape[0], _p(right), _p(left), _p(mult), right.shape[0], seed,
                                            generation, _p(out["rewards"]), _p(out["frames"]), _p(out["scores"]),
                                            ctypes.byref(total) if sync else None, _stream(self.device)), "ngp_play_matches")
        out["frames_total"] = int(total.value) if sync else None
        return out

    def record_matches(self, genomes: torch.Tensor, right: torch.Tensor, left: torch.Tensor, mult: torch.Tensor | None = None,
                       key: torch.Tensor | None = None, max_record: int = 2048, seed: int = 0, generation: int = 0, sync: bool = True):
        """play_matches with a per-frame trace of every match, recorded in the same fused launch (ngp_record_matches).
        key[m] (None = m) is the environment index of the random fall-back key, so that one match can reproduce one game of
        an evaluate call (round-robin game k of genome g: key g * games + k).  Returns play_matches' dict plus `left` (kept
        for rendering) and `record`: named views over one u8[M, T, 32] buffer (T = max_record; frame t of match m is valid
        for t < min(frames[m], T)): loc f32[M, T, 3, 2], valid u8[M, T] (bit 0 ball, 1 left, 2 right), score u8[M, T, 2],
        act u8[M, T] (left | right << 2, after the bounds clamp) and timeout i32[M, T]."""
        out = self._match_list(genomes, right, left, mult=(mult, torch.float64), key=(key, torch.int32))
        m = right.shape[0]
        raw = torch.empty((m, max(int(max_record), 0), _lib.NGP_FRAME_RECORD_BYTES), dtype=torch.uint8, device=self.device)
        total = ctypes.c_uint64(0)
        _lib.check(self._L.ngp_record_matches(self._h, _p(genomes), genomes.shape[0], _p(right), _p(left), _p(mult), _p(key), m, seed,
                                              generation, int(max_record), _p(raw), _p(out["rewards"]), _p(out["frames"]),
                                              _p(out["scores"]), ctypes.byref(total) if sync else None, _stream(self.device)),
                   "ngp_record_matches")
        out.update(frames_total=int(total.value) if sync else None, left=left, record=record_views(raw))
        return out

    def play_matches_states(self, genomes: torch.Tensor, right: torch.Tensor, left: torch.Tensor, mult: torch.Tensor | None = None,
                            key: torch.Tensor | None = None, states: torch.Tensor | None = None, start: torch.Tensor | None = None,
                            fresh: bool = False, capture_at: torch.Tensor | None = None, max_record: int = 0, seed: int = 0,
                            generation: int = 0, sync: bool = True):
        """record_matches whose matches may start from save states and capture their own (ngp_play_matches_states).
        states: u8[S, NGP_GAME_STATE_BYTES]; start[m] (None = all -1) picks match m's start state, -1 = the built-in one.  A
        state with an episode resumes it unless `fresh`; a fresh start plays a new episode from the state's console.
        capture_at[m]: after that many env.steps from the episode's start the state of match m is captured (left as zeros
        when the game ended before).  max_record > 0 records every frame as record_matches does.  Returns play_matches'
        dict plus `left`, plus `capture` u8[M, NGP_GAME_STATE_BYTES] when capture_at is given and `record` views when
        max_record > 0.  Bad entries or states raise NgpError and nothing is played."""
        out = self._match_list(genomes, right, left, mult=(mult, torch.float64), key=(key, torch.int32), start=(start, torch.int32),
                               capture_at=(capture_at, torch.int32))
        m = right.shape[0]
        n_states = 0
        if states is not None:
            self._check_tensor(states, torch.uint8, "states")
            assert states.dim() == 2 and states.shape[1] == _lib.NGP_GAME_STATE_BYTES
            n_states = states.shape[0]
        capture = torch.zeros((m, _lib.NGP_GAME_STATE_BYTES), dtype=torch.uint8, device=self.device) if capture_at is not None else None
        raw = (torch.empty((m, int(max_record), _lib.NGP_FRAME_RECORD_BYTES), dtype=torch.uint8, device=self.device)
               if max_record > 0 else None)
        total = ctypes.c_uint64(0)
        _lib.check(self._L.ngp_play_matches_states(
            self._h, _p(genomes), genomes.shape[0], _p(right), _p(left), _p(mult), _p(key), m, _p(states) if n_states else None,
            n_states, _p(start), 1 if fresh else 0, _p(capture_at), _p(capture), int(max_record), _p(raw), seed, generation,
            _p(out["rewards"]), _p(out["frames"]), _p(out["scores"]), ctypes.byref(total) if sync else None, _stream(self.device)),
            "ngp_play_matches_states")
        out.update(frames_total=int(total.value) if sync else None, left=left)
        if capture is not None:
            out["capture"] = capture
        if raw is not None:
            out["record"] = record_views(raw)
        return out

    def evaluate_host(self, genomes: np.ndarray, hof_genomes: np.ndarray | None = None, hof_fitness: np.ndarray | None = None,
                      seed: int = 0, generation: int = 0):
        """Same, through host buffers (H2D of genomes and D2H of fitness inside the call)."""
        g = np.ascontiguousarray(genomes, np.float32)
        n = g.shape[0]
        fitness = np.empty(n, np.float64)
        n_hof = 0 if hof_genomes is None else len(hof_genomes)
        hg = np.ascontiguousarray(hof_genomes, np.float32) if n_hof else None
        hf = np.ascontiguousarray(hof_fitness, np.float64) if n_hof else None
        total = ctypes.c_uint64(0)
        _lib.check(self._L.ngp_evaluate_host(self._h, g.ctypes.data_as(ctypes.c_void_p), n,
                                             hg.ctypes.data_as(ctypes.c_void_p) if n_hof else None,
                                             hf.ctypes.data_as(ctypes.c_void_p) if n_hof else None, n_hof, seed, generation,
                                             fitness.ctypes.data_as(ctypes.c_void_p), ctypes.byref(total)), "ngp_evaluate_host")
        return fitness, int(total.value)

    # ---- K4 ----------------------------------------------------------------------------------
    def init_population(self, n: int, seed: int = 0) -> torch.Tensor:
        g = torch.empty((n, self.gene_size), dtype=torch.float32, device=self.device)
        _lib.check(self._L.ngp_init_population(self._h, _p(g), n, seed, _stream(self.device)), "ngp_init_population")
        return g

    def ga_step(self, genomes: torch.Tensor, fitness: torch.Tensor, seed: int = 0, generation: int = 0, noise: dict | None = None):
        self._check_tensor(genomes, torch.float32, "genomes")
        self._check_tensor(fitness, torch.float64, "fitness")
        n = genomes.shape[0]
        nz = None
        if noise is not None:
            nz = _lib.NgpNoise()
            for k in ("sel_draws", "cx_do", "cx_u", "mut_do", "mut_u", "mut_z"):
                t = noise.get(k)
                setattr(nz, k, None if t is None else t.data_ptr())
        nxt = torch.empty_like(genomes)
        parent = torch.empty(n, dtype=torch.int32, device=self.device)
        invalid = torch.empty(n, dtype=torch.uint8, device=self.device)
        stats = torch.empty(4, dtype=torch.float64, device=self.device)
        _lib.check(self._L.ngp_ga_step(self._h, _p(genomes), _p(fitness), n, seed, generation, ctypes.byref(nz) if nz else None,
                                       _p(nxt), _p(parent), _p(invalid), _p(stats), _stream(self.device)), "ngp_ga_step")
        return {"genomes": nxt, "parent_idx": parent, "invalid": invalid, "stats": stats}

    # ---- toolbox.select / mate / mutate as separate callables (ga.py:89-94) -------------------
    def select(self, fitness: torch.Tensor, k: int, draws: torch.Tensor | None = None, seed: int = 0, generation: int = 0) -> torch.Tensor:
        """selTournament(individuals, k, tournsize=TOURNAMENT_SIZE) -> winner indices i32[k]."""
        self._check_tensor(fitness, torch.float64, "fitness")
        if draws is not None:
            self._check_tensor(draws, torch.int32, "draws")
            assert tuple(draws.shape) == (k, max(1, self.config.TOURNAMENT_SIZE))
        out = torch.empty(k, dtype=torch.int32, device=self.device)
        _lib.check(self._L.ngp_select(self._h, _p(fitness), fitness.shape[0], k, _p(draws), seed, generation, _p(out), _stream(self.device)),
                   "ngp_select")
        return out

    def mate(self, ind1: torch.Tensor, ind2: torch.Tensor, u: torch.Tensor | None = None, pair: int = 0, seed: int = 0, generation: int = 0):
        """cxBlend(ind1, ind2, CROSSOVER_BLEND_ALPHA) in place."""
        for t, nme in ((ind1, "ind1"), (ind2, "ind2")):
            self._check_tensor(t, torch.float32, nme)
            assert t.numel() == self.gene_size
        if u is not None:
            self._check_tensor(u, torch.float32, "u")
        _lib.check(self._L.ngp_mate(self._h, _p(ind1), _p(ind2), _p(u), pair, seed, generation, _stream(self.device)), "ngp_mate")
        return ind1, ind2

    def mutate(self, ind: torch.Tensor, u: torch.Tensor | None = None, z: torch.Tensor | None = None, slot: int = 0, seed: int = 0,
               generation: int = 0):
        """mutGaussian(ind, mu, sigma, indpb) in place."""
        self._check_tensor(ind, torch.float32, "ind")
        assert ind.numel() == self.gene_size
        _lib.check(self._L.ngp_mutate(self._h, _p(ind), _p(u), _p(z), slot, seed, generation, _stream(self.device)), "ngp_mutate")
        return (ind,)

    # ---- hall of fame --------------------------------------------------------------------------
    def hof_update(self, hof_genomes: torch.Tensor, hof_fitness: torch.Tensor, n_hof: int, genomes: torch.Tensor, fitness: torch.Tensor) -> int:
        """HallOfFame(maxsize).update(population) on device buffers [maxsize, G] / [maxsize]; returns the new member count."""
        self._check_tensor(hof_genomes, torch.float32, "hof_genomes")
        self._check_tensor(hof_fitness, torch.float64, "hof_fitness")
        self._check_tensor(genomes, torch.float32, "genomes")
        self._check_tensor(fitness, torch.float64, "fitness")
        maxsize = hof_genomes.shape[0]
        assert hof_fitness.shape[0] == maxsize and genomes.shape[0] == fitness.shape[0]
        cnt = ctypes.c_int32(n_hof)
        _lib.check(self._L.ngp_hof_update(self._h, _p(hof_genomes), _p(hof_fitness), ctypes.byref(cnt), maxsize, _p(genomes), _p(fitness),
                                          genomes.shape[0], _stream(self.device)), "ngp_hof_update")
        return int(cnt.value)

    # ---- multi-GPU exchange records --------------------------------------------------------------
    def exchange_bytes(self, n_max: int, k_max: int) -> int:
        return int(self._L.ngp_exchange_bytes(self._h, n_max, k_max))

    def pack_elites(self, genomes: torch.Tensor, fitness: torch.Tensor, k: int, n_max: int, k_max: int, out: torch.Tensor | None = None):
        self._check_tensor(genomes, torch.float32, "genomes")
        self._check_tensor(fitness, torch.float64, "fitness")
        if out is None:
            out = torch.zeros(self.exchange_bytes(n_max, k_max), dtype=torch.uint8, device=self.device)
        _lib.check(self._L.ngp_pack_elites(self._h, _p(genomes), _p(fitness), genomes.shape[0], k, n_max, k_max, _p(out), _stream(self.device)),
                   "ngp_pack_elites")
        return out

    def unpack_elites(self, gathered: torch.Tensor, world: int, n_max: int, k_max: int, n_total: int, k_total: int):
        self._check_tensor(gathered, torch.uint8, "gathered")
        assert gathered.numel() == world * self.exchange_bytes(n_max, k_max)
        fit = torch.empty(n_total, dtype=torch.float64, device=self.device)
        eg = torch.empty((k_total, self.gene_size), dtype=torch.float32, device=self.device)
        ef = torch.empty(k_total, dtype=torch.float64, device=self.device)
        _lib.check(self._L.ngp_unpack_elites(self._h, _p(gathered), world, n_max, k_max, _p(fit), _p(eg), _p(ef), _stream(self.device)),
                   "ngp_unpack_elites")
        return fit, eg, ef
