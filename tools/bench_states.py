"""Cost of save states in the fused rollout on one GPU, CUDA-event timed with every shape warmed first; compared calls
alternate.

1. Fresh starts: 1 024 genomes x 64 captured states (65 536 self-play matches started with fresh = 1 from mid-game states of
   64 other games) against the same list from the built-in start state, both through ngp_play_matches_states, and the latter
   against ngp_play_matches; and, as a control, the same list started with fresh = 1 from 64 captures at frame 0 (the built-in
   start state through the resume path: the same games, so it must give ngp_play_matches' results).  Lists from other start
   states play games of other lengths, and their lanes start from different positions, so the comparison is the time per
   emulated frame.
2. The ratio of ngp_record_matches to ngp_play_matches time on tools/bench_record.py's two workloads, measured again.
Prints one JSON line per workload between two lines with the card's name and power limit.
usage: python tools/bench_states.py [--reps 5]"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import neuro_genetic_pong_self_play_b200 as ngp  # noqa: E402
from bench_record import card, compare, timed  # noqa: E402


def fresh_starts(eng, reps, seed):
    n, s = 1024, 64
    dev = eng.device
    pop = eng.init_population(n, seed=0)
    # 64 states: games between population members, captured a third of the way in
    r0 = torch.arange(s, dtype=torch.int32, device=dev)
    l0 = ((r0 + 7) % n).to(torch.int32)
    probe = eng.play_matches(pop, r0, l0, seed=seed, generation=0)
    t = (probe["frames"] // 3).to(torch.int32).contiguous()
    states = eng.play_matches_states(pop, r0, l0, capture_at=t, seed=seed, generation=0)["capture"]
    # control: 64 captures at frame 0, i.e. the built-in start state, through the same resume path
    states0 = eng.play_matches_states(pop, r0, l0, capture_at=torch.zeros_like(t), seed=seed, generation=0)["capture"]
    right = torch.arange(n, dtype=torch.int32, device=dev).repeat_interleave(s)
    left = ((right + 1) % n).to(torch.int32)
    start = torch.arange(s, dtype=torch.int32, device=dev).repeat(n)
    calls = {
        "states_fresh": lambda gen: eng.play_matches_states(pop, right, left, states=states, start=start, fresh=True, seed=seed, generation=gen),
        "states_fresh_from_frame0": lambda gen: eng.play_matches_states(pop, right, left, states=states0, start=start, fresh=True, seed=seed,
                                                                        generation=gen),
        "states_builtin_start": lambda gen: eng.play_matches_states(pop, right, left, seed=seed, generation=gen),
        "play_matches": lambda gen: eng.play_matches(pop, right, left, seed=seed, generation=gen),
    }
    for f in calls.values():
        f(0)
    ms = {k: [] for k in calls}
    ns = {k: [] for k in calls}
    for rep in range(reps):
        outs = {}
        for k, f in calls.items():
            outs[k], t_ms = timed(lambda: f(1 + rep))
            ms[k].append(t_ms)
            ns[k].append(t_ms * 1e6 / outs[k]["frames_total"])
        for key in ("rewards", "frames", "scores"):
            for k in ("states_builtin_start", "states_fresh_from_frame0"):
                if not torch.equal(outs[k][key], outs["play_matches"][key]):
                    raise SystemExit(f"rep {rep}: {k} differs from ngp_play_matches in {key}")
    med = {k: sorted(v)[len(v) // 2] for k, v in ns.items()}
    print(json.dumps({"workload": f"fresh starts: {n} genomes x {s} captured states", "matches": int(right.shape[0]),
                      "ms": {k: [round(x, 2) for x in v] for k, v in ms.items()},
                      "ns_per_env_frame": {k: [round(x, 3) for x in v] for k, v in ns.items()},
                      "median_ns_per_env_frame": {k: round(v, 3) for k, v in med.items()},
                      "fresh_over_builtin_per_frame": round(med["states_fresh"] / med["states_builtin_start"], 4),
                      "fresh_from_frame0_over_builtin_per_frame": round(med["states_fresh_from_frame0"] / med["states_builtin_start"], 4),
                      "builtin_states_over_play_matches": round(med["states_builtin_start"] / med["play_matches"], 4)}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    print(json.dumps(card()), flush=True)
    n, games, seed = 1024, 6, 1
    eng = ngp.Engine(ngp.Config(SCHEDULE=ngp.SCHEDULE_ROUND_ROBIN, GAMES_TO_PLAY=games, POPULATION_SIZE=n), device=0)
    fresh_starts(eng, args.reps, seed)
    dev = eng.device
    pop = eng.init_population(n, seed=0)
    g = torch.arange(n, dtype=torch.int32, device=dev).repeat_interleave(games)
    k = torch.arange(games, dtype=torch.int32, device=dev).repeat(n)
    compare("config 2 pairing (1024 x 6 round robin)", eng, pop, g, ((g + k + 1) % n).to(torch.int32), 2048, args.reps, seed)
    a, b = eng.init_population(128, seed=3), eng.init_population(128, seed=4)
    rows = torch.arange(256, dtype=torch.int32, device=dev)
    compare("cross table 128 x 128", eng, torch.cat([a, b]), rows[:128].repeat_interleave(128), rows[128:].repeat(128), 2048,
            args.reps, seed)
    print(json.dumps(card()), flush=True)


if __name__ == "__main__":
    main()
