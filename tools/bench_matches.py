"""Throughput of ngp_play_matches (explicit match lists) on one GPU, CUDA-event timed with every shape warmed first.

1. config 2's pairing (1 024 genomes x 6 round-robin games) through ngp_evaluate and through ngp_play_matches with the same
   list, alternating the two; rewards and frame counts must be identical;
2. a 128 x 128 cross_play (16 384 games: the CTA-synchronous flavour) and 1 024 genomes against the three scripted opponents.
Prints one JSON line per workload (env-frames/s, ms per call) after a line with the card's name and power limit.
usage: python tools/bench_matches.py [--reps 3]"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import neuro_genetic_pong_self_play_b200 as ngp  # noqa: E402
from neuro_genetic_pong_self_play_b200 import reference_api as ref  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    return {"card": torch.cuda.get_device_name(0), "nvidia_smi": q}


def timed(fn):
    """(result, milliseconds) of one call, CUDA events on the current stream."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    b.synchronize()
    return out, a.elapsed_time(b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    print(json.dumps(card()), flush=True)
    n, games, seed = 1024, 6, 1
    eng = ngp.Engine(ngp.Config(SCHEDULE=ngp.SCHEDULE_ROUND_ROBIN, GAMES_TO_PLAY=games, POPULATION_SIZE=n), device=0)
    pop = eng.init_population(n, seed=0)
    dev = eng.device
    g = torch.arange(n, dtype=torch.int32, device=dev).repeat_interleave(games)            # match m = genome * games + game
    k = torch.arange(games, dtype=torch.int32, device=dev).repeat(n)
    right, left = g, ((g + k + 1) % n).to(torch.int32)

    def evaluate(gen):
        return eng.evaluate(pop, seed=seed, generation=gen, want_detail=True)

    def matches(gen):
        return eng.play_matches(pop, right, left, seed=seed, generation=gen)

    evaluate(0); matches(0)                                                                 # warm both shapes
    rows = {"evaluate": [], "play_matches": []}
    frames = {"evaluate": [], "play_matches": []}
    for rep in range(args.reps):
        gen = 1 + rep                                                                       # other fall-back keys every rep
        ev, t_ev = timed(lambda: evaluate(gen))
        pm, t_pm = timed(lambda: matches(gen))
        if not (torch.equal(pm["rewards"], ev["rewards"].reshape(-1)) and torch.equal(pm["frames"], ev["frames"].reshape(-1))):
            raise SystemExit(f"rep {rep}: ngp_play_matches differs from ngp_evaluate on the round-robin list")
        rows["evaluate"].append(t_ev); rows["play_matches"].append(t_pm)
        frames["evaluate"].append(ev["frames_total"]); frames["play_matches"].append(pm["frames_total"])
    for name in rows:
        ms = rows[name]
        print(json.dumps({"workload": f"config 2 pairing (1024 x 6 round robin) via {name}", "ms": [round(t, 2) for t in ms],
                          "env_frames_per_s": [round(f / (t / 1e3)) for f, t in zip(frames[name], ms)], "identical": True}), flush=True)

    # a 128 x 128 cross table and the whole population against the scripted opponents (reference-schedule engine)
    eng_r = ngp.Engine(ngp.Config(POPULATION_SIZE=n), device=0)
    tb = ref.Toolbox(eng_r.config, engine=eng_r, seed=seed)
    a, b = eng_r.init_population(128, seed=3), eng_r.init_population(128, seed=4)
    pop_r = eng_r.init_population(n, seed=5)
    codes = torch.tensor([ngp.OPP_HARDCODED, ngp.OPP_SCORE_HARDCODED, ngp.OPP_ROBOT], dtype=torch.int32, device=dev)
    r3 = torch.arange(n, dtype=torch.int32, device=dev).repeat_interleave(3)
    l3 = codes.repeat(n)

    def cross():
        out = ref.cross_play(tb, a, b)
        return int(out["frames"].sum().item())

    def scripted():
        return eng_r.play_matches(pop_r, r3, l3, seed=seed, generation=tb.generation)["frames_total"]

    for name, fn, count in (("cross_play 128 x 128", cross, 128 * 128), ("1024 genomes x 3 scripted opponents", scripted, 3 * n)):
        fn()
        ms, fr = [], []
        for rep in range(args.reps):
            tb.generation = 1 + rep
            f, t = timed(fn)
            ms.append(t); fr.append(f)
        print(json.dumps({"workload": name, "matches": count, "ms": [round(t, 2) for t in ms],
                          "env_frames_per_s": [round(f / (t / 1e3)) for f, t in zip(fr, ms)]}), flush=True)
    print(json.dumps(card()), flush=True)


if __name__ == "__main__":
    main()
