"""Cost of recording per-frame traces (ngp_record_matches) over ngp_play_matches on one GPU, CUDA-event timed with every
shape warmed first.  The two calls alternate on the same list and must give identical rewards, frames and scores.

1. config 2's pairing (1 024 genomes x 6 round-robin games) with max_record = 2048;
2. a 128 x 128 cross table (16 384 games: the CTA-synchronous flavour).
Prints one JSON line per workload (ms per call, env-frames/s, record / play ratio, record bytes written) between two lines
with the card's name and power limit.
usage: python tools/bench_record.py [--reps 7]"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import neuro_genetic_pong_self_play_b200 as ngp  # noqa: E402


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


def compare(name, eng, genomes, right, left, max_record, reps, seed):
    play = lambda gen: eng.play_matches(genomes, right, left, seed=seed, generation=gen)                          # noqa: E731
    rec = lambda gen: eng.record_matches(genomes, right, left, max_record=max_record, seed=seed, generation=gen)  # noqa: E731
    play(0); rec(0)                                                                                 # warm both shapes and buffers
    ms = {"play_matches": [], "record_matches": []}
    frames, written = [], []
    for rep in range(reps):
        gen = 1 + rep                                                                               # other fall-back keys every rep
        # the previous repetition's outputs (the record buffer is up to ~1 GB) are released before the timed calls, so that
        # every call finds its buffers in the caching allocator instead of allocating a new block inside the timed window
        pm = rm = None
        pm, t_pm = timed(lambda: play(gen))
        rm, t_rm = timed(lambda: rec(gen))
        for k in ("rewards", "frames", "scores"):
            if not torch.equal(pm[k], rm[k]):
                raise SystemExit(f"{name} rep {rep}: ngp_record_matches' {k} differ from ngp_play_matches'")
        if pm["frames_total"] != rm["frames_total"]:
            raise SystemExit(f"{name} rep {rep}: frames_total differs")
        ms["play_matches"].append(t_pm); ms["record_matches"].append(t_rm)
        frames.append(pm["frames_total"])
        written.append(int(torch.clamp(rm["frames"], max=max_record).sum().item()) * ngp._lib.NGP_FRAME_RECORD_BYTES)
    ratio = [r / p for r, p in zip(ms["record_matches"], ms["play_matches"])]
    med = sorted(ratio)[len(ratio) // 2]
    print(json.dumps({"workload": name, "matches": int(right.shape[0]), "max_record": max_record,
                      "ms": {k: [round(t, 2) for t in v] for k, v in ms.items()},
                      "env_frames_per_s": {k: [round(f / (t / 1e3)) for f, t in zip(frames, v)] for k, v in ms.items()},
                      "record_over_play": [round(x, 4) for x in ratio], "median_record_over_play": round(med, 4),
                      "record_bytes_written": written, "identical": True}),
          flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    print(json.dumps(card()), flush=True)
    n, games, seed = 1024, 6, 1
    eng = ngp.Engine(ngp.Config(SCHEDULE=ngp.SCHEDULE_ROUND_ROBIN, GAMES_TO_PLAY=games, POPULATION_SIZE=n), device=0)
    dev = eng.device
    pop = eng.init_population(n, seed=0)
    g = torch.arange(n, dtype=torch.int32, device=dev).repeat_interleave(games)                    # match m = genome * games + game
    k = torch.arange(games, dtype=torch.int32, device=dev).repeat(n)
    compare("config 2 pairing (1024 x 6 round robin)", eng, pop, g, ((g + k + 1) % n).to(torch.int32), 2048, args.reps, seed)

    a, b = eng.init_population(128, seed=3), eng.init_population(128, seed=4)
    rows = torch.arange(256, dtype=torch.int32, device=dev)
    compare("cross table 128 x 128", eng, torch.cat([a, b]), rows[:128].repeat_interleave(128), rows[128:].repeat(128), 2048,
            args.reps, seed)
    print(json.dumps(card()), flush=True)


if __name__ == "__main__":
    main()
