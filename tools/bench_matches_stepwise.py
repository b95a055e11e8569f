"""Throughput of ngp_play_matches_stepwise (match lists on the per-frame driver) on one GPU, CUDA-event timed with every shape
warmed first.

1. config 4's pairing ([6,512,512,2], 256 genomes x 64 round-robin games) through ngp_evaluate and through the list, alternated;
   rewards, frame counts and frames_total must be identical; the ratio list / evaluate is reported;
2. a [6,512,512,2] 128 x 128 cross table (reference_api.cross_play);
3. the skewed list: one [6,512,512,2] champion against 1 024 genomes;
4. config 2's pairing ([6,2,2], 1 024 genomes x 6 round-robin games), fused against stepwise, alternated; identical required.
For each wide list: the chunk size T, the chunk count C and the padding fraction of the row layout (computed here from the
lists by the library's rule); for every list ms per call and ms per frame (the driver runs max(frames) frames).  One JSON line
per workload, after a line with the card's name and power limit.
usage: python tools/bench_matches_stepwise.py [--reps 2]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import neuro_genetic_pong_self_play_b200 as ngp  # noqa: E402
from neuro_genetic_pong_self_play_b200 import reference_api as ref  # noqa: E402

WIDE = (6, 512, 512, 2)


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


def layout(right, left, n_genomes):
    """(T, C, padding fraction) of ngp_play_matches_stepwise's row layout for these lists (include/ngp.h)"""
    r, l = right.cpu().numpy(), left.cpu().numpy()
    counts = np.bincount(np.concatenate([r, l[l >= 0]]), minlength=n_genomes)
    rows, used = int(counts.sum()), int((counts > 0).sum())
    T = 16
    while T < 128 and T * used < rows:
        T *= 2
    C = int(((counts + T - 1) // T).sum())
    return T, C, round(1.0 - rows / (C * T), 4)


def report(name, right, left, n_genomes, ms, frames, wide=True, **extra):
    row = {"workload": name, "matches": int(right.shape[0])}
    if wide:                                             # networks the fused rollout takes run no batched MLP: no row layout
        row.update(zip(("T", "C", "padding"), layout(right, left, n_genomes)))
    row.update(ms=[round(t, 1) for t in ms], frames=frames, ms_per_frame=[round(t / frames, 4) for t in ms])
    row.update(extra)
    print(json.dumps(row), flush=True)


def round_robin(n, games, dev):
    g = torch.arange(n, dtype=torch.int32, device=dev).repeat_interleave(games)
    k = torch.arange(games, dtype=torch.int32, device=dev).repeat(n)
    return g, ((g + k + 1) % n).to(torch.int32)


def alternate(reps, a, b, same):
    """alternated timings of a() and b(); same(out_a, out_b) must hold every time"""
    a(0); b(0)
    ta, tb, last = [], [], None
    for rep in range(reps):
        oa, t1 = timed(lambda: a(1 + rep))
        ob, t2 = timed(lambda: b(1 + rep))
        if not same(oa, ob):
            raise SystemExit(f"rep {rep}: the two paths differ")
        ta.append(t1); tb.append(t2); last = ob
    return ta, tb, last


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=2)
    args = ap.parse_args()
    print(json.dumps(card()), flush=True)
    dev = torch.device("cuda", 0)

    # 1. config 4's pairing: ngp_evaluate against the same games as a list
    n, games = 256, 64
    eng = ngp.Engine(ngp.Config(SCHEDULE=ngp.SCHEDULE_ROUND_ROBIN, GAMES_TO_PLAY=games, POPULATION_SIZE=n, NETWORK_SHAPE=WIDE), device=0)
    pop = eng.init_population(n, seed=0)
    right, left = round_robin(n, games, dev)

    def same_ev(ev, pm):
        return (torch.equal(pm["rewards"], ev["rewards"].reshape(-1)) and torch.equal(pm["frames"], ev["frames"].reshape(-1))
                and pm["frames_total"] == ev["frames_total"])

    t_ev, t_pm, pm = alternate(args.reps, lambda gen: eng.evaluate(pop, seed=1, generation=gen, want_detail=True),
                               lambda gen: eng.play_matches(pop, right, left, seed=1, generation=gen), same_ev)
    frames = int(pm["frames"].max().item())
    print(json.dumps({"workload": "config 4 pairing via ngp_evaluate", "ms": [round(t, 1) for t in t_ev], "frames": frames,
                      "ms_per_frame": [round(t / frames, 4) for t in t_ev]}), flush=True)
    report("config 4 pairing (256 x 64 round robin, [6,512,512,2]) via ngp_play_matches_stepwise", right, left, n, t_pm, frames,
           identical=True, ratio_list_over_evaluate=[round(b / a, 3) for a, b in zip(t_ev, t_pm)])
    eng.close()

    # 2. and 3. a wide cross table and one champion against 1 024 genomes (reference-schedule engine: the lists alone decide)
    eng = ngp.Engine(ngp.Config(NETWORK_SHAPE=WIDE), device=0)
    tb = ref.Toolbox(eng.config, engine=eng, seed=1)
    a, b = eng.init_population(128, seed=3), eng.init_population(128, seed=4)
    rows = torch.arange(256, dtype=torch.int32, device=dev)
    cr, cl = rows[:128].repeat_interleave(128), rows[128:].repeat(128)
    champ = eng.init_population(1025, seed=5)
    sr = torch.zeros(1024, dtype=torch.int32, device=dev)
    sl = torch.arange(1, 1025, dtype=torch.int32, device=dev)
    for name, fn, r, l, ng in (("cross table 128 x 128, [6,512,512,2]", lambda: ref.cross_play(tb, a, b)["frames"], cr, cl, 256),
                               ("skewed: 1 champion vs 1024 genomes, [6,512,512,2]",
                                lambda: eng.play_matches(champ, sr, sl, seed=1, generation=tb.generation)["frames"], sr, sl, 1025)):
        fn()
        ms, fr = [], 0
        for rep in range(args.reps):
            tb.generation = 1 + rep
            f, t = timed(fn)
            ms.append(t); fr = max(fr, int(f.max().item()))
        report(name, r, l, ng, ms, fr)
    eng.close()

    # 4. config 2's pairing on both drivers
    n, games = 1024, 6
    eng = ngp.Engine(ngp.Config(SCHEDULE=ngp.SCHEDULE_ROUND_ROBIN, GAMES_TO_PLAY=games, POPULATION_SIZE=n), device=0)
    pop = eng.init_population(n, seed=0)
    right, left = round_robin(n, games, dev)

    def same(x, y):
        return all(torch.equal(x[k], y[k]) for k in ("rewards", "frames", "scores")) and x["frames_total"] == y["frames_total"]

    t_f, t_s, pm = alternate(args.reps, lambda gen: eng.play_matches(pop, right, left, seed=1, generation=gen, driver="fused"),
                             lambda gen: eng.play_matches(pop, right, left, seed=1, generation=gen, driver="stepwise"), same)
    frames = int(pm["frames"].max().item())
    print(json.dumps({"workload": "config 2 pairing (1024 x 6 round robin, [6,2,2]) via the fused rollout", "ms": [round(t, 1) for t in t_f]}),
          flush=True)
    report("config 2 pairing (1024 x 6 round robin, [6,2,2]) via ngp_play_matches_stepwise (no batched MLP)", right, left, n, t_s,
           frames, wide=False, identical=True, ratio_stepwise_over_fused=[round(b / a, 3) for a, b in zip(t_f, t_s)])
    eng.close()
    print(json.dumps(card()), flush=True)


if __name__ == "__main__":
    main()
