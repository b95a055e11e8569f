"""Throughput of match sessions (Engine.session / ngp_session_step) on one GPU, CUDA-event timed after a warm-up of every shape.

1. M matches of an external right seat, driven by a torch policy that plays dumb_ais.HardcodedAi's rule on the session's obs,
   against the scripted bot (NGP_OPP_HARDCODED) on the left, for M in --sizes: stepped eagerly (policy + step on the stream,
   the running count read every 8 steps) and replayed from a CUDA graph of 8 such steps.  Both must give the same bits.
   Reported: steps, us per step, env-frames/s (frames_total over the wall time of the whole list).
2. The same list with a genome (the library's seat) on the right against the same bot, no external seat: through a session
   (all-zero actions), through ngp_play_matches_stepwise and through the fused ngp_play_matches; identical bits required.
One JSON line per measurement, after a line with the card's name and power limit.  Games stop at --max-frames env.steps.
usage: python tools/bench_session.py [--sizes 1,64,1024,6144] [--max-frames 2000] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import neuro_genetic_pong_self_play_b200 as ngp  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    return {"card": torch.cuda.get_device_name(0), "nvidia_smi": q}


def policy(obs):
    """dumb_ais.HardcodedAi (dumb_ais.py:1-8) on utils.inference's vector: up when the ball is above the paddle"""
    return torch.where(obs[..., 1] < obs[..., 4], 1, torch.where(obs[..., 1] > obs[..., 4], 2, 0)).to(torch.uint8)


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    b.synchronize()
    return out, a.elapsed_time(b)


def play_eager(eng, right, left):
    s = eng.session(None, right, left, seed=1)
    acts = torch.zeros((right.shape[0], 2), dtype=torch.uint8, device="cuda")
    steps = 0
    while steps % 8 or s.running():
        acts[:, 1] = policy(s.obs[:, 1])
        s.step(acts)
        steps += 1
    out = s.result()
    s.close()
    return out, steps


def play_graph(eng, right, left, per_graph=8):
    s = eng.session(None, right, left, seed=1)
    acts = torch.zeros((right.shape[0], 2), dtype=torch.uint8, device="cuda")
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(per_graph):
            acts[:, 1] = policy(s.obs[:, 1])
            s.step(acts)
    steps = 0
    while s.running():                                   # the capture itself ran nothing
        graph.replay()
        steps += per_graph
    out = s.result()
    s.close()
    return out, steps


def same(a, b, what):
    for k in ("rewards", "frames", "scores"):
        assert torch.equal(a[k], b[k]), (what, k)
    assert a["frames_total"] == b["frames_total"], what


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1,64,1024,6144")
    ap.add_argument("--max-frames", type=int, default=2000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = [json.dumps(card())]
    print(lines[0], flush=True)

    def emit(row):
        lines.append(json.dumps(row))
        print(lines[-1], flush=True)

    eng = ngp.Engine(ngp.Config(MAX_FRAMES=args.max_frames), device=0)
    genome = torch.as_tensor((np.random.RandomState(0).standard_normal((1, eng.gene_size)) * 2).astype(np.float32)).cuda()
    for M in (int(v) for v in args.sizes.split(",")):
        ext = torch.full((M,), ngp.PLAYER_EXTERNAL, dtype=torch.int32, device="cuda")
        bot = torch.full((M,), ngp.OPP_HARDCODED, dtype=torch.int32, device="cuda")
        play_eager(eng, ext, bot)                         # warm-up: modules, allocator, the graph's kernels
        play_graph(eng, ext, bot)
        (ea, ea_steps), ea_ms = timed(lambda: play_eager(eng, ext, bot))
        (gr, gr_steps), gr_ms = timed(lambda: play_graph(eng, ext, bot))
        same(ea, gr, ("graph", M))
        ft = ea["frames_total"]
        for mode, steps, ms in (("eager", ea_steps, ea_ms), ("graph", gr_steps, gr_ms)):
            emit({"workload": "external seat (torch policy) vs bot", "mode": mode, "matches": M, "steps": steps, "frames_total": ft,
                  "ms": round(ms, 3), "us_per_step": round(1e3 * ms / steps, 2), "env_frames_per_s": round(ft / (ms / 1e3))})
        # the library's seat: a genome against the same bot through the three drivers
        right = torch.zeros((M,), dtype=torch.int32, device="cuda")

        def session():
            s = eng.session(genome, right, bot, seed=1)
            zeros = torch.zeros((M, 2), dtype=torch.uint8, device="cuda")
            steps = 0
            while steps % 8 or s.running():
                s.step(zeros)
                steps += 1
            out = s.result()
            s.close()
            return out

        runs = {"session": session,
                "stepwise": lambda: eng.play_matches(genome, right, bot, seed=1, driver="stepwise"),
                "fused": lambda: eng.play_matches(genome, right, bot, seed=1, driver="fused")}
        for fn in runs.values():
            fn()
        res = {name: timed(fn) for name, fn in runs.items()}
        for name, (out, ms) in res.items():
            same(out, res["fused"][0], (name, M))
            emit({"workload": "genome vs bot", "driver": name, "matches": M, "frames_total": out["frames_total"], "ms": round(ms, 3),
                  "env_frames_per_s": round(out["frames_total"] / (ms / 1e3))})
    eng.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
