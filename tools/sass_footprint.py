#!/usr/bin/env python3
"""Instruction footprint of the fused rollout kernel, per source region, static and per frame (CPU only, no GPU).

Static side: the SASS of one `rollout_kernel` instantiation (default `<1,false,256>`, the one-warp flavour of the named
workload) from an object built with `-lineinfo` (`build.py` builds with it), disassembled with `nvdisasm -gi`.  Every
instruction (16 bytes) is attributed by its inline chain:
  entry $XXXX     code of a generated dispatch entry (`generated/pong_core.inc`, split further per 6507 instruction)
  sb:<name>       a hand-fused super-block (`pong_superblocks.cuh`); `replay` code inside it is counted in its own row
  fn:<name>       an out-of-line (`__noinline__`) renderer / TIA / policy function
  dispatcher      `run_frame_compiled` around the switch
  episode         episode bookkeeping, observation, policy glue, persistent-lane loop
`CALL` sites and the local-memory traffic next to them (`LDL`/`STL` within 6 instructions of a `CALL`) are counted per region.

Dynamic side: the same sources compiled for the CPU (`tests/host_sim`) with a counter at every translated 6507 instruction
(inserted into a temporary copy of `pong_core.inc`; the product's file is untouched) and the `A26_STATS` event counters,
playing `--frames` self-play frames from `Start.2P` with both paddles driven by random up/down/none decisions held for four
frames (the kind of input the bench's policies produce).  A 6507 instruction or a super-block counts as reached in a frame
when it ran at least once in it.  Dispatcher, episode code and the out-of-line functions run every frame.

Reported: static bytes; hot bytes = bytes reached in an average frame (each region weighted by the fraction of frames that
reach it); bytes reached in at least one of the frames.
"""
from __future__ import annotations

import argparse
import collections
import ctypes
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "neuro_genetic_pong_self_play_b200")
CSRC = os.path.join(PKG, "csrc")
INC = os.path.join(CSRC, "generated", "pong_core.inc")

def _rollout(sync, maxt, rec):
    """mangled name of rollout_kernel<1, sync, maxt, rec>(RolloutParams, RecordArgs) (csrc/rollout_kernel.cuh)"""
    return f"_Z14rollout_kernelILi1ELb{int(sync)}ELi{maxt}ELb{int(rec)}EEvN4roll13RolloutParamsENS0_10RecordArgsE"


# translated-core flavours (ngp_core.cu) and their recording twins (rec_*, ngp_record.cu: ngp_record_matches)
KERNELS = {"cfg2": _rollout(0, 256, 0), "sync256": _rollout(1, 256, 0), "sync384": _rollout(1, 384, 0), "sync512": _rollout(1, 512, 0),
           "rec_cfg2": _rollout(0, 256, 1), "rec_sync256": _rollout(1, 256, 1), "rec_sync384": _rollout(1, 384, 1),
           "rec_sync512": _rollout(1, 512, 1)}


def default_object(kernel_key):
    return os.path.join(PKG, "build", ("ngp_record" if kernel_key.startswith("rec_") else "ngp_core") + ".cu.o")
NVCC = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
CUDA_BIN = os.path.dirname(NVCC)


def tool(name):
    return shutil.which(name) or os.path.join(CUDA_BIN, name)


# ---- generated code: pong_core.inc line -> (dispatch entry, 6507 instruction) ------------------------------------------
def inc_line_map():
    entry_of, insn_of = {}, {}
    entry = insn = None
    for i, line in enumerate(open(INC), 1):
        m = re.match(r"case \d+:.*/\* ---- ([0-9A-F]{4}) ---- \*/", line)
        if m:
            entry = insn = int(m.group(1), 16)
        m = re.match(r"\s*\{ /\* ([0-9A-F]{4}): ", line)
        if m:
            insn = int(m.group(1), 16)
        entry_of[i], insn_of[i] = entry, insn
    return entry_of, insn_of


def superblock_line_map():
    """pong_superblocks.cuh line -> (enclosing top-level function, enclosing lambda or None)."""
    fn_of, cur, lam, lam_end = {}, None, None, None
    for i, line in enumerate(open(os.path.join(CSRC, "pong_superblocks.cuh")), 1):
        m = re.match(r"__device__ .*?\b(\w+)\(", line)
        if m:
            cur = m.group(1)
        m = re.match(r"(\s*)auto (\w+) = \[&\]", line)
        if m:
            lam, lam_end = m.group(2), m.group(1) + "};"
        fn_of[i] = (cur, lam)
        if lam and line.startswith(lam_end):
            lam = None
    return fn_of


# ---- static side ------------------------------------------------------------------------------------------------------
LOC = re.compile(r'File "([^"]+)", line (\d+)')
INSN = re.compile(r"^\s+/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;")


def disassemble(obj, kernel, workdir):
    subprocess.check_call([tool("cuobjdump"), "-xelf", "all", obj], cwd=workdir, stdout=subprocess.DEVNULL)
    source = os.path.basename(obj).split(".")[0]                 # ngp_core.cu.o -> ngp_core.sm_100a.cubin
    cubin = [f for f in os.listdir(workdir) if f.endswith(".cubin") and source in f][0]
    sass = subprocess.run([tool("nvdisasm"), "-gi", "-c", os.path.join(workdir, cubin)], check=True, capture_output=True,
                          text=True).stdout.splitlines()
    start = next((i for i, l in enumerate(sass) if l.startswith(f".text.{kernel}:")), None)
    if start is None:
        raise SystemExit(f"{kernel} is not in {obj}: the kernel's signature changed, update KERNELS")
    end = next((i for i in range(start + 1, len(sass)) if sass[i].lstrip().startswith(".section")), len(sass))
    out, fn, chain, pending = [], "kernel", [], []
    for line in sass[start:end]:
        m = re.match(r"^\$" + re.escape(kernel) + r"\$(\S+):$", line)
        if m:
            fn = m.group(1)
            continue
        if line.lstrip().startswith("//##"):
            pending += [(os.path.basename(f), int(n)) for f, n in LOC.findall(line)]
            continue
        m = INSN.match(line)
        if m:
            if pending:
                chain, pending = pending, []
            op = m.group(2).split()[0] if not m.group(2).startswith("@") else m.group(2).split()[1]
            out.append((fn, chain, op.split(".")[0]))
    return out


FN_NAMES = re.compile(r"(render_span_quick|render_span|render_black_span|tia_catchup|tia_peek_cx|io_read_slow|io_write_slow|tia_poke_changed|player_mask|"
                      r"missile_mask|catchup_quick|mlp_small_f64|dblrcp)")


def attribute(insns, entry_of, insn_of, sb_fn):
    """-> list of (region, sub, op): region as in the module docstring; sub = 6507 instruction (entries) or '' ."""
    res = []
    for fn, chain, op in insns:
        if fn != "kernel":
            m = FN_NAMES.search(fn)
            res.append(("fn:" + (m.group(1) if m else fn), "", op))
            continue
        inc = [n for f, n in chain if f == "pong_core.inc"]
        sbl = [n for f, n in chain if f == "pong_superblocks.cuh"]
        if sbl:
            outer = sb_fn.get(sbl[-1], ("?", None))[0]
            lams = [sb_fn.get(n, (None, None))[1] for n in sbl]
            res.append(("sb:" + outer, "replay" if "replay" in lams else "", op))
        elif inc:
            n = inc[0]
            res.append((f"entry ${entry_of.get(n) or 0:04X}", insn_of.get(n) or 0, op))
        elif any(f == "a26_compiled.cuh" for f, _ in chain):
            res.append(("dispatcher", "", op))
        else:
            res.append(("episode", "", op))
    return res


def callsite_traffic(ops, window=6):
    """indices of LDL/STL within `window` instructions of a CALL (caller-side save/restore)."""
    calls = [i for i, o in enumerate(ops) if o == "CALL"]
    near = set()
    for c in calls:
        for j in range(max(0, c - window), min(len(ops), c + window + 1)):
            if ops[j] in ("LDL", "STL"):
                near.add(j)
    return near


# ---- dynamic side -----------------------------------------------------------------------------------------------------
def build_counting_sim(tmp):
    """tests/host_sim with a counter at every translated 6507 instruction (temporary copy of the sources)."""
    for sub in ("tests/host_sim", "include"):
        shutil.copytree(os.path.join(ROOT, sub), os.path.join(tmp, sub), ignore=shutil.ignore_patterns("*.so"))
    shutil.copytree(CSRC, os.path.join(tmp, "neuro_genetic_pong_self_play_b200", "csrc"))
    inc = os.path.join(tmp, "neuro_genetic_pong_self_play_b200", "csrc", "generated", "pong_core.inc")
    src = open(inc).read()
    # a statement right after the opening brace of every instruction block: same line count, lines unchanged otherwise
    src = re.sub(r"(\{ /\* ([0-9A-F]{4}): [^\n]*?\*/)", r"\1 ++fp_insn_count[0x\2 & 0x7FF];", src)
    open(inc, "w").write(src)
    shim = os.path.join(tmp, "tests", "host_sim", "fp_counts.cpp")
    open(shim, "w").write("unsigned long long fp_insn_count[2048];\n"
                          'extern "C" unsigned long long *fp_counts() { return fp_insn_count; }\n')
    pre = os.path.join(tmp, "fp_pre.h")
    open(pre, "w").write("extern unsigned long long fp_insn_count[2048];\n")
    lib = os.path.join(tmp, "libfp.so")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-Wno-unknown-pragmas",
                           "-DA26_STATS", "-include", pre, "-o", lib, os.path.join(tmp, "tests", "host_sim", "host_sim.cpp"),
                           os.path.join(tmp, "tests", "host_sim", "host_sim_stats.cpp"), shim])
    return lib


def frame_profile(frames, seed):
    """-> (list of per-frame sets of executed 6507 instruction addresses, list of per-frame super-block call counts)."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import oracle
    with tempfile.TemporaryDirectory() as tmp:
        L = ctypes.CDLL(build_counting_sim(tmp))
        vp = ctypes.c_void_p
        L.hs_create.restype = vp
        L.hs_env_reset.argtypes = [vp, ctypes.c_int]
        L.hs_env_step_fast.argtypes = [vp, ctypes.c_int] + [vp] * 4
        L.fp_counts.restype = ctypes.POINTER(ctypes.c_ulonglong * 2048)
        L.hs_stats.restype = ctypes.POINTER(ctypes.c_ulonglong * 16)
        sim = vp(L.hs_create(oracle.load_rom()))
        L.hs_env_reset(sim, 1)                                   # Start.2P
        cnt, st = L.fp_counts().contents, L.hs_stats().contents
        rng = np.random.RandomState(seed)
        ram = np.zeros(128, np.uint8); loc = np.zeros(6); valid = np.zeros(3, np.uint8)
        act = np.zeros(16, np.uint8)
        per_frame, sb = [], []
        P = lambda a: a.ctypes.data_as(vp)  # noqa: E731
        for f in range(frames):
            if f % 4 == 0:
                act = np.zeros(16, np.uint8); act[0] = act[15] = 1     # BLANK_ACTION + the two decisions (main.py:91-92)
                r, l = rng.randint(0, 3), rng.randint(0, 3)
                act[4] = r == 1; act[5] = r == 2; act[6] = l == 1; act[7] = l == 2
            for i in range(2048):
                cnt[i] = 0
            for i in range(16):
                st[i] = 0
            assert L.hs_env_step_fast(sim, 1, P(act), P(ram), P(loc), P(valid)) == 0
            per_frame.append({0xF000 | i for i in range(2048) if cnt[i]})
            sb.append({"sb:superblock_f621": st[6], "sb:superblock_f58d": st[7], "sb:superblock_f5cc": st[8]})
        return per_frame, sb


# ---- report -------------------------------------------------------------------------------------------------------------
def report(obj, kernel_key, frames, seed):
    entry_of, insn_of = inc_line_map()
    with tempfile.TemporaryDirectory() as tmp:
        insns = disassemble(obj, KERNELS[kernel_key], tmp)
    attr = attribute(insns, entry_of, insn_of, superblock_line_map())
    ops = [o for _, _, o in attr]
    near = callsite_traffic(ops)
    per_frame, sb = frame_profile(frames, seed) if frames else ([], [])
    n = max(len(per_frame), 1)

    def reach(region, sub):
        """fraction of frames that execute this code, and whether any does"""
        if region.startswith("entry"):
            k = sum(1 for s in per_frame if sub in s)
            return k / n, k > 0
        if region.startswith("sb:"):
            k = sum(1 for s in sb if s.get(region, 0))
            return k / n, k > 0
        return 1.0, True

    rows = collections.OrderedDict()
    tot = collections.Counter()
    for i, (region, sub, op) in enumerate(attr):
        key = region + (" (replay)" if sub == "replay" else "")
        r = rows.setdefault(key, collections.Counter())
        frac, anyf = reach(region, sub) if per_frame else (0.0, False)
        for c in (r, tot):
            c["bytes"] += 16
            c["hot_bytes"] += 16 * frac
            c["any_bytes"] += 16 * anyf
            c["CALL"] += op == "CALL"
            c["LDL_STL"] += op in ("LDL", "STL")
            c["callsite_LDL_STL"] += i in near
            c["hot_CALL"] += (op == "CALL") * frac
            c["hot_callsite_LDL_STL"] += (i in near) * frac
    # the generated entries as one row; the 25 with the most hot bytes are listed in the JSON report
    entries = {k: v for k, v in rows.items() if k.startswith("entry")}
    groups = collections.OrderedDict()
    for k, v in rows.items():
        g = "generated entries (all)" if k.startswith("entry") else k
        groups.setdefault(g, collections.Counter()).update(v)
    return {"kernel": KERNELS[kernel_key], "object": os.path.relpath(obj, ROOT), "frames": len(per_frame), "seed": seed,
            "total": {k: round(v, 1) for k, v in tot.items()},
            "regions": {k: {kk: round(vv, 1) for kk, vv in v.items()} for k, v in groups.items()},
            "entries_by_hot_bytes": {k: {kk: round(vv, 1) for kk, vv in v.items()}
                                     for k, v in sorted(entries.items(), key=lambda kv: -kv[1]["hot_bytes"])[:25]},
            "entries_reached_per_frame": round(sum(len(s) for s in per_frame) / n, 1)}


def print_table(r):
    print(f"{r['kernel']}  ({r['object']}; {r['frames']} self-play frames from Start.2P, seed {r['seed']})")
    print(f"{'region':34s} {'bytes':>9s} {'hot B/frame':>12s} {'B in >=1 frame':>15s} {'CALL':>6s} {'LDL/STL':>8s} "
          f"{'at CALL':>8s} {'hot CALL':>9s}")
    for k, v in list(r["regions"].items()) + [("TOTAL", r["total"])]:
        print(f"{k:34s} {v['bytes']:9.0f} {v['hot_bytes']:12.0f} {v['any_bytes']:15.0f} {v['CALL']:6.0f} {v['LDL_STL']:8.0f} "
              f"{v['callsite_LDL_STL']:8.0f} {v['hot_CALL']:9.1f}")
    print(f"6507 instructions reached per frame (translated, outside super-blocks): {r['entries_reached_per_frame']}")


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--object", help="object built with -lineinfo that holds the kernel (default: the ngp_core.cu / ngp_record.cu "
                                     "object build.py leaves; built if missing)")
    ap.add_argument("--kernel", default="cfg2", choices=sorted(KERNELS))
    ap.add_argument("--frames", type=int, default=400)
    ap.add_argument("--seed", type=int, default=7)
    ap.add_argument("--json", help="write the full report here")
    a = ap.parse_args()
    a.object = a.object or default_object(a.kernel)
    if not os.path.exists(a.object):
        sys.path.insert(0, ROOT)
        from neuro_genetic_pong_self_play_b200 import build
        build.build()
    r = report(os.path.abspath(a.object), a.kernel, a.frames, a.seed)
    print_table(r)
    if a.json:
        with open(a.json, "w") as f:
            json.dump(r, f, indent=1)


if __name__ == "__main__":
    main()
