"""Straight RTS / RTI / JMP ind / BRK jumps of the translated core (tools/gen_rom_core.py): the return sites the generator emits, the
acyclicity of the direct jumps, and a counting host-sim run (A26_STATS) of the translation with and without them, frame by
frame against each other and against the oracle."""
import ctypes
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import gen_rom_core as gen  # noqa: E402

INC = os.path.join(ROOT, "neuro_genetic_pong_self_play_b200", "csrc", "generated", "pong_core.inc")
TRIPS = {"WSYNC": 9, "RTS": 10, "JMP ind": 11, "BRK/RTI": 12, "frame end": 13, "cycle cap": 14}


def _blocks(text):
    """dispatch entry -> its generated code"""
    parts = re.split(r"(?m)^case \d+: (?:L_[0-9A-F]{4}:)? ?/\* ---- ([0-9A-F]{4}) ---- \*/", text.split("#else\n", 1)[1])
    return {int(parts[i], 16): parts[i + 1] for i in range(1, len(parts), 2)}


def test_straight_returns_are_the_jsr_return_sites(tmp_path, monkeypatch):
    """Each RTS of the committed file compares the popped address with the return sites of the JSRs whose subroutine reaches
    it (each JMP ind with the vector-table targets, RTI with the BRK return sites, BRK with its vector), in that order and leaving out the refused ones, and sends any other
    address through the dispatcher."""
    rom = gen.load_rom()
    g = gen.Gen(rom)
    monkeypatch.setattr(gen, "OUT_PATH", str(tmp_path / "pong_core.inc"))
    g.generate()
    jsr = {}
    for a, (mn, mode, _, b1, b2, n) in g.instrs.items():
        if mn == "JSR":
            jsr.setdefault(b1 | b2 << 8, set()).add(a + 3)
    expect = {}
    for t, sites in jsr.items():
        for r in _reached_rts(g.instrs, t):
            expect.setdefault(r, set()).update(sites)
    assert {r: set(v) for r, v in g.return_sites.items()} == expect
    assert len(expect) == 13 and sum(1 for ins in g.instrs.values() if ins[0] == "RTS") == 14   # one RTS is never called
    found = set()
    for entry, code in _blocks(open(INC).read()).items():
        for m in re.finditer(r"\{ /\* ([0-9A-F]{4}): [0-9A-F ]+(RTS imp|JMP ind|RTI imp|BRK imp) \*/(.*?)\n  \}", code, re.S):
            pc, body = int(m.group(1), 16), m.group(3)
            straight = [int(x, 16) for x in re.findall(r"if \(pc == 0x([0-9A-F]{4})u\) goto L_\1;", body)]
            want = {"RTS imp": g.return_sites.get(pc, []), "JMP ind": gen.vector_targets(rom), "RTI imp": g.brk_returns,
                    "BRK imp": [rom[0x7FE] | rom[0x7FF] << 8]}[m.group(2)]
            assert straight == [t for t in want if (entry, t) in g.allowed], hex(pc)
            assert body.rstrip().endswith("goto a26_next_;"), hex(pc)          # any other address: the dispatcher
            found |= {(entry, t) for t in straight}
    assert found == g.allowed and len(found) >= 30


def _reached_rts(instrs, t):
    """RTS instructions reached from t along fall-through, branches and JMP abs, stepping over nested JSRs"""
    out, seen, work = set(), set(), [t]
    while work:
        a = work.pop()
        if a in seen or a not in instrs:
            continue
        seen.add(a)
        mn, mode, _, b1, b2, n = instrs[a]
        if mn == "RTS":
            out.add(a)
        elif mn in ("RTI", "BRK") or (mn == "JMP" and mode == "ind"):
            continue
        elif mn == "JMP":
            work.append(b1 | b2 << 8)
        else:
            work.append(a + n)
            if mode == "rel":
                work.append((a + 2 + (b1 - 256 if b1 > 127 else b1)) & 0xFFFF)
    return out


def test_direct_jumps_have_no_cycle_outside_in_place_loops():
    """Every `goto L_xxxx` of the committed file and every fall-through into the next entry, except backward branches (the
    in-place loops) and the single-lane WSYNC shortcut (it checks the cycle cap itself), forms an acyclic graph."""
    blocks = _blocks(open(INC).read())
    order = sorted(blocks)
    succ = {}
    for i, entry in enumerate(order):
        targets = set()
        for m in re.finditer(r"\{ /\* ([0-9A-F]{4}): [0-9A-F ]+ [A-Z]{3} (\w+) \*/(.*?)(?=\n  \{ /\*|\Z)", blocks[entry], re.S):
            pc, mode = int(m.group(1), 16), m.group(2)
            for t in (int(x, 16) for x in re.findall(r"goto L_([0-9A-F]{4})", re.sub(r"A26_AFTER_WSYNC\([^;]*;", "", m.group(3)))):
                if not (mode == "rel" and t <= pc):
                    targets.add(t)
        last = [ln for ln in blocks[entry].splitlines() if ln.strip() not in ("", "}")][-1].rstrip()
        if i + 1 < len(order) and not re.search(r"(goto \w+|A26_AFTER_WSYNC\(.*\));$", last):
            targets.add(order[i + 1])                 # falls through into the next entry
        succ[entry] = targets
    state = {}

    def visit(n):                                     # iterative DFS: a grey node met again is a cycle
        stack = [(n, iter(succ.get(n, ())))]
        state[n] = 1
        while stack:
            node, it = stack[-1]
            nxt = next(it, None)
            if nxt is None:
                state[node] = 2
                stack.pop()
            elif state.get(nxt) == 1:
                raise AssertionError(f"direct jumps loop through {node:04X} -> {nxt:04X}")
            elif nxt not in state:
                state[nxt] = 1
                stack.append((nxt, iter(succ.get(nxt, ()))))
    for n in order:
        if n not in state:
            visit(n)
    assert sum(len(v) for v in succ.values()) > 100


def test_acyclic_extension_refuses_the_closing_edge():
    assert gen.acyclic_extension([(1, 2), (2, 3)], [(3, 1), (3, 4), (4, 2), (2, 4)]) == [(3, 4), (2, 4)]
    with pytest.raises(SystemExit):
        gen.acyclic_extension([(1, 2), (2, 1)], [])


def _counting_sim(tmp, straight):
    for sub in ("tests/host_sim", "include", "neuro_genetic_pong_self_play_b200/csrc"):
        shutil.copytree(os.path.join(ROOT, sub), os.path.join(tmp, sub), ignore=shutil.ignore_patterns("*.so"))
    inc = os.path.join(tmp, "neuro_genetic_pong_self_play_b200", "csrc", "generated", "pong_core.inc")
    subprocess.check_call([sys.executable, os.path.join(ROOT, "tools", "gen_rom_core.py"), inc] + ([] if straight else ["--no-straight-returns"]),
                          stdout=subprocess.DEVNULL)
    lib = os.path.join(tmp, "libtrips.so")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-DA26_STATS", "-o", lib,
                           os.path.join(tmp, "tests", "host_sim", "host_sim.cpp"), os.path.join(tmp, "tests", "host_sim", "host_sim_stats.cpp")])
    L = ctypes.CDLL(lib)
    vp = ctypes.c_void_p
    L.hs_create.restype = vp
    L.hs_env_reset.argtypes = [vp, ctypes.c_int]
    L.hs_env_step.argtypes = [vp, ctypes.c_int] + [vp] * 7
    L.hs_stats.restype = ctypes.POINTER(ctypes.c_ulonglong * 16)
    return L, vp(L.hs_create(oracle.load_rom()))


def dispatch_trips(tmp, frames=400, seed=7):
    """Self-play frames from Start.2P with random held paddle decisions (the input tools/sass_footprint.py plays), on the
    translation with and without straight returns; every frame must give the same RAM, registers, pixels and observation
    on both and on the oracle.  Returns {variant: per-frame trip counts by cause}."""
    sims = {k: _counting_sim(os.path.join(tmp, k), k == "straight") for k in ("straight", "dispatcher")}
    for L, sim in sims.values():
        L.hs_env_reset(sim, 1)
    env = oracle.Atari()
    env.reset_to_state(1)
    rng = np.random.RandomState(seed)
    act = np.zeros(16, np.uint8)
    totals = {k: np.zeros(16) for k in sims}
    P = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    for f in range(frames):
        if f % 4 == 0:
            act = np.zeros(16, np.uint8); act[0] = act[15] = 1
            r, l = rng.randint(0, 3), rng.randint(0, 3)
            act[4] = r == 1; act[5] = r == 2; act[6] = l == 1; act[7] = l == 2
        ofb = env.step(act)
        for k, (L, sim) in sims.items():
            st = L.hs_stats().contents
            for i in range(16):
                st[i] = 0
            ram = np.zeros(128, np.uint8); fb = np.zeros((210, 160), np.uint8); loc = np.zeros(6); valid = np.zeros(3, np.uint8)
            regs = np.zeros(8, np.uint8); dig = np.zeros(8, np.uint32)
            assert L.hs_env_step(sim, 1, P(act), P(ram), P(fb), P(loc), P(valid), P(regs), P(dig)) == 0
            assert np.array_equal(env.ram, ram), (k, f)
            assert np.array_equal(env.cpu_regs[:7], regs[:7]), (k, f)
            assert np.array_equal(ofb, fb), (k, f)
            totals[k] += np.array(st[:16], dtype=np.float64)
            if k == "straight":
                ref = (loc.copy(), valid.copy())
            else:
                assert np.array_equal(ref[0], loc) and np.array_equal(ref[1], valid), f
    out = {}
    for k, t in totals.items():
        row = {name: t[i] / frames for name, i in TRIPS.items()}
        row["other"] = (t[15] - sum(t[i] for i in TRIPS.values())) / frames
        row["arrivals"] = t[15] / frames
        row["trips"] = t[5] / frames
        out[k] = row
    return out


def test_straight_returns_take_fewer_dispatcher_trips(tmp_path):
    r = dispatch_trips(str(tmp_path))
    s, d = r["straight"], r["dispatcher"]
    assert s["trips"] < 0.6 * d["trips"], r
    assert s["RTS"] < d["RTS"] and s["JMP ind"] <= d["JMP ind"] and s["BRK/RTI"] < d["BRK/RTI"], r
    assert s["WSYNC"] == d["WSYNC"] and s["frame end"] == d["frame end"], r


if __name__ == "__main__":
    import json
    import tempfile
    with tempfile.TemporaryDirectory() as t:
        print(json.dumps(dispatch_trips(t), indent=1))
