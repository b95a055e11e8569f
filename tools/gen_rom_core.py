#!/usr/bin/env python3
"""Static translation of the bundled 2 KiB cartridge into straight-line CUDA for the 6507 side of
the fused rollout (csrc/generated/pong_core.inc), used by a26::run_frame_compiled.

Every reachable instruction becomes specialised C statements (addressing mode, operand bytes, cycle
count, page-cross penalties and RAM/TIA/RIOT/ROM address class all resolved here), grouped into basic
blocks; control transfers go back through a central dispatcher `switch (blockmap[pc])`, which is also
where diverged lanes of a warp re-converge.  Semantics follow csrc/a26_core.cuh::run_frame (the table
driven interpreter, which stays as the verify-mode core) statement for statement; both are checked
bit-for-bit against the CPU oracle.

Usage: python tools/gen_rom_core.py [OUT] [--no-straight-returns]
  (rewrites the .inc next to the other CUDA sources; --no-straight-returns sends every RTS, RTI, JMP ind and BRK through the
  dispatcher, the translation before straight returns, which tests/test_host_sim_dispatch_trips.py compares against)
"""
import hashlib
import os
import re
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from dis6507 import LEN, M  # noqa: E402  opcode -> (mnemonic, mode, cycles)

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
ROM_PATH = os.path.join(ROOT, "neuro_genetic_pong_self_play_b200", "data", "video_olympics.a26")
OUT_PATH = os.path.join(ROOT, "neuro_genetic_pong_self_play_b200", "csrc", "generated", "pong_core.inc")

READ_OPS = {"LDA", "LDX", "LDY", "ORA", "AND", "EOR", "ADC", "SBC", "CMP", "CPX", "CPY", "BIT"}
RMW_OPS = {"ASL", "LSR", "ROL", "ROR", "INC", "DEC"}
STORE_OPS = {"STA": "a", "STX": "x", "STY": "y"}
BRANCH = {"BPL": ("((nv >> 7) & 1u)", 0), "BMI": ("((nv >> 7) & 1u)", 1), "BVC": ("fv", 0), "BVS": ("fv", 1),
          "BCC": ("fc", 0), "BCS": ("fc", 1), "BNE": ("(((zv & 0xFFu) == 0u) ? 1u : 0u)", 0),
          "BEQ": ("(((zv & 0xFFu) == 0u) ? 1u : 0u)", 1)}
PAGE_PENALTY = {"abx", "aby", "izy"}          # only for read instructions
MAX_STRUCTURED_SKIP = 24                      # bytes a structured forward branch may skip
# dispatch entries tried first, hottest first (dispatches per frame measured with tests/host_sim + A26_STATS)
HOT_ENTRIES = []      # with super-blocks and closed-form loops no entry is dispatched more than four times a frame (46 in all)
# Hand-fused super-blocks (csrc/pong_superblocks.cuh): dispatch entry -> (first byte, last byte + 1, sha1 of the cartridge
# bytes the fused code was written against).  The hook is only emitted when the ROM still holds exactly those bytes.
SUPERBLOCKS = {0xF621: (0xF5E0, 0xF63E, "9cf83bee22051baf07f26f6b6fd104e7b6f90ebe"),
               0xF58D: (0xF58B, 0xF5B6, "2c60768c1cb396d94451a9af3be5bc39cdc01337"),
               0xF5CC: (0xF5B8, 0xF5CF, "f66582c70f16bda072d1617e078b396fbd1f594b")}
SUPERBLOCK_EXITS = [0xF63E, 0xF5B6, 0xF5CF]          # program counters a super-block can leave with: must be dispatch entries


def load_rom():
    rom = open(ROM_PATH, "rb").read()
    assert len(rom) == 2048
    return rom


def rb(rom, a):
    return rom[a & 0x7FF]


def vector_targets(rom):
    """targets of JMP ($00A1) / JMP ($00A3): high byte forced to $F3 ($F28D-$F291), low bytes from the 9-byte game
    records at $F659 (bytes 6 and 8 of each record); sorted"""
    return sorted({0xF300 | rb(rom, 0xF659 + 9 * rec + k) for rec in range(7) for k in (6, 8)})


def return_sites(instrs):
    """RTS address -> sorted return sites it can go back to: the instruction after every JSR whose target reaches that RTS
    without passing another RTS (a nested JSR is assumed to return to its own return site; RTI, BRK and JMP ind end the
    walk).  Any other address an RTS pops (a manipulated stack) still goes through the dispatcher."""
    sites = {}
    for j in sorted(a for a, ins in instrs.items() if ins[0] == "JSR"):
        site = j + 3
        work, seen = [instrs[j][3] | instrs[j][4] << 8], set()
        while work:
            a = 0xF000 | (work.pop() & 0x7FF)
            if a in seen or a not in instrs:
                continue
            seen.add(a)
            mn, mode, _, b1, b2, n = instrs[a]
            if mn == "RTS":
                sites.setdefault(a, set()).add(site)
            elif mn in ("RTI", "BRK") or (mn == "JMP" and mode == "ind"):
                pass
            elif mn == "JMP":
                work.append(b1 | b2 << 8)
            elif mn == "JSR":
                work.append(a + 3)
            elif mode == "rel":
                work += [a + 2, a + 2 + (b1 - 256 if b1 > 127 else b1)]
            else:
                work.append(a + n)
    return {r: sorted(v) for r, v in sites.items()}


def acyclic_extension(edges, candidates):
    """The direct jumps (`goto L_xxxx` between dispatch entries, and falling through into the next entry) bypass the
    dispatcher and with it its FRAME_CYCLE_CAP check, so they must not form a cycle: a chain of them could then run for
    ever inside one trip.  `edges` (block -> block: fall-through, JSR, forward branches and forward JMPs) must already be
    acyclic; the in-place loops of backward branches are not in it (each is a short loop of the cartridge that ends), nor
    is the single-lane WSYNC shortcut (it checks the cap itself).  A candidate (block, target) is accepted, in the given
    order, only when `target` cannot reach `block` through the edges accepted so far; a refused one keeps its trip through
    the dispatcher.  Returns the accepted candidates."""
    succ = {}
    for a, b in edges:
        succ.setdefault(a, set()).add(b)

    def reaches(a, b):
        work, seen = [a], set()
        while work:
            x = work.pop()
            if x == b:
                return True
            if x not in seen:
                seen.add(x)
                work += succ.get(x, ())
        return False
    for a in list(succ):
        if any(reaches(b, a) for b in succ[a]):
            raise SystemExit(f"the direct jumps form a cycle through entry {a:04X}")
    accepted = []
    for a, b in candidates:
        if not reaches(b, a):
            succ.setdefault(a, set()).add(b)
            accepted.append((a, b))
    return accepted


def traverse(rom):
    """Recursive-descent discovery of instruction starts and block leaders."""
    reset = rb(rom, 0xFFFC) | rb(rom, 0xFFFD) << 8
    irq = rb(rom, 0xFFFE) | rb(rom, 0xFFFF) << 8
    seeds = {reset, irq} | set(vector_targets(rom))
    instrs, leaders = {}, set(seeds)
    fwd_branches = {}          # pc -> target, forward conditional branches (candidates for structured emission)
    work = list(seeds)
    while work:
        pc = work.pop()
        while True:
            pc = 0xF000 | (pc & 0x7FF)
            if pc in instrs:
                break
            opc = rb(rom, pc)
            if opc not in M:
                raise SystemExit("undocumented opcode %02X reached at %04X" % (opc, pc))
            mn, mode, cyc = M[opc]
            n = LEN[mode]
            instrs[pc] = (mn, mode, cyc, rb(rom, pc + 1), rb(rom, pc + 2), n)
            nxt = pc + n
            if mode == "rel":
                off = rb(rom, pc + 1)
                t = (nxt + (off - 256 if off > 127 else off)) & 0xFFFF
                work.append(t)
                if t > nxt and t - nxt <= MAX_STRUCTURED_SKIP:
                    fwd_branches[pc] = t
                else:
                    leaders.add(t)
            elif mn == "JMP" and mode == "abs":
                t = rb(rom, pc + 1) | rb(rom, pc + 2) << 8
                leaders.add(t); work.append(t)
                break
            elif mn == "JSR":
                t = rb(rom, pc + 1) | rb(rom, pc + 2) << 8
                leaders.add(t); work.append(t)
                leaders.add(nxt)               # RTS comes back here
            elif mn in ("RTS", "RTI") or (mn == "JMP" and mode == "ind"):
                break
            elif mn == "BRK":
                leaders.add(pc + 2)            # RTI comes back past the padding byte
                work.append(pc + 2)
                break
            elif mn in ("STA", "STX", "STY", "PHA", "PHP") or (mn in RMW_OPS and mode != "acc"):
                # the block is left after WSYNC, and a frame can end on a VSYNC write (static, or through an
                # indexed / stack address): the next instruction must then be a dispatch entry
                static_ea = rb(rom, pc + 1) if mode == "zp" else (rb(rom, pc + 1) | rb(rom, pc + 2) << 8) if mode == "abs" else None
                if static_ea is None or (addr_class(static_ea) == "tia" and (static_ea & 0x3F) in (0x00, 0x02)):
                    leaders.add(nxt)
            pc = nxt
    leaders.update(a for a in SUPERBLOCK_EXITS if a in instrs)
    # every instruction start inside the jump-table area can be entered through the RAM vectors
    for a in instrs:
        if 0xF337 <= a <= 0xF41F:
            leaders.add(a)
    # Forward branches over a short, leader-free, properly nested run of instructions are emitted as
    # structured if/else (no trip through the dispatcher, natural SIMT re-convergence).  Fixpoint: a branch
    # that cannot be structured makes its target a leader, which may un-structure other branches.
    order = sorted(instrs)
    nxt_of = {a: a + instrs[a][5] for a in order}
    structured = dict(fwd_branches)
    changed = True
    while changed:
        changed = False
        hard = set(leaders) | {t for pc, t in fwd_branches.items() if pc not in structured}
        stack = []
        for a in order:
            while stack and stack[-1] <= a:
                stack.pop()
            if a in structured:
                t = structured[a]
                ok = not (stack and t > stack[-1])                 # proper nesting
                b = nxt_of[a]
                while ok and b < t:                                # contiguous, leader-free region
                    if b not in instrs or b in hard:
                        ok = False
                        break
                    b = nxt_of[b]
                ok = ok and b == t and t in instrs
                if not ok:
                    del structured[a]
                    changed = True
                    break
                stack.append(t)
    leaders |= {t for pc, t in fwd_branches.items() if pc not in structured}
    return instrs, leaders, structured


def addr_class(a):
    a &= 0x1FFF
    if a & 0x1000:
        return "rom"
    if not (a & 0x80):
        return "tia"
    if not (a & 0x200):
        return "ram"
    return "riot"


class Gen:
    def __init__(self, rom, straight_returns=True):
        self.rom = rom
        self.instrs, self.leaders, self.structured = traverse(rom)
        self.out = []
        self.goto_targets = set()
        self.inline_backward = True
        self.return_sites = return_sites(self.instrs)
        self.vector_targets = vector_targets(rom)
        self.brk_returns = sorted(a + 2 for a, ins in self.instrs.items() if ins[0] == "BRK")     # where RTI goes back to
        self.allowed = set()                  # (block, target) of RTS / RTI / JMP ind / BRK that may jump straight there
        self.straight_returns = straight_returns

    def direct(self, t):
        """`goto` the label of dispatch entry t from the current block (an edge of the graph acyclic_extension checks)"""
        self.goto_targets.add(t)
        self.edges.append((self.cur_block, t))
        return f"goto L_{t:04X};"

    def known_targets(self, pc, targets, trip):
        """after a transfer to a computed or constant pc (RTS, RTI, JMP ind, BRK): straight to each of the known targets, any
        other pc through the dispatcher"""
        for t in targets:
            if t in self.leaders and t in self.instrs:
                self.candidates.append((self.cur_block, t))
                if (self.cur_block, t) in self.allowed:
                    self.emit(f"if (pc == 0x{t:04X}u) {self.direct(t)}")
        self.emit(f"A26_STAT({trip}); goto a26_next_;")

    def emit(self, s):
        self.out.append("    " + s)

    def zp_pointer(self, b1):
        """the two pointer bytes of (zp),Y: straight RAM reads when both lie in console RAM"""
        lo, hi = b1, (b1 + 1) & 0xFF
        if lo >= 0x80 and hi >= 0x80:
            return f"const uint32_t lo_ = ram.rd(0x{lo:02X}u), hi_ = ram.rd(0x{hi:02X}u);"
        return (f"const uint32_t lo_ = bus_read<VERIFY>(s, T, ram, 0x{lo:02X}u, cyc, 0x{b1:02X}u, fb), "
                f"hi_ = bus_read<VERIFY>(s, T, ram, 0x{hi:02X}u, cyc, lo_, fb);")

    # -- operand fetch for read instructions: returns expression for the byte, sets cycle expression
    def read_operand(self, pc, mn, mode, cyc, b1, b2):
        """emit code defining `m` (uint32_t) and `n_` (cycles); returns nothing"""
        e = self.emit
        if mode == "imm":
            e(f"const uint32_t m = 0x{b1:02X}u; const uint32_t n_ = {cyc}u;")
            return
        if mode in ("zp", "abs"):
            ea = b1 if mode == "zp" else (b1 | b2 << 8)
            dbus = b1 if mode == "zp" else b2
            cls = addr_class(ea)
            e(f"const uint32_t n_ = {cyc}u;")
            if cls == "ram":
                e(f"const uint32_t m = ram.rd(0x{ea & 0x7F | 0x80:02X}u);")
            elif cls == "rom":
                e(f"const uint32_t m = 0x{rb(self.rom, ea):02X}u;  /* ROM constant */")
            elif cls == "tia":
                e(f"const uint32_t m = tia_peek<VERIFY>(s, T, 0x{ea & 0x0F:X}u, cyc + n_, 0x{dbus:02X}u, fb);")
            else:
                e(f"const uint32_t m = riot_peek(s, 0x{ea & 0x1FFF:04X}u, cyc + n_);")
            return
        if mode in ("zpx", "zpy"):
            r = "x" if mode == "zpx" else "y"
            e(f"const uint32_t n_ = {cyc}u; const uint32_t ea_ = (0x{b1:02X}u + {r}) & 0xFFu;")
            e(f"const uint32_t m = bus_read<VERIFY>(s, T, ram, ea_, cyc + n_, 0x{b1:02X}u, fb);")
            return
        if mode in ("abx", "aby"):
            r = "x" if mode == "abx" else "y"
            base = b1 | b2 << 8
            e(f"const uint32_t ea_ = (0x{base:04X}u + {r}) & 0xFFFFu; const uint32_t n_ = {cyc}u + ((0x{b1:02X}u + {r}) >> 8);")
            if (base & 0x1000) and ((base + 255) & 0x1000) and (base & 0x1FFF) + 255 <= 0x1FFF:
                e("const uint32_t m = rom_byte(T, ea_);")
            else:
                e(f"const uint32_t m = bus_read<VERIFY>(s, T, ram, ea_ & 0x1FFFu, cyc + n_, 0x{b2:02X}u, fb);")
            return
        if mode == "izy":
            e(self.zp_pointer(b1))
            e("const uint32_t base_ = lo_ | (hi_ << 8), ea_ = (base_ + y) & 0xFFFFu;")
            e(f"const uint32_t n_ = {cyc}u + (((base_ & 0xFFu) + y) >> 8);")
            e("const uint32_t m = bus_read<VERIFY>(s, T, ram, ea_ & 0x1FFFu, cyc + n_, hi_, fb);")
            return
        if mode == "izx":
            e(f"const uint32_t z_ = (0x{b1:02X}u + x) & 0xFFu;")
            e(f"const uint32_t lo_ = bus_read<VERIFY>(s, T, ram, z_, cyc, 0x{b1:02X}u, fb), hi_ = bus_read<VERIFY>(s, T, ram, (z_ + 1) & 0xFFu, cyc, lo_, fb);")
            e(f"const uint32_t n_ = {cyc}u;")
            e("const uint32_t m = bus_read<VERIFY>(s, T, ram, (lo_ | (hi_ << 8)) & 0x1FFFu, cyc + n_, hi_, fb);")
            return
        raise SystemExit(f"read mode {mode} at {pc:04X}")

    def effective_address(self, mode, b1, b2):
        """for stores / RMW: returns (static_ea or None, emitted dynamic name)"""
        e = self.emit
        if mode == "zp":
            return b1
        if mode == "abs":
            return b1 | b2 << 8
        if mode in ("zpx", "zpy"):
            r = "x" if mode == "zpx" else "y"
            e(f"const uint32_t ea_ = (0x{b1:02X}u + {r}) & 0xFFu;")
            return None
        if mode in ("abx", "aby"):
            r = "x" if mode == "abx" else "y"
            e(f"const uint32_t ea_ = (0x{b1 | b2 << 8:04X}u + {r}) & 0x1FFFu;")
            return None
        if mode == "izy":
            e(self.zp_pointer(b1))
            e("const uint32_t ea_ = ((lo_ | (hi_ << 8)) + y) & 0x1FFFu;")
            return None
        if mode == "izx":
            e(f"const uint32_t z_ = (0x{b1:02X}u + x) & 0xFFu;")
            e(f"const uint32_t lo_ = bus_read<VERIFY>(s, T, ram, z_, cyc, 0x{b1:02X}u, fb), hi_ = bus_read<VERIFY>(s, T, ram, (z_ + 1) & 0xFFu, cyc, lo_, fb);")
            e("const uint32_t ea_ = (lo_ | (hi_ << 8)) & 0x1FFFu;")
            return None
        raise SystemExit("store mode " + mode)

    def write(self, static_ea, val, cyc, nxt):
        """emit the store of `val` at time cyc+`cyc`; returns True when the block must end here"""
        e = self.emit
        if static_ea is None:
            e(f"A26_WRITE_DYN(ea_, {val}, cyc + {cyc}u);")
            e(f"cyc += {cyc}u + stall_;")
            e(f"if (done) {{ pc = 0x{nxt:04X}u; A26_STAT(TRIP_FRAME_END); goto a26_next_; }}")
            return False
        cls = addr_class(static_ea)
        if cls == "ram":
            e(f"ram.wr(0x{static_ea & 0x7F | 0x80:02X}u, {val}); cyc += {cyc}u;")
        elif cls == "riot":
            e(f"riot_poke(s, 0x{static_ea & 0x1FFF:04X}u, {val}, cyc + {cyc}u); cyc += {cyc}u;")
        elif cls == "rom":
            e(f"cyc += {cyc}u;  /* write to ROM ignored */")
        else:
            reg = static_ea & 0x3F
            if reg == 0x02:                      # WSYNC: park until the end of the scanline, leave the block
                # the dispatcher is where diverged lanes meet again; a warp with a single live lane goes straight on
                if nxt in self.instrs:
                    self.goto_targets.add(nxt)
                    e(f"cyc += {cyc}u; cyc += wsync_stall(cyc, cpu_ls); A26_AFTER_WSYNC(0x{nxt:04X}u, L_{nxt:04X});")
                else:
                    e(f"cyc += {cyc}u; cyc += wsync_stall(cyc, cpu_ls); pc = 0x{nxt:04X}u; A26_STAT(TRIP_WSYNC); goto a26_next_;")
                return True
            e(f"if (!poke_quick(s, 0x{reg:02X}u, {val})) tia_poke_changed<VERIFY>(s, T, 0x{reg:02X}u, {val}, cyc + {cyc}u, cpu_ls, fb);")
            e(f"cyc += {cyc}u + stall_;")
            if reg == 0x00:
                e(f"if (s.frame_done) {{ done = 1; pc = 0x{nxt:04X}u; A26_STAT(TRIP_FRAME_END); goto a26_next_; }}")
        return False

    def is_intim_wait(self, pc, nxt):
        if nxt not in self.instrs:
            return False
        mn, mode, cyc, b1, b2, n = self.instrs[nxt]
        if mn != "BNE":
            return False
        t = (nxt + 2 + (b1 - 256 if b1 > 127 else b1)) & 0xFFFF
        if t != pc:
            return False
        self.intim_taken = 3 + (1 if (t ^ (nxt + 2)) & 0xFF00 else 0)
        return True

    def closed_form_loop(self, pc, mn, mode, nxt):
        """Two-/three-instruction register-only loops of the cartridge's positioning routine, replaced by their closed form
        (exact: registers, flags and cycle count after the loop; nothing inside the loop touches memory or I/O):
          P: DEY ; BPL P                    -- delay loop
          P: INY ; SBC #k ; BCS P           -- divide by k
        The loop's other instructions must not be entered from elsewhere; they are skipped by generate()."""
        e = self.emit
        ins = self.instrs
        def rel_target(a):
            b1 = ins[a][3]
            return (a + 2 + (b1 - 256 if b1 > 127 else b1)) & 0xFFFF
        if mn == "DEY" and nxt in ins and ins[nxt][0] == "BPL" and rel_target(nxt) == pc and nxt not in self.leaders:
            taken = 3 + (1 if (pc ^ (nxt + 2)) & 0xFF00 else 0)
            e(f"/* DEY ; BPL {pc:04X}: n iterations in closed form */")
            e("const uint32_t n_ = (y >= 1u && y <= 0x80u) ? y + 1u : 1u;")
            e("y = (y - n_) & 0xFFu; nv = zv = y;")
            e(f"cyc += n_ * 2u + (n_ - 1u) * {taken}u + 2u;")
            self.skip.add(nxt)
            return True
        if mn == "INY" and nxt in ins and ins[nxt][0] == "SBC" and ins[nxt][1] == "imm":
            br = nxt + 2
            if br in ins and ins[br][0] == "BCS" and rel_target(br) == pc and nxt not in self.leaders and br not in self.leaders:
                k = ins[nxt][3]
                if k > 0:
                    taken = 3 + (1 if (pc ^ (br + 2)) & 0xFF00 else 0)
                    e(f"/* INY ; SBC #${k:02X} ; BCS {pc:04X}: closed form (every SBC but the last finds A >= k with carry set) */")
                    e("y = (y + 1) & 0xFFu;")
                    e(f"A26_ADC(0x{k ^ 0xFF:02X}u);")
                    e("cyc += 4u;")
                    e("if (fc == 1u) {")
                    e(f"    const uint32_t m_ = a / {k}u;            /* further subtractions that do not borrow */")
                    e(f"    a -= m_ * {k}u; y = (y + m_ + 1u) & 0xFFu;")
                    e(f"    A26_ADC(0x{k ^ 0xFF:02X}u);              /* the one that borrows: flags of the loop exit */")
                    e(f"    cyc += {taken}u + m_ * (4u + {taken}u) + 4u + 2u;")
                    e("} else cyc += 2u;")
                    self.skip.add(nxt); self.skip.add(br)
                    return True
        return False

    def gen_instr(self, pc):
        mn, mode, cyc, b1, b2, n = self.instrs[pc]
        nxt = (pc + n) & 0xFFFF
        e = self.emit
        raw = " ".join("%02X" % rb(self.rom, pc + i) for i in range(n))
        self.out.append(f"  {{ /* {pc:04X}: {raw:<9}{mn} {mode} */")
        self.cur_pc = pc
        ends = False
        if self.closed_form_loop(pc, mn, mode, nxt):
            self.out.append("  }")
            return False
        if mn == "LDA" and mode == "abs" and ((b1 | b2 << 8) & 0x1FFF) == 0x0284 and self.is_intim_wait(pc, nxt):
            # `LDA INTIM; BNE *-3`: skip whole iterations that are known to read non-zero (exact: nothing but
            # A, N, Z and the cycle counter changes in the loop, and the last iteration runs normally below)
            period = 4 + self.intim_taken
            e("{ const int32_t t0_ = s.timer_value - (int32_t)(cyc + 4u - s.timer_set); const int32_t unit_ = 1 << s.timer_shift;")
            e(f"  if (s.timer_shift >= 3u && t0_ >= unit_) cyc += {period}u * ((uint32_t)(t0_ - unit_) / {period}u + 1u); }}")
        if mn in READ_OPS:
            self.read_operand(pc, mn, mode, cyc, b1, b2)
            if mn == "LDA": e("a = m; nv = zv = m;")
            elif mn == "LDX": e("x = m; nv = zv = m;")
            elif mn == "LDY": e("y = m; nv = zv = m;")
            elif mn == "ORA": e("a |= m; nv = zv = a;")
            elif mn == "AND": e("a &= m; nv = zv = a;")
            elif mn == "EOR": e("a ^= m; nv = zv = a;")
            elif mn == "ADC": e("A26_ADC(m);")
            elif mn == "SBC": e("A26_ADC(m ^ 0xFFu);")
            elif mn == "CMP": e("A26_CMP(a, m);")
            elif mn == "CPX": e("A26_CMP(x, m);")
            elif mn == "CPY": e("A26_CMP(y, m);")
            elif mn == "BIT": e("nv = m; fv = (m >> 6) & 1u; zv = m & a;")
            e("cyc += n_;")
        elif mn in STORE_OPS:
            e("uint32_t stall_ = 0; (void)stall_;")
            sea = self.effective_address(mode, b1, b2)
            ends = self.write(sea, STORE_OPS[mn], cyc, nxt)
        elif mn in RMW_OPS:
            if mode == "acc":
                e("const uint32_t m = a; uint32_t wv;")
            else:
                e("uint32_t stall_ = 0; (void)stall_; uint32_t wv;")
                sea = self.effective_address(mode, b1, b2)
                if sea is not None and addr_class(sea) == "ram":
                    e(f"const uint32_t m = ram.rd(0x{sea & 0x7F | 0x80:02X}u);")
                else:
                    if sea is not None:
                        e(f"const uint32_t ea_ = 0x{sea & 0x1FFF:04X}u;")
                        sea = None
                    e(f"const uint32_t m = bus_read<VERIFY>(s, T, ram, ea_ & 0x1FFFu, cyc + {cyc - 2}u, 0x{(b2 if mode in ('abs', 'abx') else b1):02X}u, fb);")
            if mn == "ASL": e("fc = m >> 7; wv = (m << 1) & 0xFFu;")
            elif mn == "LSR": e("fc = m & 1u; wv = m >> 1;")
            elif mn == "ROL": e("wv = ((m << 1) | fc) & 0xFFu; fc = m >> 7;")
            elif mn == "ROR": e("wv = (m >> 1) | (fc << 7); fc = m & 1u;")
            elif mn == "INC": e("wv = (m + 1) & 0xFFu;")
            elif mn == "DEC": e("wv = (m - 1) & 0xFFu;")
            e("nv = zv = wv;")
            if mode == "acc":
                e(f"a = wv; cyc += {cyc}u;")
            else:
                ends = self.write(sea, "wv", cyc, nxt)
        elif mn in BRANCH:
            flag, want = BRANCH[mn]
            t = (nxt + (b1 - 256 if b1 > 127 else b1)) & 0xFFFF
            taken = 3 + (1 if (t ^ nxt) & 0xFF00 else 0)
            if pc in self.structured:
                e(f"if ({flag} == {want}u) {{ cyc += {taken}u; }} else {{ cyc += 2u;  /* structured: skips to {t:04X} */")
                self.open_regions.append(t)
                self.out.append("  /* region */")
                return False
            if t <= pc and t in self.leaders and self.inline_backward:
                # backward branch: loop without a trip through the dispatcher
                self.goto_targets.add(t)
                e(f"if ({flag} == {want}u) {{ cyc += {taken}u; goto L_{t:04X}; }}")
            elif t > pc and t in self.leaders and t in self.instrs:
                # forward branch to another block: straight there (an edge of the graph acyclic_extension checks)
                e(f"if ({flag} == {want}u) {{ cyc += {taken}u; {self.direct(t)} }}")
            else:
                e(f"if ({flag} == {want}u) {{ pc = 0x{t:04X}u; cyc += {taken}u; goto a26_next_; }}")
            e("cyc += 2u;")
        elif mn == "JMP" and mode == "abs":
            t = b1 | b2 << 8
            if t > pc and t in self.leaders and t in self.instrs:
                e(f"cyc += 3u; {self.direct(t)}")
            else:
                e(f"pc = 0x{t:04X}u; cyc += 3u; goto a26_next_;")
            ends = True
        elif mn == "JMP" and mode == "ind":
            p = b1 | b2 << 8
            p2 = (p & 0xFF00) | ((p + 1) & 0xFF)
            e(f"const uint32_t lo_ = bus_read<VERIFY>(s, T, ram, 0x{p & 0x1FFF:04X}u, cyc, 0x{b2:02X}u, fb), hi_ = bus_read<VERIFY>(s, T, ram, 0x{p2 & 0x1FFF:04X}u, cyc, lo_, fb);")
            e("pc = lo_ | (hi_ << 8); cyc += 5u;")
            self.known_targets(pc, self.vector_targets, "TRIP_JMP_IND")
            ends = True
        elif mn == "JSR":
            ret = (pc + 2) & 0xFFFF
            e("uint32_t stall_ = 0;")
            e(f"A26_WRITE_DYN(0x100u | sp, 0x{ret >> 8:02X}u, cyc + 4u); sp = (sp - 1) & 0xFFu;")
            e(f"A26_WRITE_DYN(0x100u | sp, 0x{ret & 0xFF:02X}u, cyc + 5u); sp = (sp - 1) & 0xFFu;")
            # straight to the subroutine's block (no trip through the dispatcher; the matching RTS returns straight too)
            t = b1 | b2 << 8
            if t in self.leaders and t in self.instrs:
                e(f"cyc += 6u + stall_; if (done) {{ pc = 0x{t:04X}u; A26_STAT(TRIP_FRAME_END); goto a26_next_; }} {self.direct(t)}")
            else:
                e(f"pc = 0x{t:04X}u; cyc += 6u + stall_; goto a26_next_;")
            ends = True
        elif mn == "RTS":
            e("sp = (sp + 1) & 0xFFu; const uint32_t lo_ = bus_read<VERIFY>(s, T, ram, 0x100u | sp, cyc, 0u, fb);")
            e("sp = (sp + 1) & 0xFFu; const uint32_t hi_ = bus_read<VERIFY>(s, T, ram, 0x100u | sp, cyc, lo_, fb);")
            e("pc = ((lo_ | (hi_ << 8)) + 1) & 0xFFFFu; cyc += 6u;")
            self.known_targets(pc, self.return_sites.get(pc, []), "TRIP_RTS")
            ends = True
        elif mn == "RTI":
            e("sp = (sp + 1) & 0xFFu; const uint32_t p_ = bus_read<VERIFY>(s, T, ram, 0x100u | sp, cyc, 0u, fb);")
            e("A26_UNPACK_P(p_);")
            e("sp = (sp + 1) & 0xFFu; const uint32_t lo_ = bus_read<VERIFY>(s, T, ram, 0x100u | sp, cyc, p_, fb);")
            e("sp = (sp + 1) & 0xFFu; const uint32_t hi_ = bus_read<VERIFY>(s, T, ram, 0x100u | sp, cyc, lo_, fb);")
            e("pc = lo_ | (hi_ << 8); cyc += 6u;")
            self.known_targets(pc, self.brk_returns, "TRIP_BRK_RTI")
            ends = True
        elif mn == "BRK":
            ret = (pc + 2) & 0xFFFF
            vec = rb(self.rom, 0xFFFE) | rb(self.rom, 0xFFFF) << 8
            e("uint32_t stall_ = 0; const uint32_t p_ = A26_PACK_P() | 0x30u;")
            e(f"A26_WRITE_DYN(0x100u | sp, 0x{ret >> 8:02X}u, cyc + 3u); sp = (sp - 1) & 0xFFu;")
            e(f"A26_WRITE_DYN(0x100u | sp, 0x{ret & 0xFF:02X}u, cyc + 4u); sp = (sp - 1) & 0xFFu;")
            e("A26_WRITE_DYN(0x100u | sp, p_, cyc + 5u); sp = (sp - 1) & 0xFFu;")
            e(f"fid |= 4u; pc = 0x{vec:04X}u; cyc += 7u + stall_; if (done) {{ A26_STAT(TRIP_FRAME_END); goto a26_next_; }}")
            self.known_targets(pc, [vec], "TRIP_BRK_RTI")
            ends = True
        elif mn in ("PHA", "PHP"):
            val = "a" if mn == "PHA" else "(A26_PACK_P() | 0x30u)"
            e(f"uint32_t stall_ = 0; const uint32_t v_ = {val};")
            e("A26_WRITE_DYN(0x100u | sp, v_, cyc + 3u); sp = (sp - 1) & 0xFFu;")
            e("cyc += 3u + stall_;")
            e(f"if (done) {{ pc = 0x{nxt:04X}u; A26_STAT(TRIP_FRAME_END); goto a26_next_; }}")
        elif mn == "PLA":
            e("sp = (sp + 1) & 0xFFu; a = bus_read<VERIFY>(s, T, ram, 0x100u | sp, cyc + 4u, 0u, fb); nv = zv = a; cyc += 4u;")
        elif mn == "PLP":
            e("sp = (sp + 1) & 0xFFu; const uint32_t p_ = bus_read<VERIFY>(s, T, ram, 0x100u | sp, cyc + 4u, 0u, fb); A26_UNPACK_P(p_); cyc += 4u;")
        else:
            simple = {
                "INX": "x = (x + 1) & 0xFFu; nv = zv = x;", "INY": "y = (y + 1) & 0xFFu; nv = zv = y;",
                "DEX": "x = (x - 1) & 0xFFu; nv = zv = x;", "DEY": "y = (y - 1) & 0xFFu; nv = zv = y;",
                "TAX": "x = a; nv = zv = a;", "TAY": "y = a; nv = zv = a;", "TXA": "a = x; nv = zv = a;", "TYA": "a = y; nv = zv = a;",
                "TSX": "x = sp; nv = zv = x;", "TXS": "sp = x;", "CLC": "fc = 0;", "SEC": "fc = 1;", "CLI": "fid &= ~4u;",
                "SEI": "fid |= 4u;", "CLV": "fv = 0;", "CLD": "fid &= ~8u;", "SED": "fid |= 8u;", "NOP": "",
            }
            if mn not in simple:
                raise SystemExit(f"unhandled {mn} at {pc:04X}")
            e(simple[mn] + f" cyc += {cyc}u;")
        self.out.append("  }")
        return ends

    def generate(self):
        order = sorted(self.instrs)
        leaders = sorted(a for a in self.leaders if a in self.instrs)
        ids = {a: i + 1 for i, a in enumerate(leaders)}
        blockmap = [0] * 2048
        for a, i in ids.items():
            blockmap[a & 0x7FF] = i
        self.out.append("// GENERATED by tools/gen_rom_core.py from data/video_olympics.a26 -- do not edit")
        self.out.append(f"// {len(order)} instructions, {len(leaders)} dispatch entries")
        self.out.append("#ifdef A26_COMPILED_BLOCKMAP")
        self.out.append("static const uint16_t kCompiledBlockMap[2048] = {")
        for i in range(0, 2048, 16):
            self.out.append("    " + ", ".join(str(v) for v in blockmap[i:i + 16]) + ",")
        self.out.append("};")
        fnv = 0x811C9DC5
        for b in self.rom:
            fnv = ((fnv ^ b) * 0x01000193) & 0xFFFFFFFF
        self.out.append(f"static const uint32_t kCompiledRomFnv1a = 0x{fnv:08X}u;   // FNV-1a of the 2 KiB image this file was generated from")
        self.out.append("#else")
        head = self.out
        # pass 1 without the straight RTS / RTI / JMP ind / BRK jumps finds the other direct jumps and the candidates; pass 2 emits the
        # candidates that leave the direct jumps acyclic
        self.allowed = set()
        self.code(order, ids)
        self.allowed = set(acyclic_extension(self.edges, self.candidates if self.straight_returns else []))
        self.refused = sorted({c for c in self.candidates if c not in self.allowed}) if self.straight_returns else []
        self.out = head + self.code(order, ids)
        self.out.append("#endif")
        os.makedirs(os.path.dirname(OUT_PATH), exist_ok=True)
        hot = [a for a in HOT_ENTRIES if a in ids]
        self.goto_targets.update(hot)
        chain = " ".join(f"if (pc == 0x{a:04X}u) goto L_{a:04X};" for a in hot)
        self.out.insert(2, f"#define A26_HOT_DISPATCH {chain}")
        text = "\n".join(self.out) + "\n"
        text = re.sub(r"@LABEL_([0-9A-F]{4})@", lambda m: f"L_{m.group(1)}:" if int(m.group(1), 16) in self.goto_targets else "", text)
        with open(OUT_PATH, "w") as f:
            f.write(text)
        return len(order), len(leaders)

    def code(self, order, ids):
        """the case entries of the dispatcher switch; records the direct jumps in self.edges"""
        self.out, self.goto_targets, self.edges, self.candidates = [], set(), [], []
        self.cur_block = None
        prev_fell_through = False
        self.open_regions = []
        self.skip = set()
        for idx, pc in enumerate(order):
            if pc in self.skip:                   # folded into a closed-form loop
                prev_fell_through = True
                continue
            while self.open_regions and self.open_regions[-1] == pc:
                self.open_regions.pop()
                self.out.append("  } }  /* end of structured region */")
                prev_fell_through = True          # the branch-taken path arrives here
            if pc in ids:
                if self.open_regions:
                    raise SystemExit(f"leader {pc:04X} inside a structured region")
                if prev_fell_through:
                    self.edges.append((self.cur_block, pc))
                self.cur_block = pc
                self.out.append(f"case {ids[pc]}: @LABEL_{pc:04X}@ /* ---- {pc:04X} ---- */")
                if pc in SUPERBLOCKS:
                    lo, hi, want = SUPERBLOCKS[pc]
                    got = hashlib.sha1(bytes(rb(self.rom, a) for a in range(lo, hi))).hexdigest()
                    if got == want:
                        self.out.append(f"  A26_SUPERBLOCK_{pc:04X}")
                    else:
                        print(f"note: super-block {pc:04X} not emitted (cartridge bytes {lo:04X}-{hi - 1:04X} hash {got})")
            elif not prev_fell_through:
                # unreachable by fall-through and not a leader: cannot happen (every entry is a leader)
                raise SystemExit(f"instruction {pc:04X} is neither a leader nor reached by fall-through")
            ends = self.gen_instr(pc)
            nxt = pc + self.instrs[pc][5]
            if not ends:
                if nxt not in self.instrs or (idx + 1 < len(order) and order[idx + 1] != nxt):
                    raise SystemExit(f"fall-through from {pc:04X} leaves the translated set")
            elif self.open_regions and not (idx + 1 < len(order) and order[idx + 1] == self.open_regions[-1]):
                # an unconditional transfer inside a structured region must be its last instruction
                pass
            prev_fell_through = not ends
        if self.open_regions:
            raise SystemExit("unterminated structured region")
        return self.out


if __name__ == "__main__":
    args = [a for a in sys.argv[1:] if a != "--no-straight-returns"]
    if args:
        OUT_PATH = args[0]
    g = Gen(load_rom(), straight_returns="--no-straight-returns" not in sys.argv)
    n, l = g.generate()
    print(f"wrote {os.path.relpath(OUT_PATH, ROOT)}: {n} instructions, {l} dispatch entries, {len(g.structured)} structured branches, "
          f"{len(g.allowed)} straight RTS / RTI / JMP ind / BRK targets ({len(g.refused)} refused: they would close a cycle)")
