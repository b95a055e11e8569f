// pong_superblocks.cuh -- hand-fused super-blocks of the bundled cartridge's hottest loops.
//
// The statically translated core (generated/pong_core.inc) spends ~65 % of a frame in the main display
// loop $F5E0-$F63C: 91 iterations per frame, 48 instructions and two scanlines each, from one WSYNC to
// the next.  One iteration is a pure function of X, eleven RAM cells and two paddle-capacitor reads; its
// effects are eight TIA latch writes, two conditional RAM stores and the registers it leaves behind.
// `superblock_f621` computes exactly that in one straight-line block: same values, same write order, same
// CPU cycle stamp on every write and read, no flag bookkeeping for results nobody reads.  The TIA sees the
// same (register, value, cycle) sequence as from the instruction-by-instruction translation, through the same
// poke_quick / tia_poke_changed functions.
//
// tools/gen_rom_core.py only emits the hook when the cartridge bytes of the loop are the ones this code
// was written against; the guards at the top fall back to the generic translation for any state the
// fused form does not cover (it never happens in this cartridge's own control flow).
#pragma once
#include "a26_core.cuh"

// capacity of the display-loop block's queue of deferred TIA writes; an iteration can add eight, the queue is replayed early
// when fewer than eight slots are left (tests/test_host_sim.py runs a build with 9 slots, where that happens all the time)
#ifndef A26_SB_MAX_EVENTS
#define A26_SB_MAX_EVENTS 24
#endif

namespace a26 {
#ifdef __CUDACC__

// WSYNC at the end of a loop iteration without a division: `rel` = cycles between the start of a scanline and the iteration's
// first cycle (0 from the second iteration on: the previous WSYNC aligned it), k = length of the iteration, at most three lines.
__device__ __forceinline__ uint32_t sb_wsync(uint32_t &rel, uint32_t k)
{
    const uint32_t c = rel + k;                    // cycles since that line start; the CPU parks until the next multiple of 76
    rel = 0u;
    return c <= LINE_CYCLES ? LINE_CYCLES - c : (c <= 2u * LINE_CYCLES ? 2u * LINE_CYCLES - c : 3u * LINE_CYCLES - c);
}

// SBC with carry set (the loop always executes SEC first), binary mode: result byte, carry, overflow
__device__ __forceinline__ void sb_sbc(uint32_t acc, uint32_t m, uint32_t &r, uint32_t &c, uint32_t &v)
{
    const uint32_t m2 = m ^ 0xFFu;
    const uint32_t sum = acc + m2 + 1u;
    v = ((~(acc ^ m2) & (acc ^ sum)) >> 7) & 1u;
    c = sum >> 8;
    r = sum & 0xFFu;
}
// the byte PHP pushes: N and Z from `r`, C and V as given
__device__ __forceinline__ uint32_t sb_php(uint32_t r, uint32_t c, uint32_t v, uint32_t fid)
{
    return c | ((r == 0u ? 1u : 0u) << 1) | fid | 0x30u | (v << 6) | (r & 0x80u);
}

// The display loop, entered at $F621 (the instruction after `STX WSYNC`); one iteration is
//   $F621-$F63C  second line of the pair: GRP0, ENAM1, both paddle reads (INPTx bit 7 = capacitor charged; the data bus
//                holds the operand high byte 0 before the read, so the low bits read 0), loop test
//   $F5E0-$F61F  first line of the next pair: ENAM0, GRP1, PF0-2, GRP0 value, ENABL, STX WSYNC
// Up to max_iters iterations run back to back, until the loop test ends the loop.
// Returns false (nothing touched) when a guard fails; otherwise pc is $F63E (loop ended) or $F621.
// REPLAY_AT_TOP: where the queue of deferred writes is made room for (see the loop).
template <bool VERIFY, bool REPLAY_AT_TOP>
__device__ __forceinline__ bool superblock_f621(Chip &s, const Tables &T, Ram ram, uint8_t *fb, uint32_t &a, uint32_t &x, uint32_t &y,
                                                uint32_t &sp, uint32_t &pc, uint32_t &fc, uint32_t &fv, uint32_t &nv, uint32_t &zv,
                                                uint32_t fid, uint32_t &cyc, uint32_t cpu_ls, int max_iters)
{
    if (sp != 0x1Eu || (fid & 8u)) return false;
    // RAM cells the loop only reads (it writes $84/$85 and, through the stack pointer, TIA latches): loaded once
    const uint32_t w80 = ram.rd32(0x80), wb0 = ram.rd32(0xB0), wb4 = ram.rd32(0xB4), wa4 = ram.rd32(0xA4), wa8 = ram.rd32(0xA8);
    const uint32_t w98 = ram.rd32(0x98), w9c = ram.rd32(0x9C), wa0 = ram.rd32(0xA0);
    const uint32_t sel = w80 & 0xFFu;                                   // $80: which paddle pair this frame reads
    const uint32_t p0 = (w98 >> 24) | ((w9c & 0xFFu) << 8), p1 = (w9c >> 8) & 0xFFFFu, p2 = (w9c >> 24) | ((wa0 & 0xFFu) << 8);
    // playfield rows are read from ROM for every Y the loop can produce (Y = X >> 3 < 32)
    if (sel >= 2u || !(p0 & p1 & p2 & (p0 + 31u) & (p1 + 31u) & (p2 + 31u) & 0x1000u)) return false;
    const uint32_t b2 = (wb0 >> 16) & 0xFFu, b3 = wb0 >> 24, b4 = wb4 & 0xFFu, b5 = (wb4 >> 8) & 0xFFu, b6 = (wb4 >> 16) & 0xFFu;
    const uint32_t a5 = (wa4 >> 8) & 0xFFu, a6 = (wa4 >> 16) & 0xFFu, a7 = wa4 >> 24, a8 = wa8 & 0xFFu;
    // paddle capacitors: dump state and thresholds only change in VBLANK code
    const bool dumped = s.dump_enabled != 0;
    const uint32_t dump_cyc = s.dump_cyc, need0 = s.needed[sel], need1 = s.needed[2u + sel];
    // Steady state: when an iteration writes the same eight bytes as the two before it (inside this call), the latches
    // -- including the old/new copies that GRP0/GRP1 writes shuffle -- are at the fixed point of that write sequence: every
    // one of the eight writes would find its latch unchanged, so they are skipped without reading the latches.  (Testing the
    // five plain latches byte by byte against the previous iteration instead was measured slower: eight branches per
    // iteration cost more than the latch reads they save.)
    uint32_t prev_a = 0, prev_b = 0;
    int steady = 0;
    // The sixteen hot latches live in registers while the block runs (a26_core.cuh: HotLatches).  A write that changes something
    // displayed does not stop the loop: it is queued -- register, value, cycle stamp and the latch block as it stood before the
    // write -- and the renderer is brought up to all queued writes in one go when the block is left (nothing inside the loop
    // reads renderer state: no collision read, no frame end).  Replaying an event restores the latch block of its moment and
    // calls tia_poke_changed(), i.e. performs exactly the calls the write-by-write order makes, later.  The point is the warp:
    // every lane's paddles and ball sit on other scanlines, so handled on the spot the renderer runs for one lane at a time at
    // up to 32 x 10 different iterations of a frame; replayed, lane k's n-th event is handled together with everybody else's.
    HotLatches hot;
    hot_load(hot, s);
    constexpr int MAX_EVENTS = A26_SB_MAX_EVENTS;
    static_assert(MAX_EVENTS >= 9, "an iteration can queue eight writes");
    static_assert(128 * 2 * LINE_CYCLES + 2 * LINE_CYCLES < (1 << 18), "an event's cycle stamp is stored as an 18-bit offset from the block's entry (the caller runs at most 128 iterations)");
    uint32_t ev[MAX_EVENTS][4];                                         // latch words 0..2 before the write, reg | v << 6 | dt << 14
    int n_ev = 0;
    const uint32_t t_base = cyc;
    auto replay = [&]() {
        for (int k = 0; k < n_ev; ++k) {
            HotLatches pre;
            pre.w[0] = ev[k][0]; pre.w[1] = ev[k][1]; pre.w[2] = ev[k][2]; pre.w[3] = hot.w[3];
            hot_store(pre, s);
            const uint32_t e = ev[k][3];
            tia_poke_changed<VERIFY>(s, T, e & 0x3Fu, (e >> 6) & 0xFFu, t_base + (e >> 14), cpu_ls, fb);
        }
        n_ev = 0;
        hot_store(hot, s);
    };
#define A26_SB_WRITE(REG_, V_, T_)                                                                             \
    do {                                                                                                       \
        const uint32_t pv_ = (V_) & 0xFFu, p0_ = hot.w[0], p1_ = hot.w[1], p2_ = hot.w[2];                     \
        if (!hot_write<REG_>(hot, pv_)) {                                                                      \
            ev[n_ev][0] = p0_; ev[n_ev][1] = p1_; ev[n_ev][2] = p2_;                                           \
            ev[n_ev][3] = (uint32_t)(REG_) | (pv_ << 6) | (((T_) - t_base) << 14);                             \
            ++n_ev;                                                                                            \
        }                                                                                                      \
    } while (0)
    uint32_t rel = (cyc - cpu_ls) % LINE_CYCLES;                        // see sb_wsync
    pc = 0xF621u;
    // bounded by the caller (at most one trip of X through its 8-bit range), then back through the dispatcher.
    // Every copy of replay() is a loop around a call of tia_poke_changed().  REPLAY_AT_TOP makes room at the top of every
    // iteration (an iteration queues at most eight writes) and so needs one copy besides the one after the loop: ~20
    // registers and a sixth of the spills fewer in the CTA-synchronous flavours, whose register budgets are capped (config 3:
    // 4-6 % faster, measured).  The one-warp flavour has registers to spare and keeps the test off the iteration's path: room
    // is made only where writes are queued (config 2: 2 % faster that way; profiles/r03a_rollout_ab.txt).
    // Replaying earlier or later changes nothing: the renderer reads no RAM, and every event carries its latch block.
    for (int iter = 0; iter < max_iters; ++iter) {
        if (REPLAY_AT_TOP && n_ev > MAX_EVENTS - 8) replay();
        const uint32_t x1 = (x + 1u) & 0xFFu, x2 = (x + 2u) & 0xFFu;
        const uint32_t row = x1 >> 3;                                   // TXA, LSR x3, TAY
        const uint32_t t0 = cyc;
        uint32_t r, c, v;

        // ---- $F621 STY GRP0 ; TXA ; SEC ; SBC $B5 ; AND $A8 ; PHP (sp=$1E -> ENAM1) ----
        const uint32_t v_grp0 = y;                                      // written at t0 + 3
        sb_sbc(x, b5, r, c, v);
        r &= a8;
        const uint32_t v_enam1 = sb_php(r, c, v, fid);                  // written at t0 + 16
        // ---- LDY $80 ; LDA $0038,Y ; BMI ; STX $84 ; LDA $003A,Y ; BMI ; STX $85 ----
        uint32_t k = 23u;
        const uint32_t in0 = (!dumped && (t0 + k - dump_cyc) > need0) ? 0x80u : 0u;
        if (in0) k += 3u; else { ram.wr(0x84u, x); k += 5u; }
        k += 4u;
        const uint32_t in1 = (!dumped && (t0 + k - dump_cyc) > need1) ? 0x80u : 0u;
        if (in1) k += 3u; else { ram.wr(0x85u, x); k += 5u; }
        // ---- CPX #$DC ; BNE $F5E0 ----
        if (x == 0xDCu) {
            if (!REPLAY_AT_TOP && n_ev > MAX_EVENTS - 2) replay();
            A26_SB_WRITE(0x1B, v_grp0, t0 + 3u);
            A26_SB_WRITE(0x1E, v_enam1, t0 + 16u);
            a = in1; y = sel; sp = 0x1Du; fc = 1u; fv = v; nv = zv = 0u;
            cyc = t0 + k + 4u; pc = 0xF63Eu;
            break;
        }
        k += 6u;                                                        // CPX 2 + taken branch across a page 4
        // ---- $F5E0 TXA ; LDY #$F0 ; SEC ; SBC $B3 ; AND $A6 ; BEQ ; LDY #$00 ----
        const uint32_t g1 = (((x - b3) & a6) & 0xFFu) == 0u ? 0xF0u : 0x00u;
        k += 12u + (g1 ? 3u : 4u);
        // ---- TXA ; INX ; SEC ; SBC $B4 ; AND $A7 ; PHP (sp=$1D -> ENAM0) ; STY GRP1 ----
        sb_sbc(x, b4, r, c, v);
        r &= a7;
        const uint32_t v_enam0 = sb_php(r, c, v, fid);
        k += 15u;
        const uint32_t t_enam0 = k;
        k += 3u;
        const uint32_t t_grp1 = k;
        // ---- TXA ; LSR ; LSR ; LSR ; TAY ; LDA ($9B),Y ; STA PF0 ; LDA ($9D),Y ; STA PF1 ; LDA ($9F),Y ; STA PF2 ----
        k += 10u;
        k += 8u + (((p0 & 0xFFu) + row) >> 8);
        const uint32_t t_pf0 = k, v_pf0 = rom_byte(T, p0 + row);
        k += 8u + (((p1 & 0xFFu) + row) >> 8);
        const uint32_t t_pf1 = k, v_pf1 = rom_byte(T, p1 + row);
        k += 8u + (((p2 & 0xFFu) + row) >> 8);
        const uint32_t t_pf2 = k, v_pf2 = rom_byte(T, p2 + row);
        // ---- INX ; TXA ; LDX #$1F ; TXS ; TAX ; LDY #$F0 ; SEC ; SBC $B2 ; AND $A5 ; BEQ ; LDY #$00 ----
        const uint32_t g0 = (((x2 - b2) & a5) & 0xFFu) == 0u ? 0xF0u : 0x00u;
        k += 20u + (g0 ? 3u : 4u);
        // ---- TXA ; SEC ; SBC $B6 ; AND #$FC ; PHP (sp=$1F -> ENABL) ; STX WSYNC ----
        sb_sbc(x2, b6, r, c, v);
        r &= 0xFCu;
        const uint32_t v_enabl = sb_php(r, c, v, fid);
        k += 12u;
        const uint32_t t_enabl = k;
        k += 3u;
        // ---- the eight latch writes, in program order with their cycle stamps (nothing in between reads TIA state) ----
        const uint32_t pack_a = v_grp0 | (v_enam1 << 8) | (v_enam0 << 16) | (g1 << 24);
        const uint32_t pack_b = v_pf0 | (v_pf1 << 8) | (v_pf2 << 16) | (v_enabl << 24);
        steady = (iter > 0 && pack_a == prev_a && pack_b == prev_b) ? steady + 1 : 0;
        prev_a = pack_a; prev_b = pack_b;
        if (steady < 2) {
            if (!hot_display_writes(hot, v_grp0, v_enam1, v_enam0, g1, v_pf0, v_pf1, v_pf2, v_enabl)) {
                if (!REPLAY_AT_TOP && n_ev > MAX_EVENTS - 8) replay();
                A26_SB_WRITE(0x1B, v_grp0, t0 + 3u);
                A26_SB_WRITE(0x1E, v_enam1, t0 + 16u);
                A26_SB_WRITE(0x1D, v_enam0, t0 + t_enam0);
                A26_SB_WRITE(0x1C, g1, t0 + t_grp1);
                A26_SB_WRITE(0x0D, v_pf0, t0 + t_pf0);
                A26_SB_WRITE(0x0E, v_pf1, t0 + t_pf1);
                A26_SB_WRITE(0x0F, v_pf2, t0 + t_pf2);
                A26_SB_WRITE(0x1F, v_enabl, t0 + t_enabl);
            }
        }
        a = r; x = x2; y = g0; fc = c; fv = v; nv = zv = r;
        cyc = t0 + k + sb_wsync(rel, k);                                // k <= 153: within three lines of the iteration's line start
    }
    replay();
    return true;
#undef A26_SB_WRITE
}

// The score display loop $F58B-$F5B4, entered at $F58D (the instruction after `STA WSYNC`): one scanline per iteration,
// 20 per frame.  Each line reads four digit-graphics bytes from ROM through the pointers at $C5/$C9 (left score) and
// $C7/$CB (right score), writes PF1 twice at exact cycles (the two halves of the mirrored playfield show different digits),
// keeps the scratch cell $87, counts lines in X (four per digit row) and digit rows in Y (five).
//   $F58D LDA ($C5),Y ; AND #$0F ; STA $87 ; LDA ($C9),Y ; AND #$F0 ; ORA $87 ; STA PF1
//   $F59B LDA ($C7),Y ; AND #$0F ; STA $87 ; LDA ($CB),Y ; AND #$F0 ; ORA $87 ; AND $90 ; STA PF1
//   $F5AB TXA ; INX ; AND #$03 ; BNE $F58B ; INY ; CPY #$05 ; BNE $F58B        $F58B STA WSYNC
// Returns false (nothing touched) when a guard fails; otherwise pc is $F5B6 (loop ended) or $F58D.
template <bool VERIFY>
__device__ __forceinline__ bool superblock_f58d(Chip &s, const Tables &T, Ram ram, uint8_t *fb, uint32_t &a, uint32_t &x, uint32_t &y,
                                                uint32_t &pc, uint32_t &fc, uint32_t &nv, uint32_t &zv, uint32_t &cyc, uint32_t cpu_ls, int max_iters)
{
    const uint32_t wc4 = ram.rd32(0xC4), wc8 = ram.rd32(0xC8), wcc = ram.rd32(0xCC);
    const uint32_t q5 = (wc4 >> 8) & 0xFFFFu, q7 = (wc4 >> 24) | ((wc8 & 0xFFu) << 8), q9 = (wc8 >> 8) & 0xFFFFu, qb = (wc8 >> 24) | ((wcc & 0xFFu) << 8);
    // digit rows are read from ROM for every Y of the loop (Y < 5)
    if (y >= 5u || !(q5 & q7 & q9 & qb & (q5 + 4u) & (q7 + 4u) & (q9 + 4u) & (qb + 4u) & 0x1000u)) return false;
    const uint32_t r90 = ram.rd(0x90u);
    uint32_t scratch = 0;
    // The score lines lie above the crop and no movable object is enabled there: PF1 changes are latch-only (tia_latch_only).
    // The renderer position and the object latches only change when a write does go the long way, so the test is evaluated
    // once and after such a write; per write it is a comparison of its cycle stamp with the crop's first cycle.
    bool quiet_zone = false;
    uint32_t zone_end = 0;
    auto refresh_zone = [&]() {
        quiet_zone = !VERIFY && s.line < YSTART + CROP_TOP && (s.grp0_new | s.grp0_old | s.grp1_new | s.grp1_old) == 0 &&
                     ((s.enam0 | s.enam1 | s.enabl_new | s.enabl_old) & 2) == 0;
        zone_end = s.tia_ls + (uint32_t)(YSTART + CROP_TOP - s.line) * LINE_CYCLES - 4u;
    };
    refresh_zone();
    auto write_pf1 = [&](uint32_t pv, uint32_t t) {
        if (poke_quick(s, 0x0Eu, pv)) return;
        if (quiet_zone && (int32_t)(t - zone_end) < 0) { s.pf1 = (uint8_t)pv; s.pf_dirty = 1; return; }
        tia_poke_changed<VERIFY>(s, T, 0x0Eu, pv, t, cpu_ls, fb);
        refresh_zone();
    };
    uint32_t rel = (cyc - cpu_ls) % LINE_CYCLES;
    for (int iter = 0; iter < max_iters; ++iter) {
        const uint32_t t0 = cyc;
        const uint32_t m1 = rom_byte(T, q5 + y), m2 = rom_byte(T, q9 + y), m3 = rom_byte(T, q7 + y), m4 = rom_byte(T, qb + y);
        uint32_t k = 23u + (((q5 & 0xFFu) + y) >> 8) + (((q9 & 0xFFu) + y) >> 8);
        write_pf1((m2 & 0xF0u) | (m1 & 0x0Fu), t0 + k);
        k += 26u + (((q7 & 0xFFu) + y) >> 8) + (((qb & 0xFFu) + y) >> 8);
        scratch = m3 & 0x0Fu;
        write_pf1(((m4 & 0xF0u) | scratch) & r90, t0 + k);
        // TXA ; INX ; AND #$03 ; BNE
        a = x & 3u; x = (x + 1u) & 0xFFu; nv = zv = a;
        k += 6u;
        if (a == 0u) {
            // INY ; CPY #$05 ; BNE
            y = (y + 1u) & 0xFFu;
            fc = y >= 5u ? 1u : 0u; nv = zv = (y - 5u) & 0xFFu;
            k += 2u + 4u;
            if (y == 5u) {
                ram.wr(0x87u, scratch);
                cyc = t0 + k + 2u; pc = 0xF5B6u;
                return true;
            }
        }
        k += 3u + 3u;                              // taken branch (same page) + STA WSYNC
        cyc = t0 + k + sb_wsync(rel, k);           // k <= 77
    }
    ram.wr(0x87u, scratch);
    pc = 0xF58Du;
    return true;
}

// The blank-line loop $F5B8-$F5CD, entered at $F5CC (the instruction after `STY WSYNC`): 12 scanlines per frame that write
// zero to PF0-2, GRP0/1, ENAM0/1 and ENABL and wait for the next line.
//   $F5CC DEY ; BNE $F5B8      $F5B8 LDA #$00 ; STA PF0 ; STA PF1 ; STA PF2 ; STA GRP0 ; STA GRP1 ; STA ENAM0 ; STA ENAM1 ; STA ENABL ; STY WSYNC
// From the third identical iteration of one call on, the latches are at the fixed point of the write sequence (see
// superblock_f621) and the writes are skipped.  Leaves with pc = $F5CF (Y reached 0) or $F5CC.
template <bool VERIFY>
__device__ __forceinline__ bool superblock_f5cc(Chip &s, const Tables &T, uint8_t *fb, uint32_t &a, uint32_t &y, uint32_t &pc, uint32_t &nv,
                                                uint32_t &zv, uint32_t &cyc, uint32_t cpu_ls, int max_iters)
{
    uint32_t rel = (cyc - cpu_ls) % LINE_CYCLES;
    for (int iter = 0; iter < max_iters; ++iter) {
        const uint32_t t0 = cyc;
        y = (y - 1u) & 0xFFu;                              // DEY
        if (y == 0u) { nv = zv = 0u; cyc = t0 + 4u; pc = 0xF5CFu; return true; }
        a = 0u; nv = zv = 0u;                              // taken branch (3), LDA #$00 (2)
        if (iter < 2) {
            const uint32_t regs[8] = {0x0Du, 0x0Eu, 0x0Fu, 0x1Bu, 0x1Cu, 0x1Du, 0x1Eu, 0x1Fu};
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (!poke_quick(s, regs[i], 0u)) tia_poke_changed<VERIFY>(s, T, regs[i], 0u, t0 + 10u + 3u * (uint32_t)i, cpu_ls, fb);
        }
        cyc = t0 + 34u + sb_wsync(rel, 34u);               // 2 + 3 + 2 + 8 * 3 + 3 (STY WSYNC)
    }
    pc = 0xF5CCu;
    return true;
}

#endif  // __CUDACC__
}  // namespace a26
