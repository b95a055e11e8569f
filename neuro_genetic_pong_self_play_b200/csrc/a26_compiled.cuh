// a26_compiled.cuh -- the 6507 side of the fused rollout as statically translated code.
//
// tools/gen_rom_core.py turns every reachable instruction of the bundled cartridge into specialised
// statements (generated/pong_core.inc).  This header provides the dispatcher around them.  TIA, RIOT,
// paddles, rendering and observation accumulation are the same device functions the interpreter
// (a26_core.cuh::run_frame, the verify-mode core) uses, so only instruction fetch/decode/addressing is
// specialised.  Control transfers that the generator cannot resolve to a known block (and WSYNC, see below) return to
// `switch (blockmap[pc])`, where diverged lanes re-converge;
// the loop is scanline-synchronous like the interpreter's.  A program counter outside the translated set
// raises ERR_UNTRANSLATED (never happens for this cartridge: the traversal covers all of its code).
#pragma once
#include "a26_core.cuh"
#include "pong_superblocks.cuh"

namespace a26 {

enum : int { ERR_UNTRANSLATED = 4 };
// A26_STATS counters (indices into a26_stats) of the arrivals at the dispatcher (a26_next_), by what sent the lane there; TRIP_ALL counts every arrival,
// the ones not named here (super-block exits, backward JMPs, branches too far for a direct jump) are the difference
enum : int { TRIP_WSYNC = 9, TRIP_RTS = 10, TRIP_JMP_IND = 11, TRIP_BRK_RTI = 12, TRIP_FRAME_END = 13, TRIP_CYCLE_CAP = 14, TRIP_ALL = 15 };

// hooks emitted by the generator at the head of dispatch entries $F621, $F58D and $F5CC (pong_superblocks.cuh)
#ifndef A26_NO_SUPERBLOCKS
// the display-loop block's queue placement follows the flavour (superblock_f621); tests/host_sim builds can force either one
#ifndef A26_SB_REPLAY_AT_TOP
#define A26_SB_REPLAY_AT_TOP SYNC
#endif
#define A26_SUPERBLOCK_F621 \
    if (superblock_f621<VERIFY, A26_SB_REPLAY_AT_TOP>(s, T, ram, fb, a, x, y, sp, pc, fc, fv, nv, zv, fid, cyc, cpu_ls, sb_iters)) { A26_STAT(6); goto a26_next_; }
#define A26_SUPERBLOCK_F58D \
    if (superblock_f58d<VERIFY>(s, T, ram, fb, a, x, y, pc, fc, nv, zv, cyc, cpu_ls, sb_iters)) { A26_STAT(7); goto a26_next_; }
#define A26_SUPERBLOCK_F5CC \
    if (superblock_f5cc<VERIFY>(s, T, fb, a, y, pc, nv, zv, cyc, cpu_ls, sb_iters)) { A26_STAT(8); goto a26_next_; }
#else
#define A26_SUPERBLOCK_F621
#define A26_SUPERBLOCK_F58D
#define A26_SUPERBLOCK_F5CC
#endif

// After a WSYNC the translated code returns to the dispatcher, where diverged lanes meet again at the scanline boundary.  A
// warp whose other lanes have all finished their episodes has nobody to meet: it continues at the next instruction (the cycle
// cap of the dispatcher still bounds a frame).  Measured on a single live lane: -5.4 % per frame.  The same shortcut for any warp
// whose live lanes arrive at the WSYNC together gains nothing, and going straight on always costs 7.5 % on evolved generations:
// meeting at the scanline boundary pays (profiles/README.md, r02s/r02w).
#define A26_AFTER_WSYNC(PC_, LABEL_)                                                   \
    do {                                                                               \
        if (solo && (cyc - start_cyc) < FRAME_CYCLE_CAP) goto LABEL_;                  \
        pc = (PC_);                                                                    \
        A26_STAT(solo ? TRIP_CYCLE_CAP : TRIP_WSYNC);                                  \
        goto a26_next_;                                                                \
    } while (0)

#define A26_COMPILED_BLOCKMAP
#include "generated/pong_core.inc"
#undef A26_COMPILED_BLOCKMAP

inline void fill_blockmap(uint16_t *dst) { for (int i = 0; i < 2048; ++i) dst[i] = kCompiledBlockMap[i]; }
// the translated core (and its super-blocks) is only valid for the cartridge it was generated from
inline bool rom_matches_translation(const uint8_t *rom)
{
    uint32_t h = 0x811C9DC5u;
    for (int i = 0; i < 2048; ++i) h = (h ^ rom[i]) * 0x01000193u;
    return h == kCompiledRomFnv1a;
}

#ifdef __CUDACC__

#define A26_ADC(M_)                                              \
    do {                                                         \
        const uint32_t m2_ = (M_);                               \
        if (fid & 8u) { s.error = ERR_DECIMAL; done = 1; }       \
        const uint32_t sum_ = a + m2_ + fc;                      \
        fv = ((~(a ^ m2_) & (a ^ sum_)) >> 7) & 1u;              \
        fc = sum_ >> 8;                                          \
        a = sum_ & 0xFFu; nv = zv = a;                           \
    } while (0)
#define A26_CMP(R_, M_)                                          \
    do {                                                         \
        const uint32_t t_ = (R_) - (M_);                         \
        fc = (R_) >= (M_) ? 1u : 0u;                             \
        nv = zv = t_ & 0xFFu;                                    \
    } while (0)
#define A26_PACK_P() (fc | ((((zv & 0xFFu) == 0u) ? 1u : 0u) << 1) | fid | 0x20u | (fv << 6) | (nv & 0x80u))
#define A26_UNPACK_P(P_)                                         \
    do {                                                         \
        fc = (P_) & 1u; zv = ((P_) & 2u) ? 0u : 1u; fid = (P_) & 0x0Cu; fv = ((P_) >> 6) & 1u; nv = (P_) & 0x80u; \
    } while (0)
#define A26_WRITE_DYN(ADDR_, VAL_, TAFTER_)                                                           \
    do {                                                                                              \
        const uint32_t wa_ = (ADDR_) & 0x1FFFu;                                                       \
        if ((wa_ & 0x1280u) == 0x0080u) ram.wr(wa_, (VAL_));                                          \
        else if (!(wa_ & 0x1000u)) {                                                                  \
            const uint32_t rs_ = io_write_slow<VERIFY>(s, T, wa_, (VAL_), (TAFTER_), cpu_ls, fb);     \
            stall_ += rs_ & 0xFFFFu;                                                                  \
            if (rs_ >> 16) done = 1;                                                                  \
        }                                                                                             \
    } while (0)

// SYNC: every thread of the CTA (active or not) makes one barrier call per dispatcher slot, so that all warps of the CTA walk
// through the frame together.  Warps that drift apart execute different parts of the ~250 KB of translated code and evict each
// other from the 32 KB instruction cache (measured: 21 stall cycles per issued instruction in a saturated launch without this);
// in step, one miss serves all warps.  The barrier is a vote ("is anybody still inside the frame?"), which also ends the loop:
// with the super-blocks a frame takes ~40 slots when the warps take the display loops in one go and ~260 when they do not,
// and a fixed slot count of plain barriers costs more in empty slots than the votes do (measured: +11 % saturated).
template <bool VERIFY, bool SYNC>
__device__ __forceinline__ void run_frame_compiled(Chip &s, CpuRegs &r, const Tables &T, Ram ram, uint8_t *fb, bool active = true)
{
    uint32_t a = 0, x = 0, y = 0, sp = 0, pc = 0, fc = 0, fv = 0, nv = 0, zv = 0, fid = 0, cyc = 0, cpu_ls = 0;
    uint32_t done = 1;
    if (active) {
        a = r.a; x = r.x; y = r.y; sp = r.sp; pc = r.pc;
        fc = r.c; fv = r.v; nv = r.nv; zv = r.zv; fid = r.id;
        cyc = r.cyc; cpu_ls = r.cpu_ls;
        s.frame_done = 0;
        done = s.error ? 1 : 0;
    }
    const uint32_t start_cyc = cyc;
    // a warp with a single environment still playing does not wait for anybody (see A26_AFTER_WSYNC)
    const bool solo = !SYNC && __popc(__ballot_sync(__activemask(), !done)) <= 1;
    for (uint32_t slot = 0;; ++slot) {
        // The display loop's super-block runs all of its iterations in one go only when every lane of the warp that is
        // still inside its frame stands at the loop entry: environments in different game phases reach the loop a few
        // slots apart, and a lane that ran ahead alone would execute the whole loop a second time for the others.
        // (Only a scheduling hint: any iteration count gives the same machine state.)
        const int sb_iters = (solo || __all_sync(__activemask(), done || pc == 0xF621u || pc == 0xF58Du || pc == 0xF5CCu)) ? 128 : 1;
        (void)sb_iters;
        if (!done) {
            if ((cyc - start_cyc) >= FRAME_CYCLE_CAP) done = 1;
            else {
                const uint32_t line_end = cpu_ls + LINE_CYCLES;
                while ((int32_t)(cyc - line_end) < 0 && !done) {
                    A26_STAT(5);
                    uint32_t entry;
                    A26_HOT_DISPATCH
                    entry = (pc & 0x1000u) ? T.blockmap[pc & 0x7FFu] : 0u;
                    A26_STAT_ENTRY(pc);
                    switch (entry) {
#include "generated/pong_core.inc"
                    default:
                        s.error = (uint8_t)((pc & 0x1000u) ? (int)ERR_UNTRANSLATED : (int)ERR_PC_NOT_ROM);
                        done = 1;
                        break;
                    }
                a26_next_:
                    A26_STAT(TRIP_ALL);
                }
                cpu_ls += (cyc - cpu_ls) / LINE_CYCLES * LINE_CYCLES;
            }
        }
        if (SYNC) {
            if (!__syncthreads_or(!done)) break;
        } else if (done) break;
    }
    if (!active) return;
    tia_catchup<VERIFY>(s, T, 3 * (int)(cyc - s.tia_ls), fb);
    r.a = a; r.x = x; r.y = y; r.sp = sp; r.pc = pc; r.c = fc; r.v = fv; r.nv = nv; r.zv = zv; r.id = fid;
    r.cyc = cyc; r.cpu_ls = cpu_ls;
}

#endif  // __CUDACC__
}  // namespace a26
