// a26_core.cuh -- device-side Atari 2600 core (6507 + TIA + RIOT + paddles), one environment
// per thread.  Replaces gym-retro's Stella env.step (/root/reference/main.py:77).
//
// Layout / execution model (DESIGN.md "K1"):
//   * 6507 registers, flags and cycle counters live in registers of the owning thread.
//   * The 128 bytes of console RAM live in shared memory as 32 words per lane, word-interleaved
//     across the warp (word w of lane l at ram[w*32 + l]) so that every access is bank-conflict
//     free no matter which address each lane touches.
//   * The cartridge image and the 256-entry decode table sit in shared memory (one copy per CTA).
//   * TIA/RIOT/paddle state is a per-thread struct (local memory, L1 resident); it is only touched
//     on register pokes/peeks and when a scanline span is rendered.
//   * The TIA is rendered lazily in spans of constant register state as 160-bit masks (5 words per
//     object); collisions are mask ANDs; the observation (reference find_stuff) is accumulated
//     from the priority-resolved colour classes with popcounts, so no framebuffer exists in the
//     fast path.  VERIFY builds also write every pixel to a palette-index framebuffer in HBM.
//   * The instruction loop is scanline-synchronous: all lanes of a warp re-converge at every
//     scanline boundary, which is where WSYNC parks the 6507 anyway.
#pragma once
#include <stddef.h>
#include <stdint.h>
#include <string.h>

// optional event counters for the CPU-side debugging harness (tests/host_sim): no code unless A26_STATS
#ifdef A26_STATS
extern unsigned long long a26_stats[16];
extern unsigned long long a26_entry_stats[2048];
extern unsigned long long a26_reg_stats[64];
#define A26_STAT_REG(r) (++a26_reg_stats[(r) & 63])
#define A26_STAT_SLOT(sl) (++a26_entry_stats[(sl) & 0x7FF])
#define A26_STAT(i) (++a26_stats[i])
#define A26_STAT_ENTRY(pc) (++a26_entry_stats[(pc) & 0x7FF])
#else
#define A26_STAT(i) ((void)0)
#define A26_STAT_REG(r) ((void)0)
#define A26_STAT_SLOT(sl) ((void)0)
#define A26_STAT_ENTRY(pc) ((void)0)
#endif

namespace a26 {

// ---- Stella-convention constants (named, swappable; DESIGN.md "Emulator spec") -----------------
constexpr int HBLANK_CLOCKS = 68;
constexpr int LINE_CLOCKS = 228;
constexpr int LINE_CYCLES = 76;
constexpr int YSTART = 34;
constexpr int FB_ROWS = 210;
constexpr int FB_COLS = 160;
constexpr int CROP_TOP = 34;     // config.py:9  GAME_TOP
constexpr int CROP_BOTTOM = 194; // config.py:8  GAME_BOTTOM
constexpr int TRIGMAX = 4096;
constexpr int PADDLE_DIGITAL_SENSITIVITY = 5;
constexpr int PADDLE_DIGITAL_DISTANCE = 60;
constexpr uint32_t FRAME_CYCLE_CAP = 4 * 262 * 76;

enum : int { ERR_NONE = 0, ERR_ILLEGAL_OPCODE = 1, ERR_DECIMAL = 2, ERR_PC_NOT_ROM = 3 };

// ---- decode table ---------------------------------------------------------------------------------
enum Mode : uint32_t { M_IMP, M_ACC, M_IMM, M_ZP, M_ZPX, M_ZPY, M_ABS, M_ABX, M_ABY, M_IZX, M_IZY, M_REL, M_IND };
enum Op : uint32_t {
    O_ILL, O_LDA, O_LDX, O_LDY, O_STA, O_STX, O_STY, O_ORA, O_AND, O_EOR, O_ADC, O_SBC, O_CMP, O_CPX, O_CPY, O_BIT,
    O_ASL, O_LSR, O_ROL, O_ROR, O_INC, O_DEC, O_INX, O_INY, O_DEX, O_DEY, O_TAX, O_TAY, O_TXA, O_TYA, O_TSX, O_TXS,
    O_CLC, O_SEC, O_CLI, O_SEI, O_CLV, O_CLD, O_SED, O_NOP, O_BPL, O_BMI, O_BVC, O_BVS, O_BCC, O_BCS, O_BNE, O_BEQ,
    O_JMP, O_JSR, O_RTS, O_RTI, O_BRK, O_PHA, O_PHP, O_PLA, O_PLP
};
// entry: op[0:6] mode[6:10] cycles[10:13] flags[13:16] len[16:18]
constexpr uint32_t DF_READ = 1u << 13, DF_WRITE = 1u << 14, DF_PAGE = 1u << 15;

struct DecodeTable { uint32_t e[256]; };

inline void build_decode_table(DecodeTable &t)
{
    auto set = [&](int code, Op op, Mode m, int cyc, uint32_t flags) {
        static const int len[] = {1, 1, 2, 2, 2, 2, 3, 3, 3, 2, 2, 2, 3};
        t.e[code] = (uint32_t)op | ((uint32_t)m << 6) | ((uint32_t)cyc << 10) | flags | ((uint32_t)len[m] << 16);
    };
    for (int i = 0; i < 256; ++i) t.e[i] = O_ILL | (M_IMP << 6) | (2u << 10) | (1u << 16);
    struct { int base; Op op; } alu[] = {{0x00, O_ORA}, {0x20, O_AND}, {0x40, O_EOR}, {0x60, O_ADC},
                                         {0xA0, O_LDA}, {0xC0, O_CMP}, {0xE0, O_SBC}};
    for (auto &a : alu) {
        set(a.base + 0x01, a.op, M_IZX, 6, DF_READ);
        set(a.base + 0x05, a.op, M_ZP, 3, DF_READ);
        set(a.base + 0x09, a.op, M_IMM, 2, 0);
        set(a.base + 0x0D, a.op, M_ABS, 4, DF_READ);
        set(a.base + 0x11, a.op, M_IZY, 5, DF_READ | DF_PAGE);
        set(a.base + 0x15, a.op, M_ZPX, 4, DF_READ);
        set(a.base + 0x19, a.op, M_ABY, 4, DF_READ | DF_PAGE);
        set(a.base + 0x1D, a.op, M_ABX, 4, DF_READ | DF_PAGE);
    }
    set(0x81, O_STA, M_IZX, 6, DF_WRITE); set(0x85, O_STA, M_ZP, 3, DF_WRITE); set(0x8D, O_STA, M_ABS, 4, DF_WRITE);
    set(0x91, O_STA, M_IZY, 6, DF_WRITE); set(0x95, O_STA, M_ZPX, 4, DF_WRITE); set(0x99, O_STA, M_ABY, 5, DF_WRITE);
    set(0x9D, O_STA, M_ABX, 5, DF_WRITE);
    set(0x86, O_STX, M_ZP, 3, DF_WRITE); set(0x96, O_STX, M_ZPY, 4, DF_WRITE); set(0x8E, O_STX, M_ABS, 4, DF_WRITE);
    set(0x84, O_STY, M_ZP, 3, DF_WRITE); set(0x94, O_STY, M_ZPX, 4, DF_WRITE); set(0x8C, O_STY, M_ABS, 4, DF_WRITE);
    set(0xA2, O_LDX, M_IMM, 2, 0); set(0xA6, O_LDX, M_ZP, 3, DF_READ); set(0xB6, O_LDX, M_ZPY, 4, DF_READ);
    set(0xAE, O_LDX, M_ABS, 4, DF_READ); set(0xBE, O_LDX, M_ABY, 4, DF_READ | DF_PAGE);
    set(0xA0, O_LDY, M_IMM, 2, 0); set(0xA4, O_LDY, M_ZP, 3, DF_READ); set(0xB4, O_LDY, M_ZPX, 4, DF_READ);
    set(0xAC, O_LDY, M_ABS, 4, DF_READ); set(0xBC, O_LDY, M_ABX, 4, DF_READ | DF_PAGE);
    set(0xE0, O_CPX, M_IMM, 2, 0); set(0xE4, O_CPX, M_ZP, 3, DF_READ); set(0xEC, O_CPX, M_ABS, 4, DF_READ);
    set(0xC0, O_CPY, M_IMM, 2, 0); set(0xC4, O_CPY, M_ZP, 3, DF_READ); set(0xCC, O_CPY, M_ABS, 4, DF_READ);
    set(0x24, O_BIT, M_ZP, 3, DF_READ); set(0x2C, O_BIT, M_ABS, 4, DF_READ);
    struct { int base; Op op; } sh[] = {{0x00, O_ASL}, {0x20, O_ROL}, {0x40, O_LSR}, {0x60, O_ROR}};
    for (auto &s : sh) {
        set(s.base + 0x06, s.op, M_ZP, 5, DF_READ | DF_WRITE);
        set(s.base + 0x0A, s.op, M_ACC, 2, 0);
        set(s.base + 0x0E, s.op, M_ABS, 6, DF_READ | DF_WRITE);
        set(s.base + 0x16, s.op, M_ZPX, 6, DF_READ | DF_WRITE);
        set(s.base + 0x1E, s.op, M_ABX, 7, DF_READ | DF_WRITE);
    }
    struct { int base; Op op; } id[] = {{0xC0, O_DEC}, {0xE0, O_INC}};
    for (auto &s : id) {
        set(s.base + 0x06, s.op, M_ZP, 5, DF_READ | DF_WRITE);
        set(s.base + 0x0E, s.op, M_ABS, 6, DF_READ | DF_WRITE);
        set(s.base + 0x16, s.op, M_ZPX, 6, DF_READ | DF_WRITE);
        set(s.base + 0x1E, s.op, M_ABX, 7, DF_READ | DF_WRITE);
    }
    set(0x10, O_BPL, M_REL, 2, 0); set(0x30, O_BMI, M_REL, 2, 0); set(0x50, O_BVC, M_REL, 2, 0); set(0x70, O_BVS, M_REL, 2, 0);
    set(0x90, O_BCC, M_REL, 2, 0); set(0xB0, O_BCS, M_REL, 2, 0); set(0xD0, O_BNE, M_REL, 2, 0); set(0xF0, O_BEQ, M_REL, 2, 0);
    set(0x4C, O_JMP, M_ABS, 3, 0); set(0x6C, O_JMP, M_IND, 5, 0); set(0x20, O_JSR, M_ABS, 6, 0);
    set(0x60, O_RTS, M_IMP, 6, 0); set(0x40, O_RTI, M_IMP, 6, 0); set(0x00, O_BRK, M_IMP, 7, 0);
    set(0x48, O_PHA, M_IMP, 3, 0); set(0x08, O_PHP, M_IMP, 3, 0); set(0x68, O_PLA, M_IMP, 4, 0); set(0x28, O_PLP, M_IMP, 4, 0);
    set(0x18, O_CLC, M_IMP, 2, 0); set(0x38, O_SEC, M_IMP, 2, 0); set(0x58, O_CLI, M_IMP, 2, 0); set(0x78, O_SEI, M_IMP, 2, 0);
    set(0xB8, O_CLV, M_IMP, 2, 0); set(0xD8, O_CLD, M_IMP, 2, 0); set(0xF8, O_SED, M_IMP, 2, 0); set(0xEA, O_NOP, M_IMP, 2, 0);
    set(0xAA, O_TAX, M_IMP, 2, 0); set(0xA8, O_TAY, M_IMP, 2, 0); set(0x8A, O_TXA, M_IMP, 2, 0); set(0x98, O_TYA, M_IMP, 2, 0);
    set(0xBA, O_TSX, M_IMP, 2, 0); set(0x9A, O_TXS, M_IMP, 2, 0);
    set(0xE8, O_INX, M_IMP, 2, 0); set(0xC8, O_INY, M_IMP, 2, 0); set(0xCA, O_DEX, M_IMP, 2, 0); set(0x88, O_DEY, M_IMP, 2, 0);
}

// ---- per-environment chip state (TIA + RIOT + paddles + renderer bookkeeping) -----------------
struct alignas(16) Chip {
    // The sixteen latches the display loops rewrite all the time, as one aligned 16-byte block: the super-blocks keep them in
    // four registers (HotLatches) while they run.  Byte order is what hot_* below assume.
    uint8_t pf0, pf1, pf2, grp0_new;
    uint8_t grp0_old, grp1_new, grp1_old, enam0;
    uint8_t enam1, enabl_new, enabl_old, vdelp0;
    uint8_t vdelp1, vdelbl, resmp0, resmp1;
    // the other TIA level registers
    uint8_t vsync, vblank, nusiz0, nusiz1, colup0, colup1, colupf, colubk;
    uint8_t ctrlpf, refp0, refp1, hmp0, hmp1, hmm0, hmm1, hmbl;
    uint8_t posp0, posp1, posm0, posm1, posbl, suppress, hmove_blank, frame_done;
    uint8_t swcha, swchb, dump_enabled, keyrep, error, pf_dirty, pad1, pad2;   // pf_dirty: pfmask[] is stale (rebuilt on use)
    uint16_t cx, pad3;
    // renderer
    int32_t line;            // TIA scanline relative to the frame start
    uint32_t tia_ls;         // absolute CPU cycle at which the TIA's current scanline started
    int32_t rx;              // pixels [0, rx) of the current scanline are rendered
    uint32_t pfmask[5];      // cached 160-bit playfield mask
    // RIOT timer
    int32_t timer_value;
    uint32_t timer_shift, timer_set;
    // paddles
    uint32_t dump_cyc;
    uint16_t charge[4];
    uint8_t repeat[4];
    uint32_t needed[4];
    // observation accumulators (reference find_stuff, utils.py:14-19,60-68)
    uint32_t cnt[3], sx[3], sy[3];
};

// CPU-visible part of an environment that is not in Chip
struct CpuRegs {
    uint32_t a, x, y, sp, pc;
    uint32_t c, v, nv, zv, id;   // carry, overflow, N source (bit7), Z source (==0), I|D bits
    uint32_t cyc;                // absolute CPU cycles (mod 2^32)
    uint32_t cpu_ls;             // absolute cycle of the scanline the CPU is in
};

// snapshot in HBM (start states; stepwise API state)
struct Snapshot {
    Chip chip;
    CpuRegs cpu;
    uint8_t ram[128];
};

struct Tables {               // per-CTA shared-memory tables
    uint32_t rom[512];        // 2 KiB cartridge as words
    uint32_t decode[256];
    uint8_t weight[128];      // per palette entry: 2 bits per target colour = matching channels
    uint16_t blockmap[2048];  // ROM offset -> dispatch entry of the statically translated core (0 = none)
};

#ifdef __CUDACC__

struct Masks { uint32_t w[5]; };

// Every kernel of this library keeps a thread's Chip in local memory and the Tables in shared memory.  An out-of-line function
// only sees generic references, and every generic access costs an address-space lookup plus two R2UR for its descriptor; the
// round trip through the state space lets the compiler emit LDL/STL and LDS with immediate offsets instead.
#ifdef __CUDA_ARCH__
template <typename X>
__device__ __forceinline__ X &as_local(X &g) { __builtin_assume(__isLocal(&g)); return g; }
__device__ __forceinline__ Chip &chip_local(Chip &g) { return as_local(g); }
__device__ __forceinline__ const Tables &tables_shared(const Tables &g)
{
    __builtin_assume(__isShared(&g));
    return g;
}
#else
template <typename X>
__device__ __forceinline__ X &as_local(X &g) { return g; }
__device__ __forceinline__ Chip &chip_local(Chip &g) { return g; }
__device__ __forceinline__ const Tables &tables_shared(const Tables &g) { return g; }
#endif

__device__ __forceinline__ uint32_t rom_byte(const Tables &T, uint32_t addr)
{
    return reinterpret_cast<const uint8_t *>(T.rom)[addr & 0x7FF];      // little-endian words: one byte load
}

// ---- RAM: word-interleaved shared memory ---------------------------------------------------
struct Ram {
    uint32_t *base;   // &warp_ram[lane]; byte b of word w sits at byte offset (w*32)*4 + b from base
    __device__ __forceinline__ uint32_t rd(uint32_t a) const
    {
        return reinterpret_cast<const uint8_t *>(base)[((a & 0x7C) << 5) | (a & 3)];
    }
    __device__ __forceinline__ void wr(uint32_t a, uint32_t v)
    {
        reinterpret_cast<uint8_t *>(base)[((a & 0x7C) << 5) | (a & 3)] = (uint8_t)v;
    }
    // the aligned word holding byte a (little-endian: byte a&3 of the result)
    __device__ __forceinline__ uint32_t rd32(uint32_t a) const { return base[(a & 0x7C) << 3]; }
};

// ---- 160-bit mask helpers ----------------------------------------------------------------------
__device__ __forceinline__ uint32_t expand4(uint32_t b)     // 8 bits -> 32 bits, each bit x4
{
    uint32_t t = b & 0xFF;
    t = (t | (t << 12)) & 0x000F000F;
    t = (t | (t << 6)) & 0x03030303;
    t = (t | (t << 3)) & 0x11111111;
    return t * 15u;
}
__device__ __forceinline__ uint32_t expand2(uint32_t b)     // 8 bits -> 16 bits, each bit x2
{
    uint32_t t = b & 0xFF;
    t = (t | (t << 4)) & 0x0F0F;
    t = (t | (t << 2)) & 0x3333;
    t = (t | (t << 1)) & 0x5555;
    return t * 3u;
}
__device__ __forceinline__ void place(Masks &m, uint32_t pat, int q)   // OR pat at pixel q (mod 160)
{
    q = q >= 160 ? q - 160 : q;
    int i = q >> 5, sh = q & 31;
    m.w[i] |= pat << sh;
    if (sh) m.w[i == 4 ? 0 : i + 1] |= pat >> (32 - sh);
}
__device__ __forceinline__ uint32_t range_word(int i, int x0, int x1)  // bits of word i inside [x0,x1)
{
    int lo = x0 - 32 * i, hi = x1 - 32 * i;
    lo = lo < 0 ? 0 : lo; hi = hi > 32 ? 32 : hi;
    if (hi <= lo) return 0;
    uint32_t m = hi == 32 ? 0xFFFFFFFFu : ((1u << hi) - 1u);
    return m & ~((1u << lo) - 1u);
}
// sum of the indices of set bits of v (0..31)
__device__ __forceinline__ uint32_t bit_index_sum(uint32_t v)
{
    return __popc(v & 0xAAAAAAAAu) + 2 * __popc(v & 0xCCCCCCCCu) + 4 * __popc(v & 0xF0F0F0F0u) +
           8 * __popc(v & 0xFF00FF00u) + 16 * __popc(v & 0xFFFF0000u);
}

__device__ __forceinline__ void rebuild_pfmask(Chip &s)
{
    uint32_t L = (uint32_t)(s.pf0 >> 4) | ((__brev((uint32_t)s.pf1) >> 24) << 4) | ((uint32_t)s.pf2 << 12);
    uint32_t R = (s.ctrlpf & 1) ? (__brev(L) >> 12) : L;
    uint64_t H = (uint64_t)L | ((uint64_t)R << 20);     // 40 bits, one per 4 pixels
#pragma unroll
    for (int i = 0; i < 5; ++i) s.pfmask[i] = expand4((uint32_t)(H >> (8 * i)));
}

__device__ __forceinline__ int copy_offsets(int mode, int c)
{
    // copy offsets / 16, one nibble per NUSIZ mode (0xF = no such copy):
    // 0:{0} 1:{0,16} 2:{0,32} 3:{0,16,32} 4:{0,64} 5:{0} 6:{0,32,64} 7:{0}
    if (c == 0) return 0;
    uint32_t n = ((c == 1 ? 0xF2F4121Fu : 0xF4FF2FFFu) >> (4 * mode)) & 0xF;
    return n == 0xF ? -1 : (int)n * 16;
}

static __device__ __noinline__ void player_mask(Masks &m_, int pos, uint32_t nusiz, uint32_t grp, bool reflect, bool suppress)
{
    Masks &m = as_local(m_);
    m.w[0] = m.w[1] = m.w[2] = m.w[3] = m.w[4] = 0;
    if (!grp) return;
    int mode = nusiz & 7;
    uint32_t pat = reflect ? grp : (__brev(grp) >> 24);
    int start = pos;
    if (mode == 5) { pat = expand2(pat); start += 1; }
    else if (mode == 7) { pat = expand4(pat); start += 1; }
    for (int c = 0; c < 3; ++c) {
        int off = copy_offsets(mode, c);
        if (off < 0) continue;
        if (c == 0 && suppress) continue;
        place(m, pat, (start + off) % 160);
    }
}
static __device__ __noinline__ void missile_mask(Masks &m_, int pos, uint32_t nusiz)
{
    Masks &m = as_local(m_);
    m.w[0] = m.w[1] = m.w[2] = m.w[3] = m.w[4] = 0;
    int mode = nusiz & 7;
    uint32_t pat = (1u << (1u << ((nusiz >> 4) & 3))) - 1u;
    for (int c = 0; c < 3; ++c) {
        int off = copy_offsets(mode, c);
        if (off < 0) continue;
        place(m, pat, (pos + off) % 160);
    }
}

__device__ __forceinline__ bool any_and(const Masks &a, const Masks &b)
{
    return ((a.w[0] & b.w[0]) | (a.w[1] & b.w[1]) | (a.w[2] & b.w[2]) | (a.w[3] & b.w[3]) | (a.w[4] & b.w[4])) != 0;
}
__device__ __forceinline__ bool any_bits(const Masks &a) { return (a.w[0] | a.w[1] | a.w[2] | a.w[3] | a.w[4]) != 0; }

// collision latch bit indices: 2*reg + (D7 ? 1 : 0), reg = CXM0P..CXPPMM
enum { CX_M0P0 = 0, CX_M0P1 = 1, CX_M1P1 = 2, CX_M1P0 = 3, CX_P0BL = 4, CX_P0PF = 5, CX_P1BL = 6, CX_P1PF = 7,
       CX_M0BL = 8, CX_M0PF = 9, CX_M1BL = 10, CX_M1PF = 11, CX_BLPF = 13, CX_M0M1 = 14, CX_P0P1 = 15 };

// accumulate one colour class into the observation sums
__device__ __forceinline__ void accumulate_class(Chip &s, const Tables &T, uint32_t colour, const Masks &m, int crop_row)
{
    uint32_t wts = T.weight[colour >> 1];
    if (!wts) return;
    uint32_t n = 0, sx = 0;
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        uint32_t v = m.w[i];
        if (v) { uint32_t p = __popc(v); n += p; sx += p * (32 * i) + bit_index_sum(v); }
    }
    if (!n) return;
#pragma unroll
    for (int t = 0; t < 3; ++t) {
        uint32_t w = (wts >> (2 * t)) & 3;
        s.cnt[t] += w * n; s.sx[t] += w * sx; s.sy[t] += w * n * (uint32_t)crop_row;
    }
}

// Fast accounting of a span in the fused (no framebuffer) mode.  Returns true when the span needs no
// mask rendering: (A) no movable object is enabled -- no collision is possible and only playfield /
// background colours could contribute to the observation; (B) the playfield is empty and the enabled
// objects are single copies whose boxes do not overlap -- no collision, every object pixel shows its own
// colour, so its observation sums follow from the object's pattern directly.  Anything else (playfield
// with objects, overlapping boxes, multi-copy NUSIZ modes, wrap-around, a background colour that matches
// a target channel, the HMOVE comb) goes through render_span.
struct QuickObj { int start, width; uint32_t pat, colour; };
__device__ __forceinline__ bool quick_player(QuickObj &o, uint32_t grp, uint32_t nusiz, uint32_t pos, bool reflect, bool suppress, uint32_t colour, bool &fail)
{
    if (!grp || suppress) return false;
    const uint32_t mode = nusiz & 7;
    uint32_t pat = reflect ? grp : (__brev(grp) >> 24);
    int start = (int)pos, width = 8;
    if (mode == 5) { pat = expand2(pat); start += 1; width = 16; }
    else if (mode == 7) { pat = expand4(pat); start += 1; width = 32; }
    else if (mode != 0) { fail = true; return false; }
    if (start + width > 160) { fail = true; return false; }
    o.start = start; o.width = width; o.pat = pat; o.colour = colour;
    return true;
}
__device__ __forceinline__ bool quick_missile(QuickObj &o, uint32_t nusiz, uint32_t pos, uint32_t colour, bool &fail)
{
    const uint32_t mode = nusiz & 7;
    if (mode != 0 && mode != 5 && mode != 7) { fail = true; return false; }
    const int width = 1 << ((nusiz >> 4) & 3);
    if ((int)pos + width > 160) { fail = true; return false; }
    o.start = (int)pos; o.width = width; o.pat = (1u << width) - 1u; o.colour = colour;
    return true;
}
// One to three rectangles [x0,x1) x [row_lo,row_hi) that share the current register state (a catch-up over several
// scanlines is "rest of the current line, whole lines, start of the target line"): the latches are read and the objects
// classified once.
struct QuickPart { int x0, x1, row_lo, row_hi; };
template <int NPARTS>
__device__ __forceinline__ bool render_parts_quick(Chip &s, const Tables &T, const QuickPart (&part)[NPARTS])
{
    const uint32_t grp0 = (s.vdelp0 & 1) ? s.grp0_old : s.grp0_new, grp1 = (s.vdelp1 & 1) ? s.grp1_old : s.grp1_new;
    const bool bl_on = (((s.vdelbl & 1) ? s.enabl_old : s.enabl_new) & 2) != 0;
    const bool m0_on = (s.enam0 & 2) && !(s.resmp0 & 2), m1_on = (s.enam1 & 2) && !(s.resmp1 & 2);
    // only rows inside the crop count; a part with no pixels inside it needs nothing
    uint32_t nrows[NPARTS], rowsum[NPARTS];
    bool in_crop = false, comb = false;
#pragma unroll
    for (int p = 0; p < NPARTS; ++p) {
        const int clo = part[p].row_lo < CROP_TOP ? CROP_TOP : part[p].row_lo, chi = part[p].row_hi > CROP_BOTTOM ? CROP_BOTTOM : part[p].row_hi;
        const bool live = chi > clo && part[p].x1 > part[p].x0;
        nrows[p] = live ? (uint32_t)(chi - clo) : 0u;
        rowsum[p] = nrows[p] * (uint32_t)(clo - CROP_TOP) + nrows[p] * (nrows[p] - 1) / 2;   // sum of cropped row indices
        in_crop = in_crop || live;
        comb = comb || (s.hmove_blank && part[p].x0 < 8 && part[p].x1 > part[p].x0);
    }
    const bool pf_any = ((s.pf0 & 0xF0) | s.pf1 | s.pf2) != 0;
    if (!(grp0 | grp1) && !bl_on && !m0_on && !m1_on) {
        if (!in_crop) return true;
        uint32_t wts = T.weight[s.colubk >> 1];
        if (pf_any) {
            wts |= T.weight[s.colupf >> 1];
            if ((s.ctrlpf & 6) == 2) wts |= T.weight[s.colup0 >> 1] | T.weight[s.colup1 >> 1];
        }
        if (comb) wts |= T.weight[0];
        return wts == 0;
    }
    if (pf_any || comb || T.weight[s.colubk >> 1]) return false;
    QuickObj o[5];
    bool on[5], fail = false;
    on[0] = quick_player(o[0], grp0, s.nusiz0, s.posp0, (s.refp0 & 8) != 0, (s.suppress & 1) != 0, s.colup0, fail);
    on[1] = quick_player(o[1], grp1, s.nusiz1, s.posp1, (s.refp1 & 8) != 0, (s.suppress & 2) != 0, s.colup1, fail);
    on[2] = m0_on && quick_missile(o[2], s.nusiz0, s.posm0, s.colup0, fail);
    on[3] = m1_on && quick_missile(o[3], s.nusiz1, s.posm1, s.colup1, fail);
    on[4] = false;
    if (bl_on) {
        const int width = 1 << ((s.ctrlpf >> 4) & 3);
        if ((int)s.posbl + width > 160) fail = true;
        else { o[4].start = s.posbl; o[4].width = width; o[4].pat = (1u << width) - 1u; o[4].colour = s.colupf; on[4] = true; }
    }
    if (fail) return false;
#pragma unroll
    for (int i = 0; i < 5; ++i)
#pragma unroll
        for (int j = i + 1; j < 5; ++j)
            if (on[i] && on[j] && o[i].start < o[j].start + o[j].width && o[j].start < o[i].start + o[i].width) return false;
    if (!in_crop) return true;
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        if (!on[i]) continue;
        const uint32_t wts = T.weight[o[i].colour >> 1];
        if (!wts) continue;
        uint32_t n_r = 0, sx_r = 0, n_y = 0;             // pixels x rows, column sums x rows, pixels x row-index sums
#pragma unroll
        for (int p = 0; p < NPARTS; ++p) {
            if (!nrows[p]) continue;
            int lo = part[p].x0 - o[i].start, hi = part[p].x1 - o[i].start;
            lo = lo < 0 ? 0 : lo; hi = hi > o[i].width ? o[i].width : hi;
            if (hi <= lo) continue;
            const uint32_t clip = (hi >= 32 ? 0xFFFFFFFFu : ((1u << hi) - 1u)) & ~((1u << lo) - 1u);
            const uint32_t q = o[i].pat & clip;
            if (!q) continue;
            const uint32_t n = __popc(q), sx = n * (uint32_t)o[i].start + bit_index_sum(q);
            n_r += n * nrows[p]; sx_r += sx * nrows[p]; n_y += n * rowsum[p];
        }
        if (!n_r) continue;
#pragma unroll
        for (int t = 0; t < 3; ++t) {
            const uint32_t w = (wts >> (2 * t)) & 3;
            s.cnt[t] += w * n_r; s.sx[t] += w * sx_r; s.sy[t] += w * n_y;
        }
    }
    return true;
}
static __device__ __noinline__ bool render_span_quick(Chip &s_, const Tables &T_, int x0, int x1, int row_lo, int row_hi)
{
    Chip &s = chip_local(s_);
    const Tables &T = tables_shared(T_);
    const QuickPart part[1] = {{x0, x1, row_lo, row_hi}};
    return render_parts_quick<1>(s, T, part);
}
// Catch-up over a line boundary in the fused mode: the rest of the current line [rx,160), `full` whole lines and the first
// xc pixels of the target line, all with the current register state.  Only valid while no per-line state is pending
// (HMOVE blanking, RESPx suppression: both are cleared at the next line start, so the first line would differ).
// Returns false with nothing changed when the quick rules do not apply.
static __device__ __noinline__ bool catchup_quick(Chip &s_, const Tables &T_, int full, int xc)
{
    Chip &s = chip_local(s_);
    const Tables &T = tables_shared(T_);
    const int row0 = s.line - YSTART;
    // rows outside the display window have no pixels: clip the row ranges to it (the crop lies inside the window)
    const QuickPart part[3] = {{s.rx, FB_COLS, row0, row0 + 1}, {0, FB_COLS, row0 + 1, row0 + 1 + full}, {0, xc, row0 + 1 + full, row0 + 2 + full}};
    return render_parts_quick<3>(s, T, part);
}

template <bool VERIFY>
__device__ __noinline__ void render_span(Chip &s_, const Tables &T_, int x0, int x1, int row, uint8_t *fb_row)
{
    Chip &s = chip_local(s_);
    const Tables &T = tables_shared(T_);
    A26_STAT(2);
    const uint32_t grp0 = (s.vdelp0 & 1) ? s.grp0_old : s.grp0_new, grp1 = (s.vdelp1 & 1) ? s.grp1_old : s.grp1_new;
    const bool bl_on = (((s.vdelbl & 1) ? s.enabl_old : s.enabl_new) & 2) != 0;
    const bool m0_on = (s.enam0 & 2) && !(s.resmp0 & 2), m1_on = (s.enam1 & 2) && !(s.resmp1 & 2);
    const bool in_crop_row = row >= CROP_TOP && row < CROP_BOTTOM;
    A26_STAT(3);
    Masks R, PF, BL, P0, P1, M0, M1;
#pragma unroll
    if (s.pf_dirty) { rebuild_pfmask(s); s.pf_dirty = 0; }
#pragma unroll
    for (int i = 0; i < 5; ++i) { R.w[i] = range_word(i, x0, x1); PF.w[i] = s.pfmask[i] & R.w[i]; }
    // ball
    BL.w[0] = BL.w[1] = BL.w[2] = BL.w[3] = BL.w[4] = 0;
    if (bl_on) place(BL, (1u << (1u << ((s.ctrlpf >> 4) & 3))) - 1u, s.posbl);
    player_mask(P0, s.posp0, s.nusiz0, grp0, s.refp0 & 8, s.suppress & 1);
    player_mask(P1, s.posp1, s.nusiz1, grp1, s.refp1 & 8, s.suppress & 2);
    if (m0_on) missile_mask(M0, s.posm0, s.nusiz0); else M0.w[0] = M0.w[1] = M0.w[2] = M0.w[3] = M0.w[4] = 0;
    if (m1_on) missile_mask(M1, s.posm1, s.nusiz1); else M1.w[0] = M1.w[1] = M1.w[2] = M1.w[3] = M1.w[4] = 0;
#pragma unroll
    for (int i = 0; i < 5; ++i) { BL.w[i] &= R.w[i]; P0.w[i] &= R.w[i]; P1.w[i] &= R.w[i]; M0.w[i] &= R.w[i]; M1.w[i] &= R.w[i]; }
    bool pf = any_bits(PF), bl = any_bits(BL), p0 = any_bits(P0), p1 = any_bits(P1), m0 = any_bits(M0), m1 = any_bits(M1);
    uint32_t cx = 0;
    if (m0) {
        if (p0 && any_and(M0, P0)) cx |= 1u << CX_M0P0;
        if (p1 && any_and(M0, P1)) cx |= 1u << CX_M0P1;
        if (bl && any_and(M0, BL)) cx |= 1u << CX_M0BL;
        if (pf && any_and(M0, PF)) cx |= 1u << CX_M0PF;
        if (m1 && any_and(M0, M1)) cx |= 1u << CX_M0M1;
    }
    if (m1) {
        if (p1 && any_and(M1, P1)) cx |= 1u << CX_M1P1;
        if (p0 && any_and(M1, P0)) cx |= 1u << CX_M1P0;
        if (bl && any_and(M1, BL)) cx |= 1u << CX_M1BL;
        if (pf && any_and(M1, PF)) cx |= 1u << CX_M1PF;
    }
    if (p0) {
        if (bl && any_and(P0, BL)) cx |= 1u << CX_P0BL;
        if (pf && any_and(P0, PF)) cx |= 1u << CX_P0PF;
        if (p1 && any_and(P0, P1)) cx |= 1u << CX_P0P1;
    }
    if (p1) {
        if (bl && any_and(P1, BL)) cx |= 1u << CX_P1BL;
        if (pf && any_and(P1, PF)) cx |= 1u << CX_P1PF;
    }
    if (bl && pf && any_and(BL, PF)) cx |= 1u << CX_BLPF;
    s.cx |= (uint16_t)cx;

    const bool in_crop = in_crop_row;
    if (!VERIFY && !in_crop) return;

    // priority-resolved colour classes (Stella 3.x encoder: PF priority disables score colouring)
    Masks C0, C1, CF, CB, CS0, CS1, CK;   // COLUP0, COLUP1, COLUPF, COLUBK, score-left, score-right, black
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        uint32_t a0 = P0.w[i] | M0.w[i], a1 = P1.w[i] | M1.w[i];
        uint32_t c0, c1, cf, cs0 = 0, cs1 = 0;
        if (s.ctrlpf & 4) {
            cf = PF.w[i] | BL.w[i];
            c0 = a0 & ~cf;
            c1 = a1 & ~cf & ~a0;
        } else {
            c0 = a0;
            c1 = a1 & ~a0;
            uint32_t rem = ~(a0 | a1);
            cf = BL.w[i] & rem;
            uint32_t pfo = PF.w[i] & rem & ~BL.w[i];
            if (s.ctrlpf & 2) {
                uint32_t left_half = i < 2 ? 0xFFFFFFFFu : (i == 2 ? 0x0000FFFFu : 0u);
                cs0 = pfo & left_half; cs1 = pfo & ~left_half;
            } else cf |= pfo;
        }
        uint32_t ck = 0;
        if (s.hmove_blank && i == 0) { ck = R.w[0] & 0xFFu; c0 &= ~ck; c1 &= ~ck; cf &= ~ck; cs0 &= ~ck; cs1 &= ~ck; }
        C0.w[i] = c0; C1.w[i] = c1; CF.w[i] = cf; CS0.w[i] = cs0; CS1.w[i] = cs1; CK.w[i] = ck;
        CB.w[i] = R.w[i] & ~(c0 | c1 | cf | cs0 | cs1 | ck);
    }
    if (in_crop) {
        int cr = row - CROP_TOP;
        accumulate_class(s, T, s.colup0, C0, cr);
        accumulate_class(s, T, s.colup1, C1, cr);
        accumulate_class(s, T, s.colupf, CF, cr);
        accumulate_class(s, T, s.colubk, CB, cr);
        if (s.ctrlpf & 2) { accumulate_class(s, T, s.colup0, CS0, cr); accumulate_class(s, T, s.colup1, CS1, cr); }
        if (s.hmove_blank) accumulate_class(s, T, 0, CK, cr);
    }
    if (VERIFY && fb_row) {
        for (int x = x0; x < x1; ++x) {
            int i = x >> 5; uint32_t b = 1u << (x & 31);
            uint8_t col = s.colubk;
            if ((C0.w[i] | CS0.w[i]) & b) col = s.colup0;
            else if ((C1.w[i] | CS1.w[i]) & b) col = s.colup1;
            else if (CF.w[i] & b) col = s.colupf;
            else if (CK.w[i] & b) col = 0;
            fb_row[x] = col & 0xFE;
        }
    }
}

// black VBLANK pixels x0..x1 of a crop row (only reached when a target colour has a 0 channel: out of line, so that the
// copies of render_to() do not carry it)
static __device__ __noinline__ void render_black_span(Chip &s_, const Tables &T_, int x0, int x1, int row)
{
    Chip &s = chip_local(s_);
    const Tables &T = tables_shared(T_);
    Masks R;
#pragma unroll
    for (int i = 0; i < 5; ++i) R.w[i] = range_word(i, x0, x1);
    accumulate_class(s, T, 0, R, row - CROP_TOP);
}

// advance the renderer to pixel x of the current scanline
template <bool VERIFY>
__device__ __forceinline__ void render_to(Chip &s, const Tables &T, int x, uint8_t *fb)
{
    if (x <= s.rx) return;
    int row = s.line - YSTART;
    if (row >= 0 && row < FB_ROWS) {
        uint8_t *fb_row = (VERIFY && fb) ? fb + row * FB_COLS : nullptr;
        if (!(s.vblank & 2)) {
            if (VERIFY || !render_span_quick(s, T, s.rx, x, row, row + 1)) render_span<VERIFY>(s, T, s.rx, x, row, fb_row);
        }
        // VBLANK: black; the framebuffer is pre-cleared to 0 and black matches no target channel
        // unless a target colour has a 0 channel, which accumulate_class would need to see:
        else if (row >= CROP_TOP && row < CROP_BOTTOM && T.weight[0]) render_black_span(s, T, s.rx, x, row);
    }
    s.rx = x;
}

__device__ __forceinline__ void tia_newline(Chip &s, int k)
{
    s.line += k; s.tia_ls += (uint32_t)k * LINE_CYCLES; s.rx = 0; s.hmove_blank = 0; s.suppress = 0;
}

// k complete scanlines with the current register state, starting at the TIA's current (untouched) line.
// In the fused mode they are accounted for in one step when the quick path applies.
template <bool VERIFY>
__device__ __forceinline__ void render_full_lines(Chip &s, const Tables &T, int k, uint8_t *fb)
{
    if (!VERIFY) {
        const int row0 = s.line - YSTART;
        const int lo = row0 < 0 ? 0 : row0, hi = row0 + k > FB_ROWS ? FB_ROWS : row0 + k;
        bool handled;
        if (hi <= lo) handled = true;                                   // outside the display window
        else if (s.vblank & 2) handled = T.weight[0] == 0;              // black rows
        else handled = render_span_quick(s, T, 0, FB_COLS, lo, hi);
        if (handled) { tia_newline(s, k); return; }
    }
    for (int i = 0; i < k; ++i) { render_to<VERIFY>(s, T, FB_COLS, fb); tia_newline(s, 1); }
}

// bring the TIA up to colour clock h, measured from the start of its current scanline.  Out of line: one copy of the renderer's
// catch-up serves register writes, collision reads and the end of a frame (inlined, each of them carried its own ~12 KB of SASS,
// all of it fetched every frame).
template <bool VERIFY>
__device__ __noinline__ void tia_catchup(Chip &s_, const Tables &T_, int h, uint8_t *fb)
{
    Chip &s = chip_local(s_);
    const Tables &T = tables_shared(T_);
    if (!VERIFY && h > LINE_CLOCKS && !(s.hmove_blank | s.suppress) && !(s.vblank & 2)) {
        // several lines with one register state: one classification of the objects for all of them
        const int hh = h - LINE_CLOCKS, full = (hh - 1) / LINE_CLOCKS;
        int xc = hh - full * LINE_CLOCKS - HBLANK_CLOCKS;
        xc = xc < 0 ? 0 : (xc > FB_COLS ? FB_COLS : xc);
        if (catchup_quick(s, T, full, xc)) {
            s.line += 1 + full; s.tia_ls += (uint32_t)(1 + full) * LINE_CYCLES; s.rx = xc;
            return;
        }
    }
    if (h > LINE_CLOCKS) {
        render_to<VERIFY>(s, T, FB_COLS, fb);                           // finish the current line
        tia_newline(s, 1);
        h -= LINE_CLOCKS;
        const int full = (h - 1) / LINE_CLOCKS;                         // whole lines before the target line
        if (full > 0) { render_full_lines<VERIFY>(s, T, full, fb); h -= full * LINE_CLOCKS; }
    }
    int x = h - HBLANK_CLOCKS;
    if (x > s.rx) render_to<VERIFY>(s, T, x > FB_COLS ? FB_COLS : x, fb);
}

__device__ __forceinline__ int hm_signed(uint32_t hm) { int v = (int)(hm >> 4); return v >= 8 ? v - 16 : v; }
__device__ __forceinline__ uint8_t wrap160(int v) { v %= 160; return (uint8_t)(v < 0 ? v + 160 : v); }

// Writes that need no catch-up of the lazy renderer: a write that leaves every visible latch as it was
// cannot change a pixel; HMxx/HMCLR only matter at the next HMOVE; RSYNC/audio are ignored.  Returns
// true when the write has been fully handled here.
__device__ __forceinline__ bool poke_quick(Chip &s, uint32_t reg, uint32_t v)
{
    // `same` = the bits of the register that can influence a pixel, a collision or an input are unchanged;
    // the latch still takes the new byte (it is write-only, but the parity digest reads it back)
#define A26_QUICK(FIELD, MASK) do { const bool same = ((v ^ s.FIELD) & (MASK)) == 0; if (same) s.FIELD = (uint8_t)v; return same; } while (0)
    switch (reg) {
    case 0x00: if (!((s.vsync & 2) && !(v & 2))) { s.vsync = (uint8_t)v; return true; } return false;
    case 0x01: A26_QUICK(vblank, 0x82);          // D1 blanking, D7 paddle dump
    case 0x04: A26_QUICK(nusiz0, 0x37);
    case 0x05: A26_QUICK(nusiz1, 0x37);
    case 0x06: A26_QUICK(colup0, 0xFE);
    case 0x07: A26_QUICK(colup1, 0xFE);
    case 0x08: A26_QUICK(colupf, 0xFE);
    case 0x09: A26_QUICK(colubk, 0xFE);
    case 0x0A: A26_QUICK(ctrlpf, 0x37);
    case 0x0B: A26_QUICK(refp0, 0x08);
    case 0x0C: A26_QUICK(refp1, 0x08);
    case 0x0D: A26_QUICK(pf0, 0xF0);
    case 0x0E: return v == s.pf1;
    case 0x0F: return v == s.pf2;
    // GRP0 shows its new latch unless VDELP0 is set, GRP1 shows its old latch only when VDELP1 is set (and likewise the ball
    // with VDELBL): a write whose direct effect and whose old<-new copies touch nothing that is currently displayed is applied
    // to the latches right here.
    case 0x1B:
        if (((s.vdelp0 & 1) || v == s.grp0_new) && (!(s.vdelp1 & 1) || s.grp1_old == s.grp1_new)) {
            s.grp0_new = (uint8_t)v; s.grp1_old = s.grp1_new;
            return true;
        }
        return false;
    case 0x1C:
        if (((s.vdelp1 & 1) || v == s.grp1_new) && (!(s.vdelp0 & 1) || s.grp0_old == s.grp0_new) &&
            (!(s.vdelbl & 1) || ((s.enabl_old ^ s.enabl_new) & 2) == 0)) {
            s.grp1_new = (uint8_t)v; s.grp0_old = s.grp0_new; s.enabl_old = s.enabl_new;
            return true;
        }
        return false;
    // a missile locked to its player (RESMPx.D1) is hidden whatever its enable bit says: the bit is unobservable until the lock
    // is released (a RESMPx write, which goes the long way)
    case 0x1D: if (s.resmp0 & 2) { s.enam0 = (uint8_t)v; return true; } A26_QUICK(enam0, 0x02);
    case 0x1E: if (s.resmp1 & 2) { s.enam1 = (uint8_t)v; return true; } A26_QUICK(enam1, 0x02);
    case 0x1F: if (s.vdelbl & 1) { s.enabl_new = (uint8_t)v; return true; } A26_QUICK(enabl_new, 0x02);   // delayed ball shows the old latch
    case 0x20: s.hmp0 = (uint8_t)v; return true;
    case 0x21: s.hmp1 = (uint8_t)v; return true;
    case 0x22: s.hmm0 = (uint8_t)v; return true;
    case 0x23: s.hmm1 = (uint8_t)v; return true;
    case 0x24: s.hmbl = (uint8_t)v; return true;
    case 0x25: A26_QUICK(vdelp0, 0x01);
    case 0x26: A26_QUICK(vdelp1, 0x01);
    case 0x27: A26_QUICK(vdelbl, 0x01);
    case 0x2B: s.hmp0 = s.hmp1 = s.hmm0 = s.hmm1 = s.hmbl = 0; return true;
    case 0x03: case 0x15: case 0x16: case 0x17: case 0x18: case 0x19: case 0x1A: return true;
    default: return reg > 0x2C;
    }
#undef A26_QUICK
}

// ---- register mirror of the sixteen hot latches (Chip bytes 0..15) -------------------------------------------------------
// One local-memory access costs a lone warp ~30 cycles and every test of poke_quick() a branch; the display-loop super-blocks
// therefore hold the latch block in four registers, apply a whole iteration's eight writes to a copy with plain ALU
// operations and only fall back to the memory path when one of the writes would not be quick.
struct HotLatches { uint32_t w[4]; };
static_assert(sizeof(Chip) % 16 == 0, "Chip must keep its 16-byte alignment in arrays");
static_assert(offsetof(Chip, pf0) == 0 && offsetof(Chip, pf1) == 1 && offsetof(Chip, pf2) == 2 && offsetof(Chip, grp0_new) == 3 &&
              offsetof(Chip, grp0_old) == 4 && offsetof(Chip, grp1_new) == 5 && offsetof(Chip, grp1_old) == 6 && offsetof(Chip, enam0) == 7 &&
              offsetof(Chip, enam1) == 8 && offsetof(Chip, enabl_new) == 9 && offsetof(Chip, enabl_old) == 10 && offsetof(Chip, vdelp0) == 11 &&
              offsetof(Chip, vdelp1) == 12 && offsetof(Chip, vdelbl) == 13 && offsetof(Chip, resmp0) == 14 && offsetof(Chip, resmp1) == 15,
              "hot_byte()/hot_put() index the latch block by these byte positions");
__device__ __forceinline__ void hot_load(HotLatches &h, const Chip &s)
{
#ifdef __CUDA_ARCH__
    const uint4 v = *reinterpret_cast<const uint4 *>(&s.pf0);
    h.w[0] = v.x; h.w[1] = v.y; h.w[2] = v.z; h.w[3] = v.w;
#else
    memcpy(h.w, &s.pf0, 16);
#endif
}
__device__ __forceinline__ void hot_store(const HotLatches &h, Chip &s)
{
#ifdef __CUDA_ARCH__
    *reinterpret_cast<uint4 *>(&s.pf0) = make_uint4(h.w[0], h.w[1], h.w[2], h.w[3]);
#else
    memcpy(&s.pf0, h.w, 16);
#endif
}
__device__ __forceinline__ uint32_t hot_byte(uint32_t w, int i) { return (w >> (8 * i)) & 0xFFu; }
__device__ __forceinline__ uint32_t hot_put(uint32_t w, int i, uint32_t v) { return (w & ~(0xFFu << (8 * i))) | ((v & 0xFFu) << (8 * i)); }
// The eight latch writes of one iteration of the main display loop, in program order (GRP0, ENAM1, ENAM0, GRP1, PF0, PF1, PF2,
// ENABL), applied to the mirror by exactly poke_quick()'s rules.  Returns false -- mirror untouched -- when any of them would
// have to go through the renderer.
__device__ __forceinline__ bool hot_display_writes(HotLatches &h, uint32_t v_grp0, uint32_t v_enam1, uint32_t v_enam0, uint32_t v_grp1,
                                                   uint32_t v_pf0, uint32_t v_pf1, uint32_t v_pf2, uint32_t v_enabl)
{
    uint32_t n0 = h.w[0], n1 = h.w[1], n2 = h.w[2];
    const uint32_t w3 = h.w[3];
    const bool vd0 = (hot_byte(n2, 3) & 1u) != 0, vd1 = (hot_byte(w3, 0) & 1u) != 0, vdbl = (hot_byte(w3, 1) & 1u) != 0;
    const bool rm0 = (hot_byte(w3, 2) & 2u) != 0, rm1 = (hot_byte(w3, 3) & 2u) != 0;
    bool ok;
    {   // GRP0: new latch of player 0, old latch of player 1 takes its new one
        const uint32_t grp0_new = hot_byte(n0, 3), grp1_new = hot_byte(n1, 1), grp1_old = hot_byte(n1, 2);
        ok = (vd0 | (v_grp0 == grp0_new)) & (!vd1 | (grp1_old == grp1_new));
        n0 = hot_put(n0, 3, v_grp0); n1 = hot_put(n1, 2, grp1_new);
    }
    ok &= rm1 | (((v_enam1 ^ hot_byte(n2, 0)) & 2u) == 0u);
    n2 = hot_put(n2, 0, v_enam1);
    ok &= rm0 | (((v_enam0 ^ hot_byte(n1, 3)) & 2u) == 0u);
    n1 = hot_put(n1, 3, v_enam0);
    {   // GRP1: new latch of player 1, old latches of player 0 and the ball take their new ones
        const uint32_t grp1_new = hot_byte(n1, 1), grp0_old = hot_byte(n1, 0), grp0_new = hot_byte(n0, 3);
        const uint32_t enabl_new = hot_byte(n2, 1), enabl_old = hot_byte(n2, 2);
        ok &= (vd1 | (v_grp1 == grp1_new)) & (!vd0 | (grp0_old == grp0_new)) & (!vdbl | (((enabl_old ^ enabl_new) & 2u) == 0u));
        n1 = hot_put(n1, 1, v_grp1); n1 = hot_put(n1, 0, grp0_new); n2 = hot_put(n2, 2, enabl_new);
    }
    ok &= (((v_pf0 ^ hot_byte(n0, 0)) & 0xF0u) == 0u) & (v_pf1 == hot_byte(n0, 1)) & (v_pf2 == hot_byte(n0, 2));
    n0 = hot_put(n0, 0, v_pf0);
    ok &= vdbl | (((v_enabl ^ hot_byte(n2, 1)) & 2u) == 0u);
    n2 = hot_put(n2, 1, v_enabl);
    if (ok) { h.w[0] = n0; h.w[1] = n1; h.w[2] = n2; }
    return ok;
}

// One write to a hot latch, applied to the mirror (the latch always takes the byte, with the old<-new copies of GRP0/GRP1
// writes).  Returns poke_quick()'s verdict for it: false = something displayed changes, the renderer has to be brought up to
// the write's time with the state BEFORE it (the caller kept a copy) -- see the event queue of the display-loop super-block.
template <int REG>
__device__ __forceinline__ bool hot_write(HotLatches &h, uint32_t v)
{
    uint32_t &w0 = h.w[0], &w1 = h.w[1], &w2 = h.w[2];
    const uint32_t w3 = h.w[3];
    const bool vd0 = (hot_byte(w2, 3) & 1u) != 0, vd1 = (hot_byte(w3, 0) & 1u) != 0, vdbl = (hot_byte(w3, 1) & 1u) != 0;
    bool quick;
    if (REG == 0x0D) { quick = ((v ^ hot_byte(w0, 0)) & 0xF0u) == 0u; w0 = hot_put(w0, 0, v); }
    else if (REG == 0x0E) { quick = v == hot_byte(w0, 1); w0 = hot_put(w0, 1, v); }
    else if (REG == 0x0F) { quick = v == hot_byte(w0, 2); w0 = hot_put(w0, 2, v); }
    else if (REG == 0x1B) {
        const uint32_t grp1_new = hot_byte(w1, 1);
        quick = (vd0 | (v == hot_byte(w0, 3))) & (!vd1 | (hot_byte(w1, 2) == grp1_new));
        w0 = hot_put(w0, 3, v); w1 = hot_put(w1, 2, grp1_new);
    } else if (REG == 0x1C) {
        const uint32_t grp0_new = hot_byte(w0, 3), enabl_new = hot_byte(w2, 1);
        quick = (vd1 | (v == hot_byte(w1, 1))) & (!vd0 | (hot_byte(w1, 0) == grp0_new)) & (!vdbl | (((hot_byte(w2, 2) ^ enabl_new) & 2u) == 0u));
        w1 = hot_put(w1, 1, v); w1 = hot_put(w1, 0, grp0_new); w2 = hot_put(w2, 2, enabl_new);
    } else if (REG == 0x1D) {
        quick = ((hot_byte(w3, 2) & 2u) != 0) | (((v ^ hot_byte(w1, 3)) & 2u) == 0u);
        w1 = hot_put(w1, 3, v);
    } else if (REG == 0x1E) {
        quick = ((hot_byte(w3, 3) & 2u) != 0) | (((v ^ hot_byte(w2, 0)) & 2u) == 0u);
        w2 = hot_put(w2, 0, v);
    } else {
        static_assert(REG == 0x0D || REG == 0x0E || REG == 0x0F || (REG >= 0x1B && REG <= 0x1F), "not a hot latch");
        quick = vdbl | (((v ^ hot_byte(w2, 1)) & 2u) == 0u);
        w2 = hot_put(w2, 1, v);
    }
    return quick;
}

// cycles the CPU parks after a WSYNC write that completed at cyc_after
__device__ __forceinline__ uint32_t wsync_stall(uint32_t cyc_after, uint32_t cpu_ls)
{
    const uint32_t c = (cyc_after - cpu_ls) % LINE_CYCLES;
    return c ? LINE_CYCLES - c : 0u;
}

// Fused mode, playfield / colour registers while no movable object is enabled: nothing can collide, and rows outside the crop
// add nothing to the observation whatever the registers hold.  When everything between the renderer's position and this
// write lies above the crop (score area) or below it, the renderer is left where it is (it will cross those rows later with
// the new values, to the same effect: none) and only the latch changes.  Returns true when the write has been handled.
__device__ __forceinline__ bool tia_latch_only(Chip &s, uint32_t reg, uint32_t v, uint32_t cyc_after)
{
    if (!(reg >= 0x06 && reg <= 0x0F && reg != 0x0B && reg != 0x0C)) return false;
    const int crop_first = YSTART + CROP_TOP, crop_end = YSTART + CROP_BOTTOM;     // TIA lines of the crop
    const bool above = s.line < crop_first &&
                       (int32_t)(cyc_after + 4u - (s.tia_ls + (uint32_t)(crop_first - s.line) * LINE_CYCLES)) < 0;   // +4: write delay
    const bool below = s.line >= crop_end && !s.frame_done;
    if (!(above || below)) return false;
    if ((s.grp0_new | s.grp0_old | s.grp1_new | s.grp1_old) != 0 || ((s.enam0 | s.enam1 | s.enabl_new | s.enabl_old) & 2) != 0) return false;
    switch (reg) {
    case 0x06: s.colup0 = (uint8_t)v; break;
    case 0x07: s.colup1 = (uint8_t)v; break;
    case 0x08: s.colupf = (uint8_t)v; break;
    case 0x09: s.colubk = (uint8_t)v; break;
    case 0x0A: s.ctrlpf = (uint8_t)v; s.pf_dirty = 1; break;
    case 0x0D: s.pf0 = (uint8_t)v; s.pf_dirty = 1; break;
    case 0x0E: s.pf1 = (uint8_t)v; s.pf_dirty = 1; break;
    default: s.pf2 = (uint8_t)v; s.pf_dirty = 1; break;
    }
    return true;
}

// Apply one TIA register write at its exact time: bring the lazy renderer up to the write's colour clock
// (plus the register's delay), then change the latch.  cil = CPU cycle within the scanline after the write.
template <bool VERIFY>
__device__ __forceinline__ void tia_apply(Chip &s, const Tables &T, uint32_t reg, uint32_t v, uint32_t cyc_after, uint32_t cil, uint8_t *fb)
{
    A26_STAT(1);
    A26_STAT_REG(reg);
    if (!VERIFY && tia_latch_only(s, reg, v, cyc_after)) return;
    const int hpos = 3 * (int)cil;
    int delay = 0;
    switch (reg) {
    case 0x01: case 0x0B: case 0x0C: case 0x1B: case 0x1C: case 0x1D: case 0x1E: case 0x1F: delay = 1; break;
    case 0x04: case 0x05: delay = 8; break;
    case 0x0D: case 0x0E: case 0x0F: delay = (int)((0x3254u >> (4 * (cil & 3))) & 0xF); break;   // {4,5,2,3}
    default: break;
    }
    const int h = 3 * (int)(cyc_after - s.tia_ls) + delay;
    tia_catchup<VERIFY>(s, T, h, fb);
    switch (reg) {
    case 0x00:
        if ((s.vsync & 2) && !(v & 2)) {
            s.frame_done = 1;
            // the scanline containing this write becomes frame line 0
            s.line = (3 * (int)(cyc_after - s.tia_ls) >= LINE_CLOCKS) ? -1 : 0;
        }
        s.vsync = (uint8_t)v;
        break;
    case 0x01:
        if (!(s.vblank & 0x80) && (v & 0x80)) s.dump_enabled = 1;
        if ((s.vblank & 0x80) && !(v & 0x80)) { s.dump_enabled = 0; s.dump_cyc = cyc_after; }
        s.vblank = (uint8_t)v;
        break;
    case 0x04: s.nusiz0 = (uint8_t)v; break;
    case 0x05: s.nusiz1 = (uint8_t)v; break;
    case 0x06: s.colup0 = (uint8_t)v; break;
    case 0x07: s.colup1 = (uint8_t)v; break;
    case 0x08: s.colupf = (uint8_t)v; break;
    case 0x09: s.colubk = (uint8_t)v; break;
    case 0x0A: s.ctrlpf = (uint8_t)v; s.pf_dirty = 1; break;
    case 0x0B: s.refp0 = (uint8_t)v; break;
    case 0x0C: s.refp1 = (uint8_t)v; break;
    case 0x0D: s.pf0 = (uint8_t)v; s.pf_dirty = 1; break;
    case 0x0E: s.pf1 = (uint8_t)v; s.pf_dirty = 1; break;
    case 0x0F: s.pf2 = (uint8_t)v; s.pf_dirty = 1; break;
    case 0x10: s.posp0 = (uint8_t)(hpos < HBLANK_CLOCKS ? 3 : (hpos - HBLANK_CLOCKS + 5) % 160); s.suppress |= 1; break;
    case 0x11: s.posp1 = (uint8_t)(hpos < HBLANK_CLOCKS ? 3 : (hpos - HBLANK_CLOCKS + 5) % 160); s.suppress |= 2; break;
    case 0x12: s.posm0 = (uint8_t)(hpos < HBLANK_CLOCKS ? 2 : (hpos - HBLANK_CLOCKS + 4) % 160); break;
    case 0x13: s.posm1 = (uint8_t)(hpos < HBLANK_CLOCKS ? 2 : (hpos - HBLANK_CLOCKS + 4) % 160); break;
    case 0x14: s.posbl = (uint8_t)(hpos < HBLANK_CLOCKS ? 2 : (hpos - HBLANK_CLOCKS + 4) % 160); break;
    case 0x1B: s.grp0_new = (uint8_t)v; s.grp1_old = s.grp1_new; break;
    case 0x1C: s.grp1_new = (uint8_t)v; s.grp0_old = s.grp0_new; s.enabl_old = s.enabl_new; break;
    case 0x1D: s.enam0 = (uint8_t)v; break;
    case 0x1E: s.enam1 = (uint8_t)v; break;
    case 0x1F: s.enabl_new = (uint8_t)v; break;
    case 0x20: s.hmp0 = (uint8_t)v; break;
    case 0x21: s.hmp1 = (uint8_t)v; break;
    case 0x22: s.hmm0 = (uint8_t)v; break;
    case 0x23: s.hmm1 = (uint8_t)v; break;
    case 0x24: s.hmbl = (uint8_t)v; break;
    case 0x25: s.vdelp0 = (uint8_t)v; break;
    case 0x26: s.vdelp1 = (uint8_t)v; break;
    case 0x27: s.vdelbl = (uint8_t)v; break;
    case 0x28:
        if ((s.resmp0 & 2) && !(v & 2)) { int mode = s.nusiz0 & 7; s.posm0 = wrap160(s.posp0 + (mode == 5 ? 8 : mode == 7 ? 16 : 4)); }
        s.resmp0 = (uint8_t)v;
        break;
    case 0x29:
        if ((s.resmp1 & 2) && !(v & 2)) { int mode = s.nusiz1 & 7; s.posm1 = wrap160(s.posp1 + (mode == 5 ? 8 : mode == 7 ? 16 : 4)); }
        s.resmp1 = (uint8_t)v;
        break;
    case 0x2A:
        s.posp0 = wrap160(s.posp0 - hm_signed(s.hmp0));
        s.posp1 = wrap160(s.posp1 - hm_signed(s.hmp1));
        s.posm0 = wrap160(s.posm0 - hm_signed(s.hmm0));
        s.posm1 = wrap160(s.posm1 - hm_signed(s.hmm1));
        s.posbl = wrap160(s.posbl - hm_signed(s.hmbl));
        if (hpos / 3 <= 20) s.hmove_blank = 1;
        break;
    case 0x2B: s.hmp0 = s.hmp1 = s.hmm0 = s.hmm1 = s.hmbl = 0; break;
    case 0x2C: s.cx = 0; break;
    default: break;
    }
}

// TIA register write.  cyc_after = CPU cycle count after the write cycle; cpu_ls = a CPU cycle at
// which some scanline started.  Returns the number of cycles the CPU stalls (WSYNC).
// tia_poke_changed: for callers that have already seen poke_quick() fail for this write (and reg != WSYNC).
template <bool VERIFY>
__device__ __noinline__ void tia_poke_changed(Chip &s_, const Tables &T_, uint32_t reg, uint32_t v, uint32_t cyc_after, uint32_t cpu_ls, uint8_t *fb)
{
    Chip &s = chip_local(s_);
    const Tables &T = tables_shared(T_);
    A26_STAT(0);
    tia_apply<VERIFY>(s, T, reg, v, cyc_after, (cyc_after - cpu_ls) % LINE_CYCLES, fb);
}
template <bool VERIFY>
__device__ __forceinline__ uint32_t tia_poke(Chip &s, const Tables &T, uint32_t reg, uint32_t v, uint32_t cyc_after, uint32_t cpu_ls, uint8_t *fb)
{
    if (reg == 0x02) return wsync_stall(cyc_after, cpu_ls);
    if (poke_quick(s, reg, v)) return 0;
    tia_poke_changed<VERIFY>(s, T, reg, v, cyc_after, cpu_ls, fb);
    return 0;
}

// collision latch read: needs the renderer caught up to the read
template <bool VERIFY>
__device__ __noinline__ uint32_t tia_peek_cx(Chip &s_, const Tables &T_, uint32_t reg, uint32_t cyc_after, uint8_t *fb)
{
    Chip &s = chip_local(s_);
    const Tables &T = tables_shared(T_);
    tia_catchup<VERIFY>(s, T, 3 * (int)(cyc_after - s.tia_ls), fb);
    uint32_t v = (((s.cx >> (2 * reg + 1)) & 1u) << 7) | (((s.cx >> (2 * reg)) & 1u) << 6);
    if (reg == 6) v &= 0x80;
    return v;
}

template <bool VERIFY>
__device__ __forceinline__ uint32_t tia_peek(Chip &s, const Tables &T, uint32_t reg, uint32_t cyc_after, uint32_t dbus, uint8_t *fb)
{
    A26_STAT(4);
    const uint32_t noise = dbus & 0x3F;
    reg &= 0x0F;
    if (reg >= 8 && reg < 12) {                       // INPT0-3: paddle capacitors (the hot case: 182 reads per frame)
        if (s.dump_enabled) return noise;
        return ((cyc_after - s.dump_cyc) > s.needed[reg - 8] ? 0x80u : 0u) | noise;
    }
    if (reg < 8) return tia_peek_cx<VERIFY>(s, T, reg, cyc_after, fb) | noise;
    if (reg < 14) return 0x80u | noise;               // INPT4/5: joystick triggers, never pressed
    return noise;
}

__device__ __forceinline__ uint32_t riot_peek(const Chip &s, uint32_t addr, uint32_t cyc_after)
{
    switch (addr & 7) {
    case 0: return s.swcha;
    case 2: return s.swchb;
    case 4: case 6: {
        int32_t t = s.timer_value - (int32_t)(cyc_after - s.timer_set);
        return (uint32_t)(t >= 0 ? (t >> s.timer_shift) : t) & 0xFF;
    }
    default: return 0;
    }
}
__device__ __forceinline__ void riot_poke(Chip &s, uint32_t addr, uint32_t v, uint32_t cyc_after)
{
    if ((addr & 0x14) == 0x14) {
        s.timer_shift = (0xA630u >> (4 * (addr & 3))) & 0xF;     // {0,3,6,10}
        s.timer_value = (int32_t)(v << s.timer_shift);
        s.timer_set = cyc_after;
    }
}

// paddle / switch update at the start of a frame (Stella Paddles::update digital emulation)
__device__ __forceinline__ void apply_input(Chip &s, const uint32_t *needed_tab, uint32_t swchb, uint32_t fire, uint32_t dec, uint32_t inc)
{
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        uint32_t rep = s.repeat[i];
        if ((s.keyrep >> i) & 1) { rep++; if (rep > PADDLE_DIGITAL_SENSITIVITY) rep = PADDLE_DIGITAL_DISTANCE; }
        uint32_t ch = s.charge[i];
        uint32_t key = 0;
        if ((dec >> i) & 1) { key = 1; if (ch > rep) ch -= rep; }
        if ((inc >> i) & 1) { key = 1; if (ch + rep < TRIGMAX) ch += rep; }
        s.keyrep = (uint8_t)((s.keyrep & ~(1u << i)) | (key << i));
        s.repeat[i] = (uint8_t)rep;
        if (ch != s.charge[i]) { s.charge[i] = (uint16_t)ch; s.needed[i] = needed_tab[ch]; }
    }
    uint32_t a = 0xFF;
    if (fire & 1) a &= ~0x80u;
    if (fire & 2) a &= ~0x40u;
    if (fire & 4) a &= ~0x08u;
    if (fire & 8) a &= ~0x04u;
    s.swcha = (uint8_t)a;
    s.swchb = (uint8_t)swchb;
}

__device__ __forceinline__ void clear_obs(Chip &s)
{
#pragma unroll
    for (int t = 0; t < 3; ++t) s.cnt[t] = s.sx[t] = s.sy[t] = 0;
}

// ---- bus -----------------------------------------------------------------------------------------
// device registers behind a run-time address (kept out of line: the inline expansion of every TIA/RIOT
// path at every indexed access made the translated core several hundred KB of SASS)
template <bool VERIFY>
__device__ __noinline__ uint32_t io_read_slow(Chip &s_, const Tables &T_, uint32_t addr, uint32_t cyc_after, uint32_t dbus, uint8_t *fb)
{
    Chip &s = chip_local(s_);
    const Tables &T = tables_shared(T_);
    if (addr & 0x80) return riot_peek(s, addr, cyc_after);
    return tia_peek<VERIFY>(s, T, addr, cyc_after, dbus, fb);
}
// returns stall cycles | (frame_done << 16)
template <bool VERIFY>
__device__ __noinline__ uint32_t io_write_slow(Chip &s_, const Tables &T_, uint32_t addr, uint32_t v, uint32_t cyc_after, uint32_t cpu_ls, uint8_t *fb)
{
    Chip &s = chip_local(s_);
    const Tables &T = tables_shared(T_);
    if (!(addr & 0x1080)) {
        const uint32_t reg = addr & 0x3F;
        if (reg == 0x02) return wsync_stall(cyc_after, cpu_ls);
        if (poke_quick(s, reg, v)) return 0;
        tia_poke_changed<VERIFY>(s, T, reg, v, cyc_after, cpu_ls, fb);
        return (uint32_t)s.frame_done << 16;
    }
    if ((addr & 0x1280) == 0x0280) riot_poke(s, addr, v, cyc_after);
    return 0;
}

template <bool VERIFY>
__device__ __forceinline__ uint32_t bus_read(Chip &s, const Tables &T, Ram ram, uint32_t addr, uint32_t cyc_after, uint32_t dbus, uint8_t *fb)
{
    if (addr & 0x1000) return rom_byte(T, addr);
    if ((addr & 0x280) == 0x80) return ram.rd(addr);
    return io_read_slow<VERIFY>(s, T, addr, cyc_after, dbus, fb);
}

// Run the 6507 until the frame ends (VSYNC turned off) -- one env.step of the reference.
template <bool VERIFY>
__device__ __forceinline__ void run_frame(Chip &s, CpuRegs &r, const Tables &T, Ram ram, uint8_t *fb)
{
    uint32_t a = r.a, x = r.x, y = r.y, sp = r.sp, pc = r.pc;
    uint32_t fc = r.c, fv = r.v, nv = r.nv, zv = r.zv, fid = r.id;
    uint32_t cyc = r.cyc, cpu_ls = r.cpu_ls;
    const uint32_t start_cyc = cyc;
    s.frame_done = 0;

    while (!s.frame_done && !s.error && (cyc - start_cyc) < FRAME_CYCLE_CAP) {
        // ---- one scanline worth of instructions; lanes re-converge at the bottom ----
        const uint32_t line_end = cpu_ls + LINE_CYCLES;
        while ((int32_t)(cyc - line_end) < 0 && !s.frame_done && !s.error) {
            if (!(pc & 0x1000)) { s.error = ERR_PC_NOT_ROM; break; }
            A26_STAT_ENTRY(pc);
            // fetch 4 bytes at pc (wraps inside the 2 KiB image)
            const uint32_t pa = pc & 0x7FF;
            const uint32_t w0 = T.rom[pa >> 2], w1 = T.rom[((pa >> 2) + 1) & 511];
            const uint32_t ins = __funnelshift_r(w0, w1, (pa & 3) * 8);
            const uint32_t opc = ins & 0xFF, b1 = (ins >> 8) & 0xFF, b2 = (ins >> 16) & 0xFF;
            const uint32_t d = T.decode[opc];
            const uint32_t op = d & 63, mode = (d >> 6) & 15;
            uint32_t ncyc = (d >> 10) & 7;
            pc = (pc + ((d >> 16) & 3)) & 0xFFFF;
            uint32_t ea = 0, m = b1, dbus = b1;
            switch (mode) {
            case M_ZP: ea = b1; break;
            case M_ZPX: ea = (b1 + x) & 0xFF; break;
            case M_ZPY: ea = (b1 + y) & 0xFF; break;
            case M_ABS: ea = b1 | (b2 << 8); dbus = b2; break;
            case M_ABX: { uint32_t base = b1 | (b2 << 8); ea = (base + x) & 0xFFFF; dbus = b2;
                          if ((d & DF_PAGE) && ((base ^ ea) & 0xFF00)) ncyc++; break; }
            case M_ABY: { uint32_t base = b1 | (b2 << 8); ea = (base + y) & 0xFFFF; dbus = b2;
                          if ((d & DF_PAGE) && ((base ^ ea) & 0xFF00)) ncyc++; break; }
            case M_IZX: { uint32_t z = (b1 + x) & 0xFF;
                          uint32_t lo = bus_read<VERIFY>(s, T, ram, z, cyc, b1, fb), hi = bus_read<VERIFY>(s, T, ram, (z + 1) & 0xFF, cyc, lo, fb);
                          ea = lo | (hi << 8); dbus = hi; break; }
            case M_IZY: { uint32_t lo = bus_read<VERIFY>(s, T, ram, b1, cyc, b1, fb), hi = bus_read<VERIFY>(s, T, ram, (b1 + 1) & 0xFF, cyc, lo, fb);
                          uint32_t base = lo | (hi << 8); ea = (base + y) & 0xFFFF; dbus = hi;
                          if ((d & DF_PAGE) && ((base ^ ea) & 0xFF00)) ncyc++; break; }
            case M_IND: { uint32_t p = b1 | (b2 << 8);
                          uint32_t lo = bus_read<VERIFY>(s, T, ram, p, cyc, b2, fb);
                          uint32_t hi = bus_read<VERIFY>(s, T, ram, (p & 0xFF00) | ((p + 1) & 0xFF), cyc, lo, fb);
                          ea = lo | (hi << 8); break; }
            default: break;   // IMP ACC IMM REL
            }
            const uint32_t cyc_after = cyc + ncyc;
            if (d & DF_READ) {
                // read-modify-write instructions read two cycles before the write
                m = bus_read<VERIFY>(s, T, ram, ea & 0x1FFF, (d & DF_WRITE) ? cyc_after - 2 : cyc_after, dbus, fb);
            } else if (mode == M_ACC) m = a;
            uint32_t wv = 0;        // value to write when DF_WRITE
            uint32_t stall = 0;
            switch (op) {
            case O_LDA: a = m; nv = zv = m; break;
            case O_LDX: x = m; nv = zv = m; break;
            case O_LDY: y = m; nv = zv = m; break;
            case O_STA: wv = a; break;
            case O_STX: wv = x; break;
            case O_STY: wv = y; break;
            case O_ORA: a |= m; nv = zv = a; break;
            case O_AND: a &= m; nv = zv = a; break;
            case O_EOR: a ^= m; nv = zv = a; break;
            case O_SBC: m ^= 0xFF;  /* fallthrough */
            case O_ADC: {
                if (fid & 8) s.error = ERR_DECIMAL;
                uint32_t sum = a + m + fc;
                fv = ((~(a ^ m) & (a ^ sum)) >> 7) & 1;
                fc = sum >> 8;
                a = sum & 0xFF; nv = zv = a; break;
            }
            case O_CMP: { uint32_t t = a - m; fc = a >= m; nv = zv = t & 0xFF; break; }
            case O_CPX: { uint32_t t = x - m; fc = x >= m; nv = zv = t & 0xFF; break; }
            case O_CPY: { uint32_t t = y - m; fc = y >= m; nv = zv = t & 0xFF; break; }
            case O_BIT: nv = m; fv = (m >> 6) & 1; zv = m & a; break;
            case O_ASL: fc = m >> 7; wv = (m << 1) & 0xFF; nv = zv = wv; if (mode == M_ACC) a = wv; break;
            case O_LSR: fc = m & 1; wv = m >> 1; nv = zv = wv; if (mode == M_ACC) a = wv; break;
            case O_ROL: wv = ((m << 1) | fc) & 0xFF; fc = m >> 7; nv = zv = wv; if (mode == M_ACC) a = wv; break;
            case O_ROR: wv = (m >> 1) | (fc << 7); fc = m & 1; nv = zv = wv; if (mode == M_ACC) a = wv; break;
            case O_INC: wv = (m + 1) & 0xFF; nv = zv = wv; break;
            case O_DEC: wv = (m - 1) & 0xFF; nv = zv = wv; break;
            case O_INX: x = (x + 1) & 0xFF; nv = zv = x; break;
            case O_INY: y = (y + 1) & 0xFF; nv = zv = y; break;
            case O_DEX: x = (x - 1) & 0xFF; nv = zv = x; break;
            case O_DEY: y = (y - 1) & 0xFF; nv = zv = y; break;
            case O_TAX: x = a; nv = zv = a; break;
            case O_TAY: y = a; nv = zv = a; break;
            case O_TXA: a = x; nv = zv = a; break;
            case O_TYA: a = y; nv = zv = a; break;
            case O_TSX: x = sp; nv = zv = x; break;
            case O_TXS: sp = x; break;
            case O_CLC: fc = 0; break;
            case O_SEC: fc = 1; break;
            case O_CLI: fid &= ~4u; break;
            case O_SEI: fid |= 4u; break;
            case O_CLV: fv = 0; break;
            case O_CLD: fid &= ~8u; break;
            case O_SED: fid |= 8u; break;
            case O_NOP: break;
            case O_BPL: case O_BMI: case O_BVC: case O_BVS: case O_BCC: case O_BCS: case O_BNE: case O_BEQ: {
                uint32_t flag;
                switch ((op - O_BPL) >> 1) {
                case 0: flag = (nv >> 7) & 1; break;
                case 1: flag = fv; break;
                case 2: flag = fc; break;
                default: flag = (zv & 0xFF) == 0; break;
                }
                if (flag == ((op - O_BPL) & 1)) {
                    uint32_t t = (pc + (uint32_t)(int32_t)(int8_t)b1) & 0xFFFF;
                    ncyc = 3 + (((t ^ pc) & 0xFF00) ? 1 : 0);
                    pc = t;
                }
                break;
            }
            case O_JMP: pc = ea; break;
            case O_JSR: {
                uint32_t ret = (pc - 1) & 0xFFFF;       // address of the last operand byte
                // pushes go through the full bus (the stack pointer may sit in TIA space)
                uint32_t sa = 0x100 | sp;
                if ((sa & 0x1280) == 0x0080) ram.wr(sa, ret >> 8);
                else if (!(sa & 0x1080)) stall += tia_poke<VERIFY>(s, T, sa & 0x3F, ret >> 8, cyc + 4, cpu_ls, fb);
                sp = (sp - 1) & 0xFF; sa = 0x100 | sp;
                if ((sa & 0x1280) == 0x0080) ram.wr(sa, ret & 0xFF);
                else if (!(sa & 0x1080)) stall += tia_poke<VERIFY>(s, T, sa & 0x3F, ret & 0xFF, cyc + 5, cpu_ls, fb);
                sp = (sp - 1) & 0xFF;
                pc = ea;
                break;
            }
            case O_RTS: {
                sp = (sp + 1) & 0xFF; uint32_t lo = bus_read<VERIFY>(s, T, ram, 0x100 | sp, cyc, 0, fb);
                sp = (sp + 1) & 0xFF; uint32_t hi = bus_read<VERIFY>(s, T, ram, 0x100 | sp, cyc, lo, fb);
                pc = ((lo | (hi << 8)) + 1) & 0xFFFF; break;
            }
            case O_RTI: {
                sp = (sp + 1) & 0xFF; uint32_t p = bus_read<VERIFY>(s, T, ram, 0x100 | sp, cyc, 0, fb);
                fc = p & 1; zv = (p & 2) ? 0 : 1; fid = p & 0x0C; fv = (p >> 6) & 1; nv = p & 0x80;
                sp = (sp + 1) & 0xFF; uint32_t lo = bus_read<VERIFY>(s, T, ram, 0x100 | sp, cyc, p, fb);
                sp = (sp + 1) & 0xFF; uint32_t hi = bus_read<VERIFY>(s, T, ram, 0x100 | sp, cyc, lo, fb);
                pc = lo | (hi << 8); break;
            }
            case O_BRK: {
                uint32_t ret = (pc + 1) & 0xFFFF;
                uint32_t p = fc | (((zv & 0xFF) == 0) << 1) | fid | 0x30 | (fv << 6) | (nv & 0x80);
                uint32_t vals[3] = {ret >> 8, ret & 0xFF, p};
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    uint32_t sa = 0x100 | sp;
                    if ((sa & 0x1280) == 0x0080) ram.wr(sa, vals[k]);
                    else if (!(sa & 0x1080)) stall += tia_poke<VERIFY>(s, T, sa & 0x3F, vals[k], cyc + 3 + k, cpu_ls, fb);
                    sp = (sp - 1) & 0xFF;
                }
                fid |= 4u;
                pc = rom_byte(T, 0x7FE) | (rom_byte(T, 0x7FF) << 8);
                break;
            }
            case O_PHA: case O_PHP: {
                uint32_t val = op == O_PHA ? a : (fc | (((zv & 0xFF) == 0) << 1) | fid | 0x30 | (fv << 6) | (nv & 0x80));
                ea = 0x100 | sp; wv = val; sp = (sp - 1) & 0xFF;
                break;
            }
            case O_PLA: sp = (sp + 1) & 0xFF; a = bus_read<VERIFY>(s, T, ram, 0x100 | sp, cyc_after, 0, fb); nv = zv = a; break;
            case O_PLP: {
                sp = (sp + 1) & 0xFF; uint32_t p = bus_read<VERIFY>(s, T, ram, 0x100 | sp, cyc_after, 0, fb);
                fc = p & 1; zv = (p & 2) ? 0 : 1; fid = p & 0x0C; fv = (p >> 6) & 1; nv = p & 0x80; break;
            }
            default: s.error = ERR_ILLEGAL_OPCODE; break;
            }
            if ((d & DF_WRITE) || op == O_PHA || op == O_PHP) {
                const uint32_t wa = ea & 0x1FFF;
                const uint32_t t_after = cyc + ncyc;
                if ((wa & 0x1280) == 0x0080) ram.wr(wa, wv);
                else if (!(wa & 0x1080)) stall += tia_poke<VERIFY>(s, T, wa & 0x3F, wv, t_after, cpu_ls, fb);
                else if ((wa & 0x1280) == 0x0280) riot_poke(s, wa, wv, t_after);
            }
            cyc += ncyc + stall;
        }
        while ((int32_t)(cyc - (cpu_ls + LINE_CYCLES)) >= 0) cpu_ls += LINE_CYCLES;
    }
    // complete the picture up to the CPU's clock
    tia_catchup<VERIFY>(s, T, 3 * (int)(cyc - s.tia_ls), fb);
    r.a = a; r.x = x; r.y = y; r.sp = sp; r.pc = pc; r.c = fc; r.v = fv; r.nv = nv; r.zv = zv; r.id = fid;
    r.cyc = cyc; r.cpu_ls = cpu_ls;
}

__device__ __forceinline__ uint32_t pack_p(const CpuRegs &r)
{
    return r.c | (((r.zv & 0xFF) == 0) << 1) | r.id | 0x20 | (r.v << 6) | (r.nv & 0x80);
}

// power-on state (matches a26o_power_on in the oracle)
__device__ __forceinline__ void power_on(Chip &s, CpuRegs &r, const Tables &T, Ram ram, const uint32_t *needed_tab)
{
    uint8_t *p = reinterpret_cast<uint8_t *>(&s);
    for (unsigned i = 0; i < sizeof(Chip); ++i) p[i] = 0;
    for (uint32_t a = 0; a < 128; ++a) ram.wr(a, 0);
    r.a = r.x = r.y = 0; r.sp = 0xFD;
    r.c = 0; r.v = 0; r.nv = 0; r.zv = 1; r.id = 4;
    r.pc = rom_byte(T, 0x7FC) | (rom_byte(T, 0x7FD) << 8);
    r.cyc = 0; r.cpu_ls = 0;
    s.swcha = 0xFF; s.swchb = 0x3F;
    s.timer_shift = 10; s.timer_value = 0; s.timer_set = 0;
    for (int i = 0; i < 4; ++i) { s.charge[i] = TRIGMAX / 2; s.needed[i] = needed_tab[TRIGMAX / 2]; }
}

#endif  // __CUDACC__
}  // namespace a26
