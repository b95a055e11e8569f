// game_state.cuh -- the one module that knows the byte layout of ngp_game_state (include/ngp.h): pack, unpack, validate
// and seal, as __host__ __device__ code shared by the recording twins of the fused rollout (rollout_kernel.cuh), the
// stepwise get/set kernels (ngp_core.cu) and tests/host_sim.
//
// Layout, in 32-bit little-endian words (DESIGN.md section 4, "save states"):
//   [0, 8)     header: magic, version, cartridge hash (fnv1a64 of the 2 KiB image, low word first), players (1 or 2),
//              has_episode (0 or 1), 0, 0
//   [8, 96)    console: a26::Snapshot = Chip (44 words), CpuRegs (12), RAM (32)
//   [96, 108)  episode (perform_episode's locals, main.py:70-75; all zero without one): frame, timeout, total_frames,
//              last_s1, last_s2, have_last_score | have_last_ball << 8 | left_act << 16 | right_act << 24, 0, 0,
//              last_ball[0] (f64), last_ball[1] (f64)
//   [108, 126) zero
//   [126, 128) checksum: FNV-1a over words 0..125 (one 64-bit xor-multiply per word), low word first
// Canonical bytes: Chip's playfield-mask cache is written stale (pf_dirty = 1, pfmask = 0), its observation accumulators
// (cleared by every step) and all padding as zero, and last_ball as zero while have_last_ball is false, so equal console
// and episode states give equal bytes whichever core, rollout flavour or entry point wrote them.
#pragma once
#include <stddef.h>

#include "rollout.cuh"

namespace gs {
using a26::Chip; using a26::CpuRegs; using a26::Ram; using a26::Snapshot;

constexpr uint32_t MAGIC = 0x5453474Eu;            // "NGST"
constexpr uint32_t VERSION = 1;
constexpr int WORDS = NGP_GAME_STATE_BYTES / 4;
constexpr int W_CHIP = 8, W_CPU = W_CHIP + (int)sizeof(Chip) / 4, W_RAM = W_CPU + (int)sizeof(CpuRegs) / 4, W_EPISODE = W_RAM + 32,
              W_SUM = WORDS - 2;

static_assert(sizeof(ngp_game_state) == 512, "ngp_game_state is 512 bytes");
static_assert(sizeof(Chip) == 176 && sizeof(CpuRegs) == 48 && sizeof(Snapshot) == 352, "the layout above");
static_assert(W_EPISODE + 12 <= W_SUM, "the episode fits before the checksum");
static_assert(offsetof(Chip, error) % 4 == 0 && offsetof(Chip, pf_dirty) == offsetof(Chip, error) + 1 &&
              offsetof(Chip, pad1) == offsetof(Chip, error) + 2 && offsetof(Chip, pad2) == offsetof(Chip, error) + 3,
              "error, pf_dirty, pad1, pad2 share one word");
static_assert(offsetof(Chip, cx) % 4 == 0 && offsetof(Chip, pad3) == offsetof(Chip, cx) + 2, "cx, pad3 share one word");
static_assert(offsetof(Chip, pfmask) % 4 == 0 && offsetof(Chip, cnt) % 4 == 0 &&
              offsetof(Chip, sy) + sizeof(uint32_t[3]) == offsetof(Chip, cnt) + sizeof(uint32_t[9]),
              "the observation accumulators are Chip's last members");

// word k of Chip in canonical form
__host__ __device__ __forceinline__ uint32_t chip_word(const Chip &s, int k)
{
    const size_t b = 4 * (size_t)k;
    if (b >= offsetof(Chip, pfmask) && b < offsetof(Chip, pfmask) + sizeof(s.pfmask)) return 0;   // a cache, rebuilt on use
    if (b >= offsetof(Chip, cnt)) return 0;                // cnt, sx, sy (clear_obs resets them every step) and tail padding
    const uint32_t w = reinterpret_cast<const uint32_t *>(&s)[k];
    if (b == offsetof(Chip, error)) return (w & 0xFFu) | 0x100u;     // error; pf_dirty = 1; pad1 = pad2 = 0
    if (b == offsetof(Chip, cx)) return w & 0xFFFFu;                  // cx; pad3 = 0
    return w;
}

__host__ __device__ __forceinline__ uint32_t lo32(double v)
{
#ifdef __CUDA_ARCH__
    return (uint32_t)__double2loint(v);
#else
    uint64_t u; memcpy(&u, &v, 8); return (uint32_t)u;
#endif
}
__host__ __device__ __forceinline__ uint32_t hi32(double v)
{
#ifdef __CUDA_ARCH__
    return (uint32_t)__double2hiint(v);
#else
    uint64_t u; memcpy(&u, &v, 8); return (uint32_t)(u >> 32);
#endif
}
__host__ __device__ __forceinline__ double f64(uint32_t lo, uint32_t hi)
{
#ifdef __CUDA_ARCH__
    return __hiloint2double((int)hi, (int)lo);
#else
    const uint64_t u = (uint64_t)hi << 32 | lo; double v; memcpy(&v, &u, 8); return v;
#endif
}

// 16-byte chunk c of a state: one vector access on the device (state arrays are 16-byte aligned)
__host__ __device__ __forceinline__ void load4(const ngp_game_state *st, int c, uint32_t w[4])
{
#ifdef __CUDA_ARCH__
    const uint4 q = reinterpret_cast<const uint4 *>(st)[c];
    w[0] = q.x; w[1] = q.y; w[2] = q.z; w[3] = q.w;
#else
    memcpy(w, st->b + 16 * c, 16);
#endif
}
__host__ __device__ __forceinline__ void store4(ngp_game_state *st, int c, const uint32_t w[4])
{
#ifdef __CUDA_ARCH__
    reinterpret_cast<uint4 *>(st)[c] = make_uint4(w[0], w[1], w[2], w[3]);
#else
    memcpy(st->b + 16 * c, w, 16);
#endif
}

__host__ __device__ __forceinline__ uint64_t checksum_step(uint64_t h, uint32_t w) { return (h ^ w) * 1099511628211ull; }
constexpr uint64_t CHECKSUM_INIT = 14695981039346656037ull;

// perform_episode's locals as the 12 episode words
__host__ __device__ __forceinline__ void episode_words(const roll::Episode &ep, uint32_t w[12])
{
    w[0] = (uint32_t)ep.frame; w[1] = (uint32_t)ep.timeout; w[2] = (uint32_t)ep.total_frames;
    w[3] = (uint32_t)ep.last_s1; w[4] = (uint32_t)ep.last_s2;
    w[5] = (uint32_t)ep.have_last_score | (uint32_t)ep.have_last_ball << 8 | (uint32_t)ep.left_act << 16 | (uint32_t)ep.right_act << 24;
    w[6] = w[7] = 0;
    const double b0 = ep.have_last_ball ? ep.last_ball[0] : 0.0, b1 = ep.have_last_ball ? ep.last_ball[1] : 0.0;
    w[8] = lo32(b0); w[9] = hi32(b0); w[10] = lo32(b1); w[11] = hi32(b1);
}

// RAM word sources: the rollout lane's interleaved shared memory, or a Snapshot's bytes
struct LaneRam {
    Ram ram;
    __host__ __device__ __forceinline__ uint32_t get(int i) const { return ram.base[i * 32]; }
    __host__ __device__ __forceinline__ void set(int i, uint32_t v) const { ram.base[i * 32] = v; }
};
struct SnapRam {
    uint8_t *bytes;
    __host__ __device__ __forceinline__ uint32_t get(int i) const { return reinterpret_cast<const uint32_t *>(bytes)[i]; }
    __host__ __device__ __forceinline__ void set(int i, uint32_t v) const { reinterpret_cast<uint32_t *>(bytes)[i] = v; }
};

// Writes and seals state `dst` from a console and, when `ep` is given, an episode: 32 16-byte stores.  The loops over the
// 16-byte chunks here and below stay rolled: this is cold code inside the rollout kernels, whose speed depends on the
// instruction footprint of the hot code around it.
template <class RamSrc>
__host__ __device__ __forceinline__ void pack(ngp_game_state *dst, uint64_t cart, int players, const Chip &s, const CpuRegs &r, RamSrc ram,
                                              const uint32_t *ep)
{
    uint64_t h = CHECKSUM_INIT;
#pragma unroll 1
    for (int c = 0; c < WORDS / 4; ++c) {
        uint32_t w[4];
        for (int j = 0; j < 4; ++j) {
            const int i = 4 * c + j;
            uint32_t v;
            if (i == 0) v = MAGIC;
            else if (i == 1) v = VERSION;
            else if (i == 2) v = (uint32_t)cart;
            else if (i == 3) v = (uint32_t)(cart >> 32);
            else if (i == 4) v = (uint32_t)players;
            else if (i == 5) v = ep ? 1u : 0u;
            else if (i < W_CHIP) v = 0;
            else if (i < W_CPU) v = chip_word(s, i - W_CHIP);
            else if (i < W_RAM) v = reinterpret_cast<const uint32_t *>(&r)[i - W_CPU];
            else if (i < W_EPISODE) v = ram.get(i - W_RAM);
            else if (i < W_EPISODE + 12) v = ep ? ep[i - W_EPISODE] : 0u;
            else if (i < W_SUM) v = 0;
            else v = i == W_SUM ? (uint32_t)h : (uint32_t)(h >> 32);
            if (i < W_SUM) h = checksum_step(h, v);
            w[j] = v;
        }
        store4(dst, c, w);
    }
}

// Console (and, when `ep` is given and the state has one, the episode) of a state that validate() accepted.
template <class RamDst>
__host__ __device__ __forceinline__ void unpack(const ngp_game_state *st, Chip &s, CpuRegs &r, RamDst ram, roll::Episode *ep)
{
    uint32_t *cw = reinterpret_cast<uint32_t *>(&s), *rw = reinterpret_cast<uint32_t *>(&r);
    bool has_episode = false;
#pragma unroll 1
    for (int c = 0; c < W_SUM / 4; ++c) {
        uint32_t w[4];
        load4(st, c, w);
        for (int j = 0; j < 4; ++j) {
            const int i = 4 * c + j;
            if (i == 5) has_episode = w[j] != 0;
            else if (i >= W_CHIP && i < W_CPU) cw[i - W_CHIP] = w[j];
            else if (i >= W_CPU && i < W_RAM) rw[i - W_CPU] = w[j];
            else if (i >= W_RAM && i < W_EPISODE) ram.set(i - W_RAM, w[j]);
        }
    }
    if (!ep || !has_episode) return;
    uint32_t e[12];
    for (int c = 0; c < 3; ++c) load4(st, W_EPISODE / 4 + c, e + 4 * c);
    ep->frame = (int)e[0]; ep->timeout = (int)e[1]; ep->total_frames = (int)e[2]; ep->last_s1 = (int)e[3]; ep->last_s2 = (int)e[4];
    ep->have_last_score = (e[5] & 0xFF) != 0; ep->have_last_ball = (e[5] >> 8 & 0xFF) != 0;
    ep->left_act = (int)(e[5] >> 16 & 0xFF); ep->right_act = (int)(e[5] >> 24);
    ep->last_ball[0] = f64(e[8], e[9]); ep->last_ball[1] = f64(e[10], e[11]);
}

// The players value (1 or 2) of a valid state, 0 when it is not one: right magic and version, this cartridge's hash, players
// 1 or 2, has_episode 0 or 1, decisions that are NGP_ACT_* codes, and a matching checksum.  Nothing else may reach unpack.
__host__ __device__ __forceinline__ int validate(const ngp_game_state *st, uint64_t cart)
{
    uint64_t h = CHECKSUM_INIT;
    uint32_t hdr[8], acts = 0, sum[2] = {0, 0};
#pragma unroll 1
    for (int c = 0; c < WORDS / 4; ++c) {
        uint32_t w[4];
        load4(st, c, w);
        for (int j = 0; j < 4; ++j) {
            const int i = 4 * c + j;
            if (i < 8) hdr[i] = w[j];
            if (i == W_EPISODE + 5) acts = w[j] >> 16;
            if (i < W_SUM) h = checksum_step(h, w[j]);
            else sum[i - W_SUM] = w[j];
        }
    }
    const bool ok = hdr[0] == MAGIC && hdr[1] == VERSION && hdr[2] == (uint32_t)cart && hdr[3] == (uint32_t)(cart >> 32) &&
                    (hdr[4] == 1 || hdr[4] == 2) && hdr[5] <= 1 && (acts & 0xFF) <= 2 && (acts >> 8) <= 2 &&
                    sum[0] == (uint32_t)h && sum[1] == (uint32_t)(h >> 32);
    return ok ? (int)hdr[4] : 0;
}

// The argument check of the match-list entry points for match m (match_check_kernel, ngp_core.cu): the number of faults of
// entry m -- a right row outside [0, n_genomes), a left entry that is neither a row nor an NGP_OPP_* code, a negative key, a
// negative capture frame, a start index outside [-1, n_states), a start state whose players value disagrees with left[m].
// Start states themselves are validated once each by the caller.
__host__ __device__ __forceinline__ int match_entry_faults(int m, const int32_t *right, const int32_t *left, int n_genomes,
                                                           const int32_t *key, const int32_t *capture_at, const int32_t *start,
                                                           const ngp_game_state *states, int n_states)
{
    const int r = right[m], l = left[m];
    int c = (r < 0 || r >= n_genomes) + (l < NGP_OPP_ROBOT || l >= n_genomes) + (key && key[m] < 0) + (capture_at && capture_at[m] < 0);
    if (start) {
        const int k = start[m];
        if (k < -1 || k >= n_states) ++c;
        else if (k >= 0) {
            uint32_t w[4];
            load4(states + k, 1, w);                        // header word 4: players
            c += w[0] != (l == NGP_OPP_ROBOT ? 1u : 2u);
        }
    }
    return c;
}

}  // namespace gs

namespace roll {
// ngp_play_matches_states: match ep.env starts from rec.states[k] (validated by the list check).  Out of line like
// record_frame: the unpack's stores, inlined, would be spread over the register-capped twins.
static __device__ __noinline__ void resume_state(const RecordArgs &rec, int k, Episode &ep, Chip &s, CpuRegs &r, Ram ram)
{
    gs::unpack(rec.states + k, s, r, gs::LaneRam{ram}, rec.fresh ? nullptr : &ep);
}

// ngp_play_matches_states: the state of match ep.env (console and episode) to rec.capture[ep.env], as 16-byte stores.
static __device__ __noinline__ void capture_state(const RecordArgs &rec, const Episode &ep, const Chip &s, const CpuRegs &r, Ram ram)
{
    uint32_t w[12];
    gs::episode_words(ep, w);
    gs::pack(rec.capture + ep.env, rec.cart, ep.plan.state == NGP_STATE_START_1P ? 1 : 2, s, r, gs::LaneRam{ram}, w);
}
}  // namespace roll
