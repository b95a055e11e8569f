// host_sim.cpp -- TEST INFRASTRUCTURE.  Compiles the device-side source of the CUDA core
// (csrc/a26_core.cuh, policy.cuh, rollout.cuh) for the CPU behind a small intrinsics shim, so the
// kernel logic can be debugged against the oracle in the build container, which has no GPU.  It is
// not part of the product library, is never loaded by the package, and proves nothing about the
// GPU build: the `-m gpu` parity tests do that through libngp.so.
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <vector>

#define __CUDACC__ 1
#define __device__
#define __host__
#define __global__
#define __forceinline__ inline
#define __noinline__
static inline int __popc(uint32_t v) { return __builtin_popcount(v); }
static inline uint32_t __brev(uint32_t v)
{
    v = ((v >> 1) & 0x55555555u) | ((v & 0x55555555u) << 1);
    v = ((v >> 2) & 0x33333333u) | ((v & 0x33333333u) << 2);
    v = ((v >> 4) & 0x0F0F0F0Fu) | ((v & 0x0F0F0F0Fu) << 4);
    return __builtin_bswap32(v);
}
static inline uint32_t __funnelshift_r(uint32_t lo, uint32_t hi, uint32_t sh)
{
    sh &= 31;
    return sh ? (lo >> sh) | (hi << (32 - sh)) : lo;
}
static inline uint32_t __umulhi(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }
static inline double __ddiv_rn(double a, double b) { return a / b; }
static inline double __dmul_rn(double a, double b) { return a * b; }
static inline double __dadd_rn(double a, double b) { return a + b; }
static inline double __dsub_rn(double a, double b) { return a - b; }
static inline double __longlong_as_double(long long v) { double d; memcpy(&d, &v, 8); return d; }
template <typename T> static inline T __ldg(const T *p) { return *p; }
static inline void __syncthreads() {}
static inline unsigned __activemask() { return 1u; }
static inline int __all_sync(unsigned, int v) { return v; }
static inline unsigned __ballot_sync(unsigned, int v) { return v ? 1u : 0u; }
static inline int __syncthreads_or(int v) { return v; }

#include "../../neuro_genetic_pong_self_play_b200/csrc/game_state.cuh"
#include "../../neuro_genetic_pong_self_play_b200/csrc/host_tables.h"

namespace {
struct Sim {
    a26::Tables T;
    std::vector<uint32_t> needed;
    a26::Snapshot start[2];
    // one stepwise env
    a26::Chip s;
    a26::CpuRegs r;
    uint32_t ram_words[32 * 32];   // lane 0 of a warp-interleaved block
    int players = 2;               // the robot game ('Start') is made with players=1 (main.py:40)
    uint8_t button_map[16];        // ngp_default_config's
};
}  // namespace

extern "C" {

// a simulator whose find_stuff looks for other target colours (ngp_config.ball_colour / left_colour / right_colour): a colour
// that matches nothing hides that object from the observation, e.g. to force get_actions' random fall-back
void *hs_create_colours(const uint8_t *rom, const uint8_t *ball, const uint8_t *left, const uint8_t *right)
{
    Sim *sim = new Sim();
    ngp_host::build_tables(sim->T, rom, ball, left, right, ngp_host::ntsc_palette);
    ngp_host::default_button_map(sim->button_map);
    sim->needed.resize(a26::TRIGMAX + 1);
    ngp_host::build_paddle_table(sim->needed.data());
    a26::Ram ram{sim->ram_words};
    for (int st = 0; st < 2; ++st) {
        roll::build_start_state(st, sim->s, sim->r, sim->T, ram, sim->needed.data());
        roll::store_snapshot(&sim->start[st], sim->s, sim->r, ram);
    }
    return sim;
}
void *hs_create(const uint8_t *rom)
{
    const uint8_t ball[3] = {236, 236, 236}, left[3] = {213, 130, 74}, right[3] = {92, 186, 92};     // ngp_default_config's
    return hs_create_colours(rom, ball, left, right);
}
void hs_destroy(void *h) { delete (Sim *)h; }

void hs_env_reset(void *h, int state)
{
    Sim *sim = (Sim *)h;
    roll::load_snapshot(&sim->start[state], sim->s, sim->r, a26::Ram{sim->ram_words});
    sim->players = state == NGP_STATE_START_1P ? 1 : 2;
}
void hs_env_power_on(void *h)
{
    Sim *sim = (Sim *)h;
    a26::power_on(sim->s, sim->r, sim->T, a26::Ram{sim->ram_words}, sim->needed.data());
    sim->players = 2;
}

// raw console input step (like a26o_run_frame)
int hs_env_run_frame(void *h, int core, int swchb, int fire, int dec, int inc, uint8_t *ram_out, uint8_t *fb, double *loc, uint8_t *valid,
                     uint8_t *regs, uint32_t *digest)
{
    Sim *sim = (Sim *)h;
    a26::Ram ram{sim->ram_words};
    a26::Chip &s = sim->s;
    a26::apply_input(s, sim->needed.data(), (uint32_t)swchb, (uint32_t)fire, (uint32_t)dec, (uint32_t)inc);
    a26::clear_obs(s);
    if (fb) memset(fb, 0, 210 * 160);
    if (core) a26::run_frame_compiled<true, false>(s, sim->r, sim->T, ram, fb);
    else a26::run_frame<true>(s, sim->r, sim->T, ram, fb);
    if (ram_out) for (int i = 0; i < 128; ++i) ram_out[i] = (uint8_t)ram.rd(i);
    if (loc && valid)
        for (int t = 0; t < 3; ++t) {
            valid[t] = s.cnt[t] > 0;
            loc[2 * t] = s.cnt[t] ? (double)s.sy[t] / (double)s.cnt[t] : 0.0;
            loc[2 * t + 1] = s.cnt[t] ? (double)s.sx[t] / (double)s.cnt[t] : 0.0;
        }
    if (regs) {
        const a26::CpuRegs &r = sim->r;
        regs[0] = (uint8_t)r.a; regs[1] = (uint8_t)r.x; regs[2] = (uint8_t)r.y; regs[3] = (uint8_t)r.sp; regs[4] = (uint8_t)a26::pack_p(r);
        regs[5] = (uint8_t)r.pc; regs[6] = (uint8_t)(r.pc >> 8); regs[7] = s.error;
    }
    if (digest) {
        digest[0] = s.cx;
        digest[1] = (uint32_t)s.posp0 | ((uint32_t)s.posp1 << 8) | ((uint32_t)s.posm0 << 16) | ((uint32_t)s.posm1 << 24);
        digest[2] = (uint32_t)s.posbl | ((uint32_t)s.vblank << 8) | ((uint32_t)s.ctrlpf << 16) | ((uint32_t)s.vdelbl << 24);
        digest[3] = (uint32_t)s.charge[0] | ((uint32_t)s.charge[1] << 16);
        digest[4] = (uint32_t)s.charge[2] | ((uint32_t)s.charge[3] << 16);
        digest[5] = (uint32_t)s.grp0_new | ((uint32_t)s.grp1_new << 8) | ((uint32_t)s.enabl_new << 16) | ((uint32_t)s.enabl_old << 24);
        digest[6] = (sim->r.cyc - sim->r.cpu_ls) % a26::LINE_CYCLES;
        digest[7] = s.dump_enabled;
    }
    return s.error;
}

// the fused (no framebuffer) flavour of one frame: what rollout_kernel executes
int hs_env_step_fast(void *h, int core, const uint8_t *action16, uint8_t *ram_out, double *loc, uint8_t *valid)
{
    Sim *sim = (Sim *)h;
    a26::Ram ram{sim->ram_words};
    a26::Chip &s = sim->s;
    const uint32_t in = roll::action_to_input(action16, sim->players, sim->button_map);
    a26::apply_input(s, sim->needed.data(), in & 0xFF, (in >> 8) & 15, (in >> 12) & 15, (in >> 16) & 15);
    a26::clear_obs(s);
    if (core) a26::run_frame_compiled<false, false>(s, sim->r, sim->T, ram, nullptr);
    else a26::run_frame<false>(s, sim->r, sim->T, ram, nullptr);
    for (int i = 0; i < 128; ++i) ram_out[i] = (uint8_t)ram.rd(i);
    for (int t = 0; t < 3; ++t) {
        valid[t] = s.cnt[t] > 0;
        loc[2 * t] = s.cnt[t] ? (double)s.sy[t] / (double)s.cnt[t] : 0.0;
        loc[2 * t + 1] = s.cnt[t] ? (double)s.sx[t] / (double)s.cnt[t] : 0.0;
    }
    return s.error;
}

int hs_env_step(void *h, int core, const uint8_t *action16, uint8_t *ram_out, uint8_t *fb, double *loc, uint8_t *valid, uint8_t *regs, uint32_t *digest)
{
    const Sim *sim = (Sim *)h;
    const uint32_t in = roll::action_to_input(action16, sim->players, sim->button_map);
    return hs_env_run_frame(h, core, in & 0xFF, (int)((in >> 8) & 15), (int)((in >> 12) & 15), (int)((in >> 16) & 15), ram_out, fb, loc, valid, regs, digest);
}

}  // extern "C"

// RolloutParams as rollout_params (csrc/ngp_core.cu) fills them for ngp_default_config with this network, core and max_frames;
// the caller adds the population or the match list and the outputs
static roll::RolloutParams rollout_params(Sim *sim, int core, const int32_t *nodes, int n_layers, int bias, int max_frames, uint64_t seed,
                                          uint64_t generation)
{
    roll::RolloutParams p = {};
    p.tables = &sim->T; p.needed = sim->needed.data(); p.start = sim->start;
    p.win_score = 3; p.timeout_thresh = 2000; p.max_frames = max_frames;
    p.core = core; p.time_scaler = 100.0; p.paddle_height = 16.0; p.seed = seed; p.generation = generation;
    p.shape.n_layers = n_layers; p.shape.bias = bias;
    for (int i = 0; i < n_layers; ++i) p.shape.nodes[i] = nodes[i];
    p.G = pol::gene_size(p.shape);
    roll::fill_input_table(p, sim->button_map);
    return p;
}

// One lane of rollout_kernel (csrc/rollout_kernel.cuh) from the start to the end of environment e's episode, in the kernel's
// order: episode_begin; with REC the start state and the capture at frame 0; every frame episode_frame, then with REC
// record_frame and the capture after that frame; at the end reward, frame count and scores as the kernel stores them.
// Returns the frames played.
template <int CORE, bool REC>
static uint64_t play_lane(Sim *sim, const roll::RolloutParams &p, const roll::RecordArgs &rec, int e)
{
    a26::Ram ram{sim->ram_words};
    a26::Chip s; a26::CpuRegs r;
    roll::Episode ep;
    roll::episode_begin(ep, p, e, s, r, ram);
    if (REC && rec.start && rec.start[e] >= 0) roll::resume_state(rec, rec.start[e], ep, s, r, ram);
    const int capture_at = REC && rec.capture_at ? rec.capture_at[e] : -1;
    if (capture_at == ep.frame) roll::capture_state(rec, ep, s, r, ram);
    uint64_t frames = 0;
    double reward;
    for (bool done = false; !done; ++frames) {
        done = roll::episode_frame<CORE, false, REC>(ep, p, s, r, sim->T, ram, &reward, true, &rec);
        if (REC && rec.record && ep.frame <= rec.max_record) roll::record_frame(rec, ep, s, ep.last_s1, ep.last_s2);
        if (REC && !done && ep.frame == capture_at) roll::capture_state(rec, ep, s, r, ram);
    }
    p.rewards[e] = reward;
    p.frames[e] = ep.frame;
    if (p.scores) { p.scores[2 * e] = ep.last_s1; p.scores[2 * e + 1] = ep.last_s2; }
    return frames;
}

// every environment of p, lanes executed one after another; returns the frames played
template <bool REC>
static uint64_t play_lanes(Sim *sim, const roll::RolloutParams &p, const roll::RecordArgs &rec)
{
    uint64_t frames = 0;
    for (int e = 0; e < p.n * p.games; ++e) frames += p.core ? play_lane<1, REC>(sim, p, rec, e) : play_lane<0, REC>(sim, p, rec, e);
    return frames;
}

extern "C" {

// fused evaluation (ngp_evaluate)
void hs_evaluate(void *h, int core, const int32_t *nodes, int n_layers, int bias, int schedule, int games, int max_frames, const float *genomes, int n,
                 const float *hof_genomes, const double *hof_fitness, int n_hof, const int32_t *hof_pick, uint64_t seed,
                 uint64_t generation, double *rewards, int32_t *frames)
{
    roll::RolloutParams p = rollout_params((Sim *)h, core, nodes, n_layers, bias, max_frames, seed, generation);
    p.genomes = genomes; p.hof_genomes = hof_genomes; p.hof_fitness = hof_fitness; p.hof_pick = hof_pick;
    p.n = n; p.n_hof = n_hof; p.games = games; p.schedule = schedule;
    p.rewards = rewards; p.frames = frames;
    play_lanes<false>((Sim *)h, p, roll::RecordArgs{});
}

int hs_validate_state(const ngp_game_state *st, uint64_t cart) { return gs::validate(st, cart); }

// A match list: ngp_play_matches, ngp_record_matches and ngp_play_matches_states.  First the list check of match_check_kernel
// (gs::match_entry_faults per match, gs::validate per start state): with any fault nothing is played or written and the
// number of faults is returned.  Then every match plays as one lane.  With none of record, key, states, start and capture_at
// the lanes mirror the flavours ngp_play_matches launches (REC = false); with any of them, the recording twins that
// ngp_record_matches and ngp_play_matches_states launch (REC = true).  *frames_total (when given) = the frames played.
long hs_play_list(void *h, int core, const int32_t *nodes, int n_layers, int bias, int max_frames, const float *genomes, int n_genomes,
                  const int32_t *right, const int32_t *left, const double *mult, const int32_t *key, int n_matches,
                  const ngp_game_state *states, int n_states, const int32_t *start, int fresh, const int32_t *capture_at,
                  ngp_game_state *capture, int max_record, ngp_frame_record *record, uint64_t cart, uint64_t seed, uint64_t generation,
                  double *rewards, int32_t *frames, int32_t *scores, uint64_t *frames_total)
{
    long faults = 0;
    for (int m = 0; m < n_matches; ++m)
        faults += gs::match_entry_faults(m, right, left, n_genomes, key, capture_at, start, states, n_states);
    for (int k = 0; k < n_states; ++k) faults += gs::validate(states + k, cart) == 0;
    if (faults) return faults;
    roll::RolloutParams p = rollout_params((Sim *)h, core, nodes, n_layers, bias, max_frames, seed, generation);
    p.genomes = genomes; p.n = n_matches; p.games = 1;
    p.match_right = right; p.match_left = left; p.match_mult = mult;
    p.rewards = rewards; p.frames = frames; p.scores = scores;
    roll::RecordArgs rec = {};
    rec.record = record; rec.key = key; rec.max_record = record ? max_record : 0;
    rec.fresh = fresh; rec.states = states; rec.start = start; rec.capture_at = capture_at; rec.capture = capture; rec.cart = cart;
    const bool twin = record || key || states || start || capture_at;
    const uint64_t total = twin ? play_lanes<true>((Sim *)h, p, rec) : play_lanes<false>((Sim *)h, p, rec);
    if (frames_total) *frames_total = total;
    return 0;
}

// Self-test of the register mirror of the hot latches (csrc/a26_core.cuh: HotLatches, hot_write, hot_display_writes) against
// poke_quick() + the latch effects of tia_apply(), on RANDOM latch states and values -- including states the cartridge never
// visits (delayed players and ball, unlocked missiles).  Returns the number of disagreements (0 = none).
static uint32_t hs_rng(uint64_t &st) { st = st * 6364136223846793005ull + 1442695040888963407ull; return (uint32_t)(st >> 33); }
// what the write-by-write order does with one write: poke_quick's verdict, and the latch effect either way
static bool hs_reference_write(a26::Chip &c, uint32_t reg, uint32_t v)
{
    if (a26::poke_quick(c, reg, v)) {
        if (reg == 0x0E) c.pf1 = (uint8_t)v;          // equal already: poke_quick leaves these two alone
        if (reg == 0x0F) c.pf2 = (uint8_t)v;
        return true;
    }
    switch (reg) {                                    // tia_apply's latch effects (a26_core.cuh)
    case 0x0D: c.pf0 = (uint8_t)v; break;
    case 0x0E: c.pf1 = (uint8_t)v; break;
    case 0x0F: c.pf2 = (uint8_t)v; break;
    case 0x1B: c.grp0_new = (uint8_t)v; c.grp1_old = c.grp1_new; break;
    case 0x1C: c.grp1_new = (uint8_t)v; c.grp0_old = c.grp0_new; c.enabl_old = c.enabl_new; break;
    case 0x1D: c.enam0 = (uint8_t)v; break;
    case 0x1E: c.enam1 = (uint8_t)v; break;
    default: c.enabl_new = (uint8_t)v; break;
    }
    return false;
}
int hs_hot_latch_selftest(uint64_t seed, int rounds)
{
    int bad = 0;
    uint64_t st = seed * 2 + 1;
    for (int it = 0; it < rounds; ++it) {
        a26::Chip c;
        memset(&c, 0, sizeof(c));
        uint8_t *b = &c.pf0;
        for (int i = 0; i < 16; ++i) {
            const uint32_t r = hs_rng(st);
            // a few distinct values per byte, so that equal/unequal, enabled/disabled and delayed/undelayed all come up often
            const uint8_t pool[6] = {0x00, 0xF0, 0x02, 0x01, 0x03, (uint8_t)(r >> 8)};
            b[i] = pool[r % 6];
        }
        uint32_t v[8];
        for (int i = 0; i < 8; ++i) { const uint32_t r = hs_rng(st); const uint8_t pool[6] = {0x00, 0xF0, 0x02, 0x32, 0xB1, (uint8_t)(r >> 8)}; v[i] = pool[r % 6]; }
        const uint32_t regs[8] = {0x1B, 0x1E, 0x1D, 0x1C, 0x0D, 0x0E, 0x0F, 0x1F};        // the display loop's program order
        // (1) one write at a time, every register
        for (int i = 0; i < 8; ++i) {
            a26::Chip ref = c;
            a26::HotLatches h;
            a26::hot_load(h, c);
            const bool q_ref = hs_reference_write(ref, regs[i], v[i]);
            bool q;
            switch (regs[i]) {
            case 0x0D: q = a26::hot_write<0x0D>(h, v[i]); break;
            case 0x0E: q = a26::hot_write<0x0E>(h, v[i]); break;
            case 0x0F: q = a26::hot_write<0x0F>(h, v[i]); break;
            case 0x1B: q = a26::hot_write<0x1B>(h, v[i]); break;
            case 0x1C: q = a26::hot_write<0x1C>(h, v[i]); break;
            case 0x1D: q = a26::hot_write<0x1D>(h, v[i]); break;
            case 0x1E: q = a26::hot_write<0x1E>(h, v[i]); break;
            default: q = a26::hot_write<0x1F>(h, v[i]); break;
            }
            a26::Chip got = c;
            a26::hot_store(h, got);
            if (q != q_ref || memcmp(&got.pf0, &ref.pf0, 16) != 0) ++bad;
        }
        // (2) the whole iteration at once: all-quick or nothing
        {
            a26::Chip ref = c;
            bool all = true;
            for (int i = 0; i < 8; ++i) all = hs_reference_write(ref, regs[i], v[i]) && all;
            a26::HotLatches h;
            a26::hot_load(h, c);
            const bool ok = a26::hot_display_writes(h, v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7]);
            a26::Chip got = c;
            a26::hot_store(h, got);
            if (ok != all) ++bad;
            else if (ok && memcmp(&got.pf0, &ref.pf0, 16) != 0) ++bad;
            else if (!ok && memcmp(&got.pf0, &c.pf0, 16) != 0) ++bad;                      // refused: the mirror must be untouched
        }
    }
    return bad;
}

}  // extern "C"
