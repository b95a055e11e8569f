// rollout.cuh -- per-lane pieces of the fused population-evaluation rollout (device functions
// without any thread-index dependence, so tests/host_sim can execute the same source on the CPU
// for debugging).  Reference path: main.evaluate 28-66, main.perform_episode 69-112,
// main.get_actions 138-154, main.calculate_timeout_and_frames 128-135, utils.calculate_reward 104-109.
#pragma once
#include <string.h>

#include "../../include/ngp.h"
#include "a26_compiled.cuh"
#include "policy.cuh"

namespace roll {
using a26::Chip; using a26::CpuRegs; using a26::Ram; using a26::Snapshot; using a26::Tables;

#ifdef __CUDACC__

__device__ __forceinline__ void load_snapshot(const Snapshot *__restrict__ src, Chip &s, CpuRegs &r, Ram ram)
{
    s = src->chip;
    r = src->cpu;
    const uint32_t *w = reinterpret_cast<const uint32_t *>(src->ram);
#pragma unroll 4
    for (int i = 0; i < 32; ++i) ram.base[i * 32] = w[i];
}
__device__ __forceinline__ void store_snapshot(Snapshot *dst, const Chip &s, const CpuRegs &r, Ram ram)
{
    dst->chip = s;
    dst->cpu = r;
    uint32_t *w = reinterpret_cast<uint32_t *>(dst->ram);
#pragma unroll 4
    for (int i = 0; i < 32; ++i) w[i] = ram.base[i * 32];
}

// gym-retro button vector -> console input through the configurable button map (ngp_config.button_map; include/ngp.h
// NGP_BTN_*; DESIGN.md "button map").  An environment made with players=1 (main.py:40) consumes only a[0:8].
// FILTERED (main.py:23,55): UP+DOWN or LEFT+RIGHT of one player cancel.  Returns swchb | fire << 8 | dec << 12 | inc << 16.
__host__ __device__ __forceinline__ uint32_t action_to_input(const uint8_t *a, int players, const uint8_t *map)
{
    uint32_t swchb = 0x3F, fire = 0, dec = 0, inc = 0;
    for (int i = 0; i < 8 * players; ++i) {
        if (!a[i]) continue;
        const int j = i & 7;
        if (j >= 4 && a[i ^ 1]) continue;            // opposite direction held too (pairs 4/5 and 6/7)
        const int code = map[i];
        if (code >= NGP_BTN_FIRE_P0 && code <= NGP_BTN_FIRE_P0 + 3) fire |= 1u << (code - NGP_BTN_FIRE_P0);
        else if (code >= NGP_BTN_UP_P0 && code < NGP_BTN_UP_P0 + 8) {
            const int k = code - NGP_BTN_UP_P0;
            if (k & 1) inc |= 1u << (k >> 1); else dec |= 1u << (k >> 1);      // up = lower resistance
        } else if (code == NGP_BTN_SELECT) swchb &= ~0x02u;
        else if (code == NGP_BTN_RESET) swchb &= ~0x01u;
    }
    return swchb | (fire << 8) | (dec << 12) | (inc << 16);
}

// power-on + scripted console switches up to the reference's save states (DESIGN.md "start states")
__device__ __forceinline__ void build_start_state(int state, Chip &s, CpuRegs &r, const Tables &T, Ram ram, const uint32_t *needed)
{
    a26::power_on(s, r, T, ram, needed);
    auto idle = [&](uint32_t swchb, int frames) {
        for (int i = 0; i < frames; ++i) { a26::apply_input(s, needed, swchb, 0, 0, 0); a26::run_frame<false>(s, r, T, ram, nullptr); }
    };
    idle(0x3F, 8);
    if (state == NGP_STATE_START_2P) {              // SELECT twice: game 1 -> game 3 (2-player Pong)
        idle(0x3F & ~0x02u, 1); idle(0x3F, 1);
        idle(0x3F & ~0x02u, 1); idle(0x3F, 1);
    }
    idle(0x3F & ~0x01u, 2);                          // RESET
    idle(0x3F, 1);                                   // <- 'Start' / 'Start.2P'
    idle(0x3F, 1);                                   // gym-retro reset(): one frame without buttons
}

struct RolloutParams {
    const Tables *tables;
    const uint32_t *needed;
    const Snapshot *start;          // [2]
    const float *genomes;           // [n][G]
    const float *hof_genomes;       // [n_hof][G]
    const double *hof_fitness;      // [n_hof]
    const int32_t *hof_pick;        // [n][3] or null
    int n, n_hof, G, games, schedule, win_score, timeout_thresh, max_frames;
    int core;                       // 0 = table-driven interpreter, 1 = statically translated cartridge
    // console input of perform_episode's action vector (BLANK_ACTION with the two decisions written to a[4:6] / a[6:8],
    // config.py:21-23, main.py:91-92) for players = 1, 2 and every (left_act, right_act): action_to_input() done on the host
    uint32_t input_table[2][9];
    double time_scaler, paddle_height;
    uint64_t seed, generation;
    pol::Shape shape;
    double *rewards;                // [n*games]
    int32_t *frames;                // [n*games]
    unsigned long long *counters;   // [0] next env, [1] frames, [2] errors
    // ngp_play_matches (null for ngp_evaluate): environment e is match e of an explicit list, played with games = 1
    const int32_t *match_right;     // [n] genome rows
    const int32_t *match_left;      // [n] genome rows or NGP_OPP_*
    const double *match_mult;       // [n] or null (1.0)
    int32_t *scores;                // [n][2] (score1, score2) at the end of the episode, or null
};

// p.input_table through the button map `map` (ngp_config.button_map)
__host__ inline void fill_input_table(RolloutParams &p, const uint8_t map[16])
{
    for (int players = 1; players <= 2; ++players)
        for (int la = 0; la < 3; ++la)
            for (int ra = 0; ra < 3; ++ra) {
                uint8_t a[16] = {0};
                a[0] = 1; a[15] = 1;                                          // BLANK_ACTION, config.py:21-23
                a[4] = ra == pol::ACT_UP; a[5] = ra == pol::ACT_DOWN;         // action[4:6] = right (main.py:91)
                a[6] = la == pol::ACT_UP; a[7] = la == pol::ACT_DOWN;         // action[6:8] = left (main.py:92)
                p.input_table[players - 1][la * 3 + ra] = action_to_input(a, players, map);
            }
}

// ngp_record_matches and ngp_play_matches_states: a separate kernel argument that only the recording twins of rollout_kernel
// read, so the flavours ngp_evaluate and ngp_play_matches run compile as before
struct RecordArgs {
    ngp_frame_record *record;       // [n][max_record], 16-byte aligned, or null (ngp_play_matches_states without a record)
    const int32_t *key;             // [n] environment index of the fall-back key, or null (= match index)
    int max_record;
    // ngp_play_matches_states (all null otherwise)
    int fresh;                      // states start new episodes from their consoles
    const ngp_game_state *states;   // start states
    const int32_t *start;           // [n] index into states, -1 = the built-in start state
    const int32_t *capture_at;      // [n] env.steps after which the state of match e is written to capture[e]
    ngp_game_state *capture;        // [n]
    uint64_t cart;                  // the cartridge hash written into captured states
};

// Half `half` (16 bytes) of record entry (env, frame): one vector store on the device.
__device__ __forceinline__ void record_store(const RecordArgs &rec, int env, int frame, int half, uint32_t a, uint32_t b, uint32_t c,
                                             uint32_t d)
{
    uint32_t *dst = reinterpret_cast<uint32_t *>(rec.record + (size_t)env * rec.max_record + frame) + 4 * half;
#ifdef __CUDA_ARCH__
    *reinterpret_cast<uint4 *>(dst) = make_uint4(a, b, c, d);
#else
    dst[0] = a; dst[1] = b; dst[2] = c; dst[3] = d;
#endif
}

// the bits of v rounded to float (ngp_env_step's loc rounding)
__device__ __forceinline__ uint32_t f32_bits(double v)
{
    const float f = (float)v;
#ifdef __CUDA_ARCH__
    return __float_as_uint(f);
#else
    uint32_t u;
    memcpy(&u, &f, 4);
    return u;
#endif
}

struct EnvPlan {
    int state;
    int left_kind;
    const float *left_genome;
    const float *right_genome;
    double mult;
};

__device__ __forceinline__ EnvPlan plan_env(const RolloutParams &p, int e)
{
    EnvPlan pl;
    if (p.match_right) {                                   // an explicit match list (ngp_play_matches)
        const int l = p.match_left[e];
        pl.right_genome = p.genomes + (size_t)p.match_right[e] * p.G;
        pl.state = l == NGP_OPP_ROBOT ? NGP_STATE_START_1P : NGP_STATE_START_2P;
        pl.left_kind = l >= 0 ? pol::KIND_MLP : l == NGP_OPP_SCORE_HARDCODED ? pol::KIND_SCORE_HARDCODED : pol::KIND_HARDCODED;
        pl.left_genome = l >= 0 ? p.genomes + (size_t)l * p.G : nullptr;
        pl.mult = p.match_mult ? p.match_mult[e] : 1.0;
        return pl;
    }
    const int g = e / p.games, k = e % p.games;
    pl.right_genome = p.genomes + (size_t)g * p.G;
    pl.state = NGP_STATE_START_2P;
    pl.left_kind = pol::KIND_HARDCODED;
    pl.left_genome = nullptr;
    pl.mult = 1.0;
    if (p.schedule == NGP_SCHEDULE_ROUND_ROBIN) {
        pl.left_kind = pol::KIND_MLP;
        pl.left_genome = p.genomes + (size_t)((g + k + 1) % p.n) * p.G;
    } else {                                               // main.py:33-58
        if (k == 1) pl.state = NGP_STATE_START_1P;
        else if (k == 2) pl.left_kind = pol::KIND_SCORE_HARDCODED;
        else if (k >= 3 && p.n_hof > 0) {
            int h;
            if (p.hof_pick) h = p.hof_pick[g * 3 + (k - 3) % 3];
            else {
                uint32_t o[4];
                pol::philox4x32((uint32_t)g, (uint32_t)k, (uint32_t)p.generation, 0x484F4621u, (uint32_t)p.seed, (uint32_t)(p.seed >> 32), o);
                h = (int)(o[0] % (uint32_t)p.n_hof);
            }
            pl.left_kind = pol::KIND_MLP;
            pl.left_genome = p.hof_genomes + (size_t)h * p.G;
            pl.mult = p.hof_fitness[h];
        }
    }
    return pl;
}

__device__ __forceinline__ int run_policy(const pol::Shape &sh, int kind, const float *genome, const double ball[2], const double last[2],
                                          double me_row, double enemy_row, int s1, int s2)
{
    double x[6] = {__ddiv_rn(ball[1], 160.0), __ddiv_rn(ball[0], 160.0), __ddiv_rn(last[1], 160.0),
                   __ddiv_rn(last[0], 160.0), __ddiv_rn(me_row, 160.0), __ddiv_rn(enemy_row, 160.0)};
    if (kind == pol::KIND_HARDCODED) return pol::hardcoded_ai(x);
    if (kind == pol::KIND_SCORE_HARDCODED) return s1 <= s2 ? pol::hardcoded_ai(x) : pol::ACT_NONE;
    return pol::mlp_small_f64(sh, genome, x, nullptr);
}


// main.perform_episode locals (main.py:70-75)
struct Episode {
    int env;                 // environment index = genome * games + game, or -1 when the lane is idle
    int frame, timeout, total_frames, last_s1, last_s2;
    bool have_last_score, have_last_ball;
    double last_ball[2];
    int left_act, right_act;
    EnvPlan plan;
};

// Record entry ep.frame - 1 of match ep.env (include/ngp.h ngp_frame_record), the frame episode_frame<.., REC = true> has
// just played, as two 16-byte stores; s1, s2 = its scores.  The centroids are recomputed from the chip's counters exactly
// as episode_frame computes them.  Out of line on purpose: inlined (at this point or inside episode_frame, in one or two
// halves) the stores cost the register-capped CTA-synchronous flavours 8-16 B more spill stores and 20-40 B more spill
// loads per frame than the flavours they twin; called, they spill less than those (profiles/r03c_ptxas.txt).
static __device__ __noinline__ void record_frame(const RecordArgs &rec, const Episode &ep, const Chip &s, int s1, int s2)
{
    uint32_t w[6], vb = 0;
#pragma unroll
    for (int t = 0; t < 3; ++t) {
        const bool v = s.cnt[t] > 0;
        vb |= (uint32_t)v << t;
        w[2 * t] = f32_bits(v ? __ddiv_rn((double)s.sy[t], (double)s.cnt[t]) : 0.0);
        w[2 * t + 1] = f32_bits(v ? __ddiv_rn((double)s.sx[t], (double)s.cnt[t]) : 0.0);
    }
    record_store(rec, ep.env, ep.frame - 1, 0, w[0], w[1], w[2], w[3]);
    record_store(rec, ep.env, ep.frame - 1, 1, w[4], w[5], vb | (uint32_t)s1 << 8 | (uint32_t)s2 << 16 | (uint32_t)(ep.left_act | ep.right_act << 2) << 24,
                 (uint32_t)ep.timeout);
}

__device__ __forceinline__ void episode_begin(Episode &ep, const RolloutParams &p, int e, Chip &s, CpuRegs &r, Ram ram)
{
    ep.env = e;
    ep.plan = plan_env(p, e);
    load_snapshot(&p.start[ep.plan.state], s, r, ram);
    ep.frame = 0; ep.timeout = 0; ep.total_frames = 0; ep.last_s1 = ep.last_s2 = 0;
    ep.have_last_score = false; ep.have_last_ball = false;
    ep.last_ball[0] = ep.last_ball[1] = 0.0;
    ep.left_act = ep.right_act = pol::ACT_NONE;
}

// One iteration of perform_episode's loop (main.py:76-107).  Returns true when the episode ended;
// then *reward holds main.py:109-112's value.
// `active` = this lane owns an environment; with SYNC every thread of the CTA must come through here (the
// frame contains CTA-wide barriers), inactive lanes only take part in the barriers.
// REC (ngp_record_matches): the fall-back key is rec->key[ep.env] when given; rollout_kernel then stores the frame with
// record_frame.
template <int CORE, bool SYNC = false, bool REC = false>
__device__ __forceinline__ bool episode_frame(Episode &ep, const RolloutParams &p, Chip &s, CpuRegs &r, const Tables &T, Ram ram,
                                              double *reward, bool active = true, const RecordArgs *rec = nullptr)
{
    if (active) {
        const uint32_t in = p.input_table[ep.plan.state == NGP_STATE_START_1P ? 0 : 1][ep.left_act * 3 + ep.right_act];
        a26::apply_input(s, p.needed, in & 0xFF, (in >> 8) & 15, (in >> 12) & 15, (in >> 16) & 15);
        a26::clear_obs(s);
    }
    if (CORE) a26::run_frame_compiled<false, SYNC>(s, r, T, ram, nullptr, active);
    else if (active) a26::run_frame<false>(s, r, T, ram, nullptr);
    if (!active) return false;
    const int s1 = (int)ram.rd(13), s2 = (int)ram.rd(14);          // score1 = $8D, score2 = $8E
    // ---- observation (find_stuff) ----
    bool valid[3]; double loc[3][2];
#pragma unroll
    for (int t = 0; t < 3; ++t) {
        valid[t] = s.cnt[t] > 0;
        loc[t][0] = valid[t] ? __ddiv_rn((double)s.sy[t], (double)s.cnt[t]) : 0.0;
        loc[t][1] = valid[t] ? __ddiv_rn((double)s.sx[t], (double)s.cnt[t]) : 0.0;
    }
    // ---- get_actions (main.py:138-154) ----
    // the reference draws two random actions every frame (main.py:139-140); with a counter-based generator the draw is a pure
    // function of (seed, env, frame, player), so it is only evaluated on the one path that uses it
    int left_act = pol::ACT_NONE, right_act = pol::ACT_NONE;
    if (valid[0]) {
        const double lb[2] = {ep.have_last_ball ? ep.last_ball[0] : loc[0][0], ep.have_last_ball ? ep.last_ball[1] : loc[0][1]};
        // deviation (SURVEY Appendix A5): the reference raises TypeError when one paddle is missing
        // while the ball is visible; the random action is kept instead
        if (valid[1] && valid[2]) {
            const double fball[2] = {loc[0][0], __dsub_rn(160.0, loc[0][1])}, flast[2] = {lb[0], __dsub_rn(160.0, lb[1])};
            left_act = run_policy(p.shape, ep.plan.left_kind, ep.plan.left_genome, fball, flast, loc[1][0], loc[2][0], s1, s2);
            right_act = run_policy(p.shape, pol::KIND_MLP, ep.plan.right_genome, loc[0], lb, loc[2][0], loc[1][0], s1, s2);
        } else {
            const uint32_t key = REC && rec->key ? (uint32_t)rec->key[ep.env] : (uint32_t)ep.env;
            left_act = pol::random_action_bit(p.seed, p.generation, key, (uint32_t)ep.frame, 0) ? pol::ACT_DOWN : pol::ACT_UP;
            right_act = pol::random_action_bit(p.seed, p.generation, key, (uint32_t)ep.frame, 1) ? pol::ACT_DOWN : pol::ACT_UP;
        }
    }
    ep.have_last_ball = valid[0];
    if (valid[0]) { ep.last_ball[0] = loc[0][0]; ep.last_ball[1] = loc[0][1]; }
    ep.left_act = pol::clamp_action(valid[1], loc[1][0], left_act, p.paddle_height);
    ep.right_act = pol::clamp_action(valid[2], loc[2][0], right_act, p.paddle_height);
    // ---- calculate_timeout_and_frames (main.py:128-135) ----
    if (ep.have_last_score) {
        if (ep.last_s1 == s1 && ep.last_s2 == s2) ep.timeout += 1;
        else { ep.total_frames += ep.timeout; ep.timeout = 0; }
    }
    ep.have_last_score = true; ep.last_s1 = s1; ep.last_s2 = s2;
    ep.frame++;
    const bool done = s1 >= p.win_score || s2 >= p.win_score || ep.timeout > p.timeout_thresh ||
                      (p.max_frames > 0 && ep.frame >= p.max_frames) || s.error;
    if (done) {
        double rw = 0.0;
        if (s1 != s2) {                                   // utils.calculate_reward, utils.py:104-109
            const double diff = (double)(s2 - s1);
            const double scaled = __ddiv_rn((double)ep.total_frames, p.time_scaler);
            const double bonus = __dmul_rn((double)s2, ep.plan.mult);
            rw = __ddiv_rn(__dadd_rn(diff, bonus), scaled);
        }
        *reward = rw;
    }
    return done;
}

#endif  // __CUDACC__
}  // namespace roll
