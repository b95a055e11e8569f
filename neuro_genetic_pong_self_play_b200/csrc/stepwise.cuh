// stepwise.cuh -- the per-environment state of the per-frame driver (ngp_stepwise.cu: wide ngp_evaluate;
// ngp_stepwise_lists.cu: ngp_play_matches_stepwise; ngp_session.cu: match sessions), kept in HBM between its kernels, and the
// pieces of the frame kernel the drivers share.
#pragma once
#include "ngp_internal.h"
#include "rollout.cuh"

namespace {

constexpr int CHECK_EVERY = 8;       // frames between two reads of the finished-environment count

// StepEnv::ext: the seats of a match session whose decisions the caller supplies (NGP_PLAYER_EXTERNAL)
constexpr uint8_t EXT_LEFT = 1, EXT_RIGHT = 2;

struct StepEnv {
    a26::Snapshot snap;
    // perform_episode's locals (main.py:70-75)
    int32_t done, frame, timeout, total_frames, last_s1, last_s2;
    uint8_t have_last_score, have_last_ball, left_act, right_act;
    double last_ball[2];
    // what the frame kernel saw (consumed by the decide kernel)
    double loc[3][2];
    uint8_t valid[3], s1, s2, emu_error, ext, pad_;     // ext: EXT_* bits (0 outside a match session)
    // plan (main.py:33-58 / round-robin)
    int32_t state, left_kind, left_row, right_row;      // rows of the batched MLP input / action arrays (-1: no MLP on the left)
    double mult;
};

__device__ __forceinline__ void load_tables_cta(a26::Tables &dst, const a26::Tables *__restrict__ src)
{
    const uint32_t *s = reinterpret_cast<const uint32_t *>(src);
    uint32_t *d = reinterpret_cast<uint32_t *>(&dst);
    for (unsigned i = threadIdx.x; i < sizeof(a26::Tables) / 4; i += blockDim.x) d[i] = s[i];
    __syncthreads();
}

__device__ __forceinline__ void write_inference_row(float *__restrict__ x, const double ball[2], const double last[2], double me_row, double enemy_row)
{
    // utils.inference (utils.py:139-153): ball x, ball y, last x, last y, my row, enemy row, all divided by 160
    x[0] = (float)__ddiv_rn(ball[1], 160.0); x[1] = (float)__ddiv_rn(ball[0], 160.0);
    x[2] = (float)__ddiv_rn(last[1], 160.0); x[3] = (float)__ddiv_rn(last[0], 160.0);
    x[4] = (float)__ddiv_rn(me_row, 160.0);  x[5] = (float)__ddiv_rn(enemy_row, 160.0);
}

// env.step (main.py:77) and find_stuff (main.py:82) of the running environment v by one lane (ram_lane: its column of the CTA's
// interleaved RAM): the console plays one frame on v's decisions; v gets the scores, the emulator error, the found objects and
// their centroids, which also go to loc.  Returns true on the frames on which main.get_actions calls the models (ball and both
// paddles found); lb is then the last ball of utils.inference.
template <int CORE>
__device__ __forceinline__ bool step_env_frame(const roll::RolloutParams &p, StepEnv &v, const a26::Tables &T, uint32_t *ram_lane,
                                               double loc[3][2], double lb[2])
{
    a26::Ram ram{ram_lane};
    a26::Chip s; a26::CpuRegs r;
    roll::load_snapshot(&v.snap, s, r, ram);
    const uint32_t in = p.input_table[v.state == NGP_STATE_START_1P ? 0 : 1][v.left_act * 3 + v.right_act];
    a26::apply_input(s, p.needed, in & 0xFF, (in >> 8) & 15, (in >> 12) & 15, (in >> 16) & 15);
    a26::clear_obs(s);
    if (CORE) a26::run_frame_compiled<false, false>(s, r, T, ram, nullptr);
    else a26::run_frame<false>(s, r, T, ram, nullptr);
    roll::store_snapshot(&v.snap, s, r, ram);
    v.s1 = (uint8_t)ram.rd(13); v.s2 = (uint8_t)ram.rd(14); v.emu_error = s.error;
#pragma unroll
    for (int t = 0; t < 3; ++t) {
        const bool ok = s.cnt[t] > 0;
        v.valid[t] = ok;
        loc[t][0] = ok ? __ddiv_rn((double)s.sy[t], (double)s.cnt[t]) : 0.0;
        loc[t][1] = ok ? __ddiv_rn((double)s.sx[t], (double)s.cnt[t]) : 0.0;
        v.loc[t][0] = loc[t][0]; v.loc[t][1] = loc[t][1];
    }
    if (!(v.valid[0] && v.valid[1] && v.valid[2])) return false;
    lb[0] = v.have_last_ball ? v.last_ball[0] : loc[0][0];
    lb[1] = v.have_last_ball ? v.last_ball[1] : loc[0][1];
    return true;
}

}  // namespace

// A match session's step (ngp_session.cu) as list_decide_kernel sees it; zero for ngp_play_matches_stepwise.
struct SessionStep {
    const uint8_t *actions;         // [n][2] (left, right) NGP_ACT_* of the external seats, or null
    int capture_all;                // capture every match still running after the decisions to rec.capture
};

// ngp_stepwise.cu: one frame of every running environment of `envs` (StepEnv[total]; step_frame_kernel, p.core picks the core); the
// inference rows of model-call frames go to x[right_row], and x_hof[left_row] (reference schedule) or x[left_row]
int ngp_step_frame(ngp_handle *h, const roll::RolloutParams &p, void *envs, int total, float *x, float *x_hof, cudaStream_t st);

// ngp_stepwise_lists.cu: the per-frame driver of a match list, in the pieces ngp_play_matches_stepwise and a match session share.
// ngp_list_begin: after the list check (p.n matches, p.games = 1), every environment planned and started (list_begin_kernel)
// in `envs`; wide networks also get the chunk layout of their MLP rows (chunk, x and act sized for *C chunks of *T rows, from
// the counts ngp_list_layout_count left in h_counters[8 .. 14)).  ext: null, or the EXT_* bits of every match (external seats
// get no MLP row; p's lists then hold a genome row or NGP_OPP_* code for every seat, never NGP_PLAYER_EXTERNAL).
int ngp_list_begin(ngp_handle *h, const roll::RolloutParams &p, const roll::RecordArgs &rec, int n_genomes, bool wide, const uint8_t *ext,
                   Buffer<uint8_t> &envs, Buffer<float> &x, Buffer<uint8_t> &act, Buffer<int32_t> &chunk, int *T, long long *C,
                   cudaStream_t st);
// ngp_list_decide: the decisions of the frame every running environment has just played (list_decide_kernel); act = the wide
// MLP's actions, or null for the FP64 policies of the fused rollout
int ngp_list_decide(ngp_handle *h, const roll::RolloutParams &p, const roll::RecordArgs &rec, void *envs, int total, const uint8_t *act,
                    const SessionStep &ss, cudaStream_t st);
