// ngp_stepwise.cu -- ngp_evaluate for networks too wide for the fused rollout (any layer wider than
// pol::FUSED_MAX_WIDTH; BASELINE config 4: [6,512,512,2] with 64 environments per genome).
//
// The reference evaluates whatever NETWORK_SHAPE says (config.py:30-32, utils.create_model_from_genes
// utils.py:80-87, main.py:29); a 512-wide net does not fit a thread's registers, so here one frame of every
// live environment is one pass over three kinds of kernels instead of one fused launch:
//
//   step_frame_kernel   env.step (main.py:77) + find_stuff (main.py:82) + utils.inference's six-vector for both players
//                       (utils.py:139-153), written as rows of the batched MLP input
//   ngp_mlp_forward     NeuralNetwork.run for every (genome, environment) pair at once: with the round-robin schedule a genome
//                       is the right player of `games` environments and the left player of `games` others, so each genome's
//                       weights are streamed once per frame for 2*games rows (the wide hidden layers run on tcgen05)
//   step_decide_kernel  get_actions' fall-backs, bots, bounds clamp, calculate_timeout_and_frames, termination, reward
//                       (main.py:84-107, 128-154; utils.py:71-77, 104-109)
//
// Per-environment state (console snapshot + perform_episode's locals, stepwise.cuh) lives in HBM between the kernels.  The host
// loop launches frames without synchronising and reads the count of finished environments back every CHECK_EVERY frames.
// ngp_play_matches_stepwise (ngp_stepwise_lists.cu) runs match lists through the same frame kernel (ngp_step_frame).
#include "ngp_internal.h"
#include "rollout.cuh"
#include "stepwise.cuh"

using a26::Chip; using a26::CpuRegs; using a26::Ram; using a26::Snapshot; using a26::Tables;
using roll::RolloutParams;

namespace {

// rows of the MLP batch: round-robin -> x[n][2*games][6]: genome g's row k = its game k as the right player, row games+k = the
// game it plays on the left (environment ((g-k-1) mod n, k)); reference schedule -> right rows x[n][games][6], hall-of-fame
// opponents one row each in a second batch x_hof[3n][1][6] over the gathered opponent genomes.
__global__ void step_begin_kernel(RolloutParams p, StepEnv *envs, int total)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total) return;
    StepEnv &v = envs[e];
    const roll::EnvPlan pl = roll::plan_env(p, e);
    v.snap = p.start[pl.state];
    v.done = 0; v.frame = 0; v.timeout = 0; v.total_frames = 0; v.last_s1 = v.last_s2 = 0;
    v.have_last_score = 0; v.have_last_ball = 0; v.left_act = v.right_act = pol::ACT_NONE;
    v.last_ball[0] = v.last_ball[1] = 0.0;
    v.state = pl.state; v.left_kind = pl.left_kind; v.mult = pl.mult;
    const int g = e / p.games, k = e % p.games;
    if (p.schedule == NGP_SCHEDULE_ROUND_ROBIN) {
        v.right_row = g * 2 * p.games + k;
        v.left_row = ((g + k + 1) % p.n) * 2 * p.games + p.games + k;
    } else {
        v.right_row = e;
        v.left_row = pl.left_kind == pol::KIND_MLP ? g * 3 + (k - 3) % 3 : -1;
    }
}

// dense copy of every hall-of-fame opponent the plan picked: opp[g*3 + j] = hof_genomes[pick(g, game 3+j)]
__global__ void step_gather_opponents_kernel(RolloutParams p, float *__restrict__ opp)
{
    const int row = blockIdx.x;                  // g*3 + j
    const roll::EnvPlan pl = roll::plan_env(p, (row / 3) * p.games + 3 + row % 3);
    const float *src = pl.left_genome;
    float *dst = opp + (size_t)row * p.G;
    for (int i = threadIdx.x; i < p.G; i += blockDim.x) dst[i] = src ? src[i] : 0.f;
}

template <int CORE>
__global__ void __launch_bounds__(32) step_frame_kernel(RolloutParams p, StepEnv *envs, int total, float *__restrict__ x, float *__restrict__ x_hof)
{
    __shared__ Tables T;
    __shared__ uint32_t ram_smem[32 * 32];
    load_tables_cta(T, p.tables);
    const int e = blockIdx.x * 32 + threadIdx.x;
    if (e >= total) return;
    StepEnv &v = envs[e];
    if (v.done) return;
    // the body of step_env_frame (stepwise.cuh), kept inline here: through the helper the compiler inlines the frame differently
    // (168 registers instead of 128 for the translated core), and this kernel stays as the wide ngp_evaluate has measured it
    Ram ram{&ram_smem[threadIdx.x]};
    Chip s; CpuRegs r;
    roll::load_snapshot(&v.snap, s, r, ram);
    const uint32_t in = p.input_table[v.state == NGP_STATE_START_1P ? 0 : 1][v.left_act * 3 + v.right_act];
    a26::apply_input(s, p.needed, in & 0xFF, (in >> 8) & 15, (in >> 12) & 15, (in >> 16) & 15);
    a26::clear_obs(s);
    if (CORE) a26::run_frame_compiled<false, false>(s, r, T, ram, nullptr);
    else a26::run_frame<false>(s, r, T, ram, nullptr);
    roll::store_snapshot(&v.snap, s, r, ram);
    v.s1 = (uint8_t)ram.rd(13); v.s2 = (uint8_t)ram.rd(14); v.emu_error = s.error;
    double loc[3][2];
#pragma unroll
    for (int t = 0; t < 3; ++t) {
        const bool ok = s.cnt[t] > 0;
        v.valid[t] = ok;
        loc[t][0] = ok ? __ddiv_rn((double)s.sy[t], (double)s.cnt[t]) : 0.0;
        loc[t][1] = ok ? __ddiv_rn((double)s.sx[t], (double)s.cnt[t]) : 0.0;
        v.loc[t][0] = loc[t][0]; v.loc[t][1] = loc[t][1];
    }
    if (v.valid[0] && v.valid[1] && v.valid[2]) {                       // the frames on which main.get_actions calls the models
        const double lb[2] = {v.have_last_ball ? v.last_ball[0] : loc[0][0], v.have_last_ball ? v.last_ball[1] : loc[0][1]};
        write_inference_row(x + (size_t)v.right_row * 6, loc[0], lb, loc[2][0], loc[1][0]);
        if (v.left_kind == pol::KIND_MLP) {
            const double fball[2] = {loc[0][0], __dsub_rn(160.0, loc[0][1])}, flast[2] = {lb[0], __dsub_rn(160.0, lb[1])};
            float *row = (p.schedule == NGP_SCHEDULE_ROUND_ROBIN ? x : x_hof) + (size_t)v.left_row * 6;
            write_inference_row(row, fball, flast, loc[1][0], loc[2][0]);
        }
    }
}

__global__ void step_decide_kernel(RolloutParams p, StepEnv *envs, int total, const uint8_t *__restrict__ act, const uint8_t *__restrict__ act_hof)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    bool stepped = false, finished = false;
    if (e < total && !envs[e].done) {
        StepEnv &v = envs[e];
        stepped = true;
        const int s1 = v.s1, s2 = v.s2;
        const bool vb = v.valid[0], vl = v.valid[1], vr = v.valid[2];
        // ---- get_actions (main.py:138-154) ----
        int left_act = pol::ACT_NONE, right_act = pol::ACT_NONE;
        if (vb) {
            if (vl && vr) {
                right_act = act[v.right_row];
                if (v.left_kind == pol::KIND_MLP) left_act = (p.schedule == NGP_SCHEDULE_ROUND_ROBIN ? act : act_hof)[v.left_row];
                else {
                    const double lb[2] = {v.have_last_ball ? v.last_ball[0] : v.loc[0][0], v.have_last_ball ? v.last_ball[1] : v.loc[0][1]};
                    const double fball[2] = {v.loc[0][0], __dsub_rn(160.0, v.loc[0][1])}, flast[2] = {lb[0], __dsub_rn(160.0, lb[1])};
                    left_act = roll::run_policy(p.shape, v.left_kind, nullptr, fball, flast, v.loc[1][0], v.loc[2][0], s1, s2);
                }
            } else {            // same deviation as the fused path: the reference raises TypeError here; the random action is kept
                left_act = pol::random_action_bit(p.seed, p.generation, (uint32_t)e, (uint32_t)v.frame, 0) ? pol::ACT_DOWN : pol::ACT_UP;
                right_act = pol::random_action_bit(p.seed, p.generation, (uint32_t)e, (uint32_t)v.frame, 1) ? pol::ACT_DOWN : pol::ACT_UP;
            }
        }
        v.have_last_ball = vb;
        if (vb) { v.last_ball[0] = v.loc[0][0]; v.last_ball[1] = v.loc[0][1]; }
        v.left_act = (uint8_t)pol::clamp_action(vl, v.loc[1][0], left_act, p.paddle_height);
        v.right_act = (uint8_t)pol::clamp_action(vr, v.loc[2][0], right_act, p.paddle_height);
        // ---- calculate_timeout_and_frames (main.py:128-135) ----
        if (v.have_last_score) {
            if (v.last_s1 == s1 && v.last_s2 == s2) v.timeout += 1;
            else { v.total_frames += v.timeout; v.timeout = 0; }
        }
        v.have_last_score = 1; v.last_s1 = s1; v.last_s2 = s2;
        v.frame++;
        finished = s1 >= p.win_score || s2 >= p.win_score || v.timeout > p.timeout_thresh || (p.max_frames > 0 && v.frame >= p.max_frames) ||
                   v.emu_error;
        if (finished) {
            double rw = 0.0;
            if (s1 != s2) {                                   // utils.calculate_reward, utils.py:104-109
                const double diff = (double)(s2 - s1);
                const double scaled = __ddiv_rn((double)v.total_frames, p.time_scaler);
                rw = __ddiv_rn(__dadd_rn(diff, __dmul_rn((double)s2, v.mult)), scaled);
            }
            p.rewards[e] = rw; p.frames[e] = v.frame;
            v.done = 1;
            if (v.emu_error) atomicAdd(&p.counters[2], 1ull);
        }
    }
    const unsigned m_step = __ballot_sync(0xFFFFFFFFu, stepped), m_fin = __ballot_sync(0xFFFFFFFFu, finished);
    if ((threadIdx.x & 31) == 0) {
        if (m_step) atomicAdd(&p.counters[1], (unsigned long long)__popc(m_step));
        if (m_fin) atomicAdd(&p.counters[3], (unsigned long long)__popc(m_fin));
    }
}

}  // namespace

// one frame of every running environment (step_frame_kernel): the frame kernel of ngp_play_matches_stepwise's loop
int ngp_step_frame(ngp_handle *h, const RolloutParams &p, void *envs, int total, float *x, float *x_hof, cudaStream_t st)
{
    StepEnv *e = static_cast<StepEnv *>(envs);
    if (p.core) step_frame_kernel<1><<<(total + 31) / 32, 32, 0, st>>>(p, e, total, x, x_hof);
    else step_frame_kernel<0><<<(total + 31) / 32, 32, 0, st>>>(p, e, total, x, x_hof);
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    return NGP_OK;
}

// called by ngp_evaluate (ngp_core.cu) with the rollout parameters filled in; synchronises the stream
int ngp_evaluate_stepwise(ngp_handle *h, const RolloutParams &p, cudaStream_t st)
{
    const int total = p.n * p.games;
    const bool rr = p.schedule == NGP_SCHEDULE_ROUND_ROBIN;
    const bool hof = !rr && p.n_hof > 0 && p.games > 3;
    const long long rows = rr ? 2ll * total : total, rows_hof = hof ? 3ll * p.n : 0;
    const size_t n_x = (size_t)(rows + rows_hof) * 6, n_act = (size_t)(rows + rows_hof), n_opp = (size_t)rows_hof * p.G;
    if (n_opp * sizeof(float) > (size_t)32 << 30) {
        ngp_set_error("ngp_evaluate: %lld hall-of-fame opponents of %d genes need more than 32 GiB of gathered weights", rows_hof, p.G);
        return NGP_ERR_UNSUPPORTED;
    }
    NGP_CUDA(h->step_envs.ensure((size_t)total * sizeof(StepEnv)));
    NGP_CUDA(h->step_x.ensure(n_x));
    NGP_CUDA(h->step_act.ensure(n_act));
    if (hof) NGP_CUDA(h->step_opp.ensure(n_opp));
    StepEnv *envs = reinterpret_cast<StepEnv *>(h->step_envs.p);
    float *x = h->step_x.p, *x_hof = x + rows * 6;
    uint8_t *act = h->step_act.p, *act_hof = act + rows;
    NGP_CUDA(cudaMemsetAsync(x, 0, n_x * sizeof(float), st));    // rows of frames without a model call are never read, but keep them finite
    NGP_CUDA(cudaMemsetAsync(act, 0, n_act, st));
    step_begin_kernel<<<(total + 127) / 128, 128, 0, st>>>(p, envs, total);
    h->launches++;
    if (hof) {
        step_gather_opponents_kernel<<<(unsigned)rows_hof, 256, 0, st>>>(p, h->step_opp.p);
        h->launches++;
    }
    NGP_CUDA(cudaGetLastError());
    const int per_genome = rr ? 2 * p.games : p.games;
    {   // the population's networks are built once per evaluation (main.py:29) and run every frame
        const int rc = ngp_mlp_prepare(h, p.genomes, p.n, st);
        if (rc != NGP_OK) return rc;
    }
    for (long long frame = 1;; ++frame) {
        if (p.core) step_frame_kernel<1><<<(total + 31) / 32, 32, 0, st>>>(p, envs, total, x, x_hof);
        else step_frame_kernel<0><<<(total + 31) / 32, 32, 0, st>>>(p, envs, total, x, x_hof);
        h->launches++;
        NGP_CUDA(cudaGetLastError());
        int rc = ngp_mlp_forward_prepared(h, p.genomes, x, p.n, per_genome, act, nullptr, st);
        if (rc != NGP_OK) return rc;
        if (hof) {
            rc = ngp_mlp_forward(h, h->step_opp.p, x_hof, (int32_t)rows_hof, 1, act_hof, nullptr, st);
            if (rc != NGP_OK) return rc;
        }
        step_decide_kernel<<<(total + 127) / 128, 128, 0, st>>>(p, envs, total, act, act_hof);
        h->launches++;
        NGP_CUDA(cudaGetLastError());
        if (frame % CHECK_EVERY == 0) {
            NGP_CUDA(cudaMemcpyAsync(h->h_counters.p, h->d_counters.p, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
            NGP_CUDA(cudaStreamSynchronize(st));
            if (h->h_counters.p[3] >= (unsigned long long)total) break;
        }
    }
    return NGP_OK;
}
