// ngp_stepwise_lists.cu -- ngp_play_matches_stepwise: a match list (ngp_play_matches_states' arguments) on the per-frame driver of
// wide ngp_evaluate (ngp_stepwise.cu), for networks of any width.  Match sessions (ngp_session.cu) play lists on the same pieces.  Environment m is match m, planned from the lists by
// roll::plan_env, started from a save state when asked (list_begin_kernel), stepped by ngp_evaluate's frame kernel
// (ngp_step_frame), decided, recorded and captured by list_decide_kernel.  Wide networks' MLP rows are grouped by genome into
// chunks of T rows (the layout kernels below) and run by ngp_mlp_forward_chunks.  A translation unit of its own, so that wide
// ngp_evaluate's kernels compile exactly as before.
#include <algorithm>

#include <cub/cub.cuh>

#include "game_state.cuh"
#include "stepwise.cuh"

using roll::RecordArgs; using roll::RolloutParams;

namespace {

// perform_episode's locals of an environment as a roll::Episode (the save-state packer's view) and back
__device__ __forceinline__ roll::Episode episode_of(const StepEnv &v)
{
    roll::Episode ep;
    ep.frame = v.frame; ep.timeout = v.timeout; ep.total_frames = v.total_frames; ep.last_s1 = v.last_s1; ep.last_s2 = v.last_s2;
    ep.have_last_score = v.have_last_score; ep.have_last_ball = v.have_last_ball;
    ep.last_ball[0] = v.last_ball[0]; ep.last_ball[1] = v.last_ball[1];
    ep.left_act = v.left_act; ep.right_act = v.right_act;
    return ep;
}

// the state of match e (console and episode) to rec.capture[e], as roll::capture_state writes it in the fused rollout
static __device__ __noinline__ void capture_env(const RecordArgs &rec, StepEnv &v, int e)
{
    uint32_t w[12];
    gs::episode_words(episode_of(v), w);
    gs::pack(rec.capture + e, rec.cart, v.state == NGP_STATE_START_1P ? 1 : 2, v.snap.chip, v.snap.cpu, gs::SnapRam{v.snap.ram}, w);
}

// Match list (ngp_play_matches_stepwise): match e = environment e.  The plan comes from the lists; with rec.start the match
// starts from a save state (resuming its episode unless rec.fresh), and rec.capture_at[e] == the start frame captures at once,
// as rollout_kernel does after episode_begin.  With `base`, each MLP side takes the next free row of its genome's chunks
// (genome g's rows are base[g] * T ..; cursor[g] counts the rows handed out): the ranks depend on the atomics' order, the
// results do not, since every row is computed on its own.  Without, no MLP batch runs: match e writes its rows 2e, 2e + 1
// (which nothing reads), so that wide ngp_evaluate's frame kernel serves both drivers unchanged.  ext (a match session): the
// EXT_* bits of match e; an external seat takes no MLP row.
__global__ void list_begin_kernel(RolloutParams p, RecordArgs rec, StepEnv *envs, int total, const int32_t *__restrict__ base,
                                  int32_t *__restrict__ cursor, int T, const uint8_t *__restrict__ ext)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total) return;
    StepEnv &v = envs[e];
    const roll::EnvPlan pl = roll::plan_env(p, e);
    roll::Episode ep;
    ep.frame = 0; ep.timeout = 0; ep.total_frames = 0; ep.last_s1 = ep.last_s2 = 0;
    ep.have_last_score = false; ep.have_last_ball = false;
    ep.last_ball[0] = ep.last_ball[1] = 0.0;
    ep.left_act = ep.right_act = pol::ACT_NONE;
    v.snap = p.start[pl.state];
    if (rec.start && rec.start[e] >= 0)
        gs::unpack(rec.states + rec.start[e], v.snap.chip, v.snap.cpu, gs::SnapRam{v.snap.ram}, rec.fresh ? nullptr : &ep);
    v.done = 0; v.frame = ep.frame; v.timeout = ep.timeout; v.total_frames = ep.total_frames; v.last_s1 = ep.last_s1; v.last_s2 = ep.last_s2;
    v.have_last_score = ep.have_last_score; v.have_last_ball = ep.have_last_ball;
    v.left_act = (uint8_t)ep.left_act; v.right_act = (uint8_t)ep.right_act;
    v.last_ball[0] = ep.last_ball[0]; v.last_ball[1] = ep.last_ball[1];
    v.state = pl.state; v.left_kind = pl.left_kind; v.mult = pl.mult;
    v.ext = ext ? ext[e] : 0;
    if (base) {
        const int r = p.match_right[e], l = p.match_left[e];
        v.right_row = v.ext & EXT_RIGHT ? -1 : base[r] * T + atomicAdd(&cursor[r], 1);
        v.left_row = l >= 0 && !(v.ext & EXT_LEFT) ? base[l] * T + atomicAdd(&cursor[l], 1) : -1;
    } else {
        v.right_row = 2 * e; v.left_row = 2 * e + 1;
    }
    if (rec.capture_at && rec.capture_at[e] == v.frame) capture_env(rec, v, e);
}

// step_decide_kernel (ngp_stepwise.cu) for a match list: the fall-back key is rec.key[e] (or e), rec.record gets entry
// frame - 1 after the clamp and the timeout update (the fields of roll::record_frame), a running episode is captured when its
// frame reaches rec.capture_at[e], and p.scores gets the last scores.  Left MLP rows are in `act` too.  act == NULL: networks the
// fused rollout takes, run here in FP64 by roll::run_policy as the fused rollout runs them.
// A match session's step (ss.actions set): an external seat (v.ext) plays ss.actions[e][0] (left) or [1] (right) on the frames on
// which a model is called, a value outside 0..2 as NGP_ACT_NONE, counted in p.counters[4]; p.scores gets every frame's scores;
// with ss.capture_all every match still running is captured.
__global__ void list_decide_kernel(RolloutParams p, RecordArgs rec, StepEnv *envs, int total, const uint8_t *__restrict__ act, SessionStep ss)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    bool stepped = false, finished = false;
    int bad = 0;
    if (e < total && !envs[e].done) {
        StepEnv &v = envs[e];
        stepped = true;
        const int s1 = v.s1, s2 = v.s2;
        const bool vb = v.valid[0], vl = v.valid[1], vr = v.valid[2];
        // ---- get_actions (main.py:138-154) ----
        int left_act = pol::ACT_NONE, right_act = pol::ACT_NONE;
        if (vb) {
            if (vl && vr) {
                const double lb[2] = {v.have_last_ball ? v.last_ball[0] : v.loc[0][0], v.have_last_ball ? v.last_ball[1] : v.loc[0][1]};
                const double fball[2] = {v.loc[0][0], __dsub_rn(160.0, v.loc[0][1])}, flast[2] = {lb[0], __dsub_rn(160.0, lb[1])};
                const float *lg = nullptr, *rg = nullptr;
                if (!act) { const roll::EnvPlan pl = roll::plan_env(p, e); lg = pl.left_genome; rg = pl.right_genome; }
                if (v.ext & EXT_LEFT) {
                    left_act = ss.actions[2 * e];
                    if (left_act > pol::ACT_DOWN) { left_act = pol::ACT_NONE; ++bad; }
                } else if (act && v.left_kind == pol::KIND_MLP) left_act = act[v.left_row];
                else left_act = roll::run_policy(p.shape, v.left_kind, lg, fball, flast, v.loc[1][0], v.loc[2][0], s1, s2);
                if (v.ext & EXT_RIGHT) {
                    right_act = ss.actions[2 * e + 1];
                    if (right_act > pol::ACT_DOWN) { right_act = pol::ACT_NONE; ++bad; }
                } else if (act) right_act = act[v.right_row];
                else right_act = roll::run_policy(p.shape, pol::KIND_MLP, rg, v.loc[0], lb, v.loc[2][0], v.loc[1][0], s1, s2);
            } else {            // same deviation as the fused path: the reference raises TypeError here; the random action is kept
                const uint32_t key = rec.key ? (uint32_t)rec.key[e] : (uint32_t)e;
                left_act = pol::random_action_bit(p.seed, p.generation, key, (uint32_t)v.frame, 0) ? pol::ACT_DOWN : pol::ACT_UP;
                right_act = pol::random_action_bit(p.seed, p.generation, key, (uint32_t)v.frame, 1) ? pol::ACT_DOWN : pol::ACT_UP;
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
        if (rec.record && v.frame <= rec.max_record) {
            uint32_t w[6], vbits = 0;
#pragma unroll
            for (int t = 0; t < 3; ++t) {
                vbits |= (uint32_t)(v.valid[t] != 0) << t;
                w[2 * t] = roll::f32_bits(v.loc[t][0]); w[2 * t + 1] = roll::f32_bits(v.loc[t][1]);
            }
            roll::record_store(rec, e, v.frame - 1, 0, w[0], w[1], w[2], w[3]);
            roll::record_store(rec, e, v.frame - 1, 1, w[4], w[5],
                               vbits | (uint32_t)s1 << 8 | (uint32_t)s2 << 16 | (uint32_t)(v.left_act | v.right_act << 2) << 24, (uint32_t)v.timeout);
        }
        if (p.scores && (finished || ss.actions)) { p.scores[2 * e] = s1; p.scores[2 * e + 1] = s2; }
        if (!finished && (ss.capture_all || (rec.capture_at && v.frame == rec.capture_at[e]))) capture_env(rec, v, e);
    }
    const unsigned m_step = __ballot_sync(0xFFFFFFFFu, stepped), m_fin = __ballot_sync(0xFFFFFFFFu, finished);
    if ((threadIdx.x & 31) == 0) {
        if (m_step) atomicAdd(&p.counters[1], (unsigned long long)__popc(m_step));
        if (m_fin) atomicAdd(&p.counters[3], (unsigned long long)__popc(m_fin));
    }
    if (ss.actions) {
        bad = __reduce_add_sync(0xFFFFFFFFu, bad);
        if ((threadIdx.x & 31) == 0 && bad) atomicAdd(&p.counters[4], (unsigned long long)bad);
    }
}

// ---- the chunk layout of a match list's MLP rows ----
// Every MLP side of every match is one row per frame.  Rows are grouped by genome into chunks of T rows (one genome per
// chunk, the last chunk of a genome padded), so the batch is x[C][T][6] with the weights of genome chunk_genome[c] for chunk c.

// count[g] = the rows of genome g (entries that name no row are left to the list check)
__global__ void list_count_kernel(const int32_t *__restrict__ right, const int32_t *__restrict__ left, int n, int n_genomes, int32_t *__restrict__ count)
{
    for (int m = blockIdx.x * blockDim.x + threadIdx.x; m < n; m += gridDim.x * blockDim.x) {
        const int r = right[m], l = left[m];
        if (r >= 0 && r < n_genomes) atomicAdd(&count[r], 1);
        if (l >= 0 && l < n_genomes) atomicAdd(&count[l], 1);
    }
}

// the chunk sizes list_stats_kernel counts for: 1 (= rows), 16, 32, 64, 128
__host__ __device__ constexpr int layout_t(int i) { return i ? 8 << i : 1; }
// stats[0] = genomes with rows; stats[1 + i] = chunks of layout_t(i) rows (stats[1] = the rows)
__global__ void list_stats_kernel(const int32_t *__restrict__ count, int n_genomes, unsigned long long *__restrict__ stats)
{
    unsigned long long v[6] = {0, 0, 0, 0, 0, 0};
    for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < n_genomes; g += gridDim.x * blockDim.x) {
        const int c = count[g];
        v[0] += c > 0;
#pragma unroll
        for (int i = 0; i < 5; ++i) v[1 + i] += (unsigned)(c + layout_t(i) - 1) / layout_t(i);
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        for (int off = 16; off; off >>= 1) v[i] += __shfl_down_sync(0xFFFFFFFFu, v[i], off);
        if ((threadIdx.x & 31) == 0 && v[i]) atomicAdd(&stats[i], v[i]);
    }
}

__global__ void list_chunks_kernel(const int32_t *__restrict__ count, int n_genomes, int T, int32_t *__restrict__ nchunk)
{
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g < n_genomes) nchunk[g] = (count[g] + T - 1) / T;
}

// chunk_genome[base[g] ..] = g for genome g's chunks; count[g] = 0, so that list_begin_kernel can hand out ranks from it
__global__ void list_fill_kernel(int32_t *__restrict__ count, const int32_t *__restrict__ nchunk, const int32_t *__restrict__ base, int n_genomes,
                                 int32_t *__restrict__ chunk_genome)
{
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_genomes) return;
    for (int j = 0; j < nchunk[g]; ++j) chunk_genome[base[g] + j] = g;
    count[g] = 0;
}

}  // namespace

// ngp_play_matches_stepwise, wide networks: counts the rows per genome and the chunk counts of every T (list_stats_kernel) into
// d_counters[8 .. 14), which play_match_list (ngp_core.cu) reads back with the list check
int ngp_list_layout_count(ngp_handle *h, const int32_t *right, const int32_t *left, int n_matches, int n_genomes, cudaStream_t st)
{
    NGP_CUDA(h->list_genome.ensure(3 * (size_t)n_genomes));
    NGP_CUDA(cudaMemsetAsync(h->list_genome.p, 0, (size_t)n_genomes * sizeof(int32_t), st));
    NGP_CUDA(cudaMemsetAsync(h->d_counters.p + 8, 0, 6 * sizeof(unsigned long long), st));
    const int mb = (int)std::min<long long>((n_matches + 255) / 256, 4ll * h->sm_count), gb = (int)std::min<long long>((n_genomes + 255) / 256, 4ll * h->sm_count);
    list_count_kernel<<<mb, 256, 0, st>>>(right, left, n_matches, n_genomes, h->list_genome.p);
    list_stats_kernel<<<gb, 256, 0, st>>>(h->list_genome.p, n_genomes, h->d_counters.p + 8);
    h->launches += 2;
    NGP_CUDA(cudaGetLastError());
    return NGP_OK;
}

int ngp_list_begin(ngp_handle *h, const RolloutParams &p, const RecordArgs &rec, int n_genomes, bool wide, const uint8_t *ext,
                   Buffer<uint8_t> &envs_buf, Buffer<float> &x_buf, Buffer<uint8_t> &act_buf, Buffer<int32_t> &chunk, int *T_out,
                   long long *C_out, cudaStream_t st)
{
    const int total = p.n;
    NGP_CUDA(envs_buf.ensure((size_t)total * sizeof(StepEnv)));
    StepEnv *envs = reinterpret_cast<StepEnv *>(envs_buf.p);
    int T = 0;
    long long C = 0;
    if (wide && n_genomes > 0) {
        // T: the smallest power of two in [16, 128] not below the mean rows per genome with rows (a heuristic, not measured)
        const unsigned long long *stats = h->h_counters.p + 8, rows = stats[1], used = stats[0];
        int ti = 1;
        while (ti < 4 && (unsigned long long)layout_t(ti) * used < rows) ++ti;
        T = layout_t(ti);
        C = (long long)stats[1 + ti];
        if (C > INT32_MAX) {
            ngp_set_error("ngp_play_matches_stepwise: %lld chunks of %d rows are too many", C, T);
            return NGP_ERR_UNSUPPORTED;
        }
    }
    *T_out = T; *C_out = C;
    if (C > 0) {
        int32_t *count = h->list_genome.p, *nchunk = count + n_genomes, *base = nchunk + n_genomes;
        NGP_CUDA(chunk.ensure((size_t)C));
        NGP_CUDA(x_buf.ensure((size_t)C * T * 6));
        NGP_CUDA(act_buf.ensure((size_t)C * T));
        NGP_CUDA(cudaMemsetAsync(x_buf.p, 0, (size_t)C * T * 6 * sizeof(float), st));     // padding rows are computed, never read: keep them finite
        NGP_CUDA(cudaMemsetAsync(act_buf.p, 0, (size_t)C * T, st));
        const int gb = (n_genomes + 255) / 256;
        list_chunks_kernel<<<gb, 256, 0, st>>>(count, n_genomes, T, nchunk);
        h->launches++;
        NGP_CUDA(cudaGetLastError());
        size_t tmp_bytes = 0;
        NGP_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, nchunk, base, n_genomes, st));
        NGP_CUDA(h->list_scan_tmp.ensure(tmp_bytes));
        NGP_CUDA(cub::DeviceScan::ExclusiveSum(h->list_scan_tmp.p, tmp_bytes, nchunk, base, n_genomes, st));
        h->launches++;
        list_fill_kernel<<<gb, 256, 0, st>>>(count, nchunk, base, n_genomes, chunk.p);
        h->launches++;
        NGP_CUDA(cudaGetLastError());
        list_begin_kernel<<<(total + 127) / 128, 128, 0, st>>>(p, rec, envs, total, base, count, T, ext);
    } else {
        list_begin_kernel<<<(total + 127) / 128, 128, 0, st>>>(p, rec, envs, total, nullptr, nullptr, 0, ext);
    }
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    return NGP_OK;
}

int ngp_list_decide(ngp_handle *h, const RolloutParams &p, const RecordArgs &rec, void *envs, int total, const uint8_t *act,
                    const SessionStep &ss, cudaStream_t st)
{
    list_decide_kernel<<<(total + 127) / 128, 128, 0, st>>>(p, rec, static_cast<StepEnv *>(envs), total, act, ss);
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    return NGP_OK;
}

// ngp_play_matches_stepwise after the list check: p and rec are filled in (p.n = matches, p.games = 1).  Wide networks use the
// counts ngp_list_layout_count left in h_counters[8 .. 14).  Synchronises the stream every CHECK_EVERY frames and at the end;
// h_counters[1], [2] then hold the frames and the emulator errors.
int ngp_play_list_stepwise(ngp_handle *h, const RolloutParams &p, const RecordArgs &rec, int n_genomes, bool wide, cudaStream_t st)
{
    const int total = p.n;
    int T = 0;
    long long C = 0;
    int rc = ngp_list_begin(h, p, rec, n_genomes, wide, nullptr, h->step_envs, h->step_x, h->step_act, h->list_chunk, &T, &C, st);
    if (rc != NGP_OK) return rc;
    StepEnv *envs = reinterpret_cast<StepEnv *>(h->step_envs.p);
    if (!wide) NGP_CUDA(h->step_x.ensure((size_t)total * 2 * 6));      // the rows 2e, 2e + 1 ngp_step_frame writes and nothing reads
    float *x = h->step_x.p;
    uint8_t *act = wide ? h->step_act.p : nullptr;
    if (wide) {     // the table's networks are built once per call and run every frame
        rc = ngp_mlp_prepare(h, p.genomes, n_genomes, st);
        if (rc != NGP_OK) return rc;
    }
    for (long long frame = 1;; ++frame) {
        rc = ngp_step_frame(h, p, envs, total, x, x, st);
        if (rc != NGP_OK) return rc;
        if (wide) {
            rc = ngp_mlp_forward_chunks(h, p.genomes, h->list_chunk.p, x, (int)C, T, act, st);
            if (rc != NGP_OK) return rc;
        }
        rc = ngp_list_decide(h, p, rec, envs, total, act, SessionStep{}, st);
        if (rc != NGP_OK) return rc;
        if (frame % CHECK_EVERY == 0) {
            NGP_CUDA(cudaMemcpyAsync(h->h_counters.p, h->d_counters.p, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
            NGP_CUDA(cudaStreamSynchronize(st));
            if (h->h_counters.p[3] >= (unsigned long long)total) break;
        }
    }
    return NGP_OK;
}
