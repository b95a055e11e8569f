// ngp_session.cu -- match sessions (include/ngp.h ngp_session_*): ngp_play_matches_stepwise's per-frame driver with its loop
// turned inside out, so that the caller advances the list one env.step at a time and supplies the decisions of the seats named
// NGP_PLAYER_EXTERNAL.  A step is list_decide_kernel (ngp_stepwise_lists.cu; the external seats' decisions come from the
// caller's actions), the frame kernel below (ngp_step_frame's env.step + find_stuff, plus the caller's observations and flags)
// and, for wide networks, ngp_mlp_forward_chunks over the genome seats' rows.  Nothing in a step synchronises or allocates.
// A translation unit of its own, so that the kernels of the other drivers compile as before.
#include <memory>

#include "stepwise.cuh"

using roll::RecordArgs; using roll::RolloutParams;

// Everything a session reads or writes between two steps is its own; only the handle's immutable tables, its MLP scratch
// (used inside one step) and its packed wide weights (re-packed when another call replaced them) are shared.
struct ngp_session {
    ngp_handle *h;
    RolloutParams p;                                  // p.match_right / match_left = `lists`, p.counters = `counters`
    RecordArgs rec;
    int n, n_genomes, T;
    long long C;                                      // chunks of T MLP rows (wide networks); 0: no MLP batch
    bool wide;
    Buffer<uint8_t> envs;                             // StepEnv[n]
    Buffer<int32_t> lists;                            // [2][n]: right, left with every external seat resolved (session_lists_kernel)
    Buffer<uint8_t> ext;                              // [n] EXT_* bits
    Buffer<float> x; Buffer<uint8_t> act; Buffer<int32_t> chunk;      // the chunk layout of the genome seats' MLP rows
    Buffer<int32_t> frames;                           // frames[n] when the caller passes none
    Buffer<unsigned long long> counters;              // list_decide_kernel's [1] frames, [2] emulator errors, [3] finished, [4] bad actions
    HostBuffer<unsigned long long> h_counters;
};

namespace {

// The lists as roll::plan_env may read them: an external right seat becomes row 0 and an external left seat NGP_OPP_HARDCODED,
// so that no genome pointer is ever formed from NGP_PLAYER_EXTERNAL (the seat's plan is never used: list_decide_kernel takes
// its decisions from the caller); ext[m] records which seats were external.
__global__ void session_lists_kernel(const int32_t *__restrict__ right, const int32_t *__restrict__ left, int n, int32_t *__restrict__ lists,
                                     uint8_t *__restrict__ ext)
{
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n) return;
    const int r = right[m], l = left[m];
    lists[m] = r == NGP_PLAYER_EXTERNAL ? 0 : r;
    lists[n + m] = l == NGP_PLAYER_EXTERNAL ? NGP_OPP_HARDCODED : l;
    ext[m] = (l == NGP_PLAYER_EXTERNAL ? EXT_LEFT : 0) | (r == NGP_PLAYER_EXTERNAL ? EXT_RIGHT : 0);
}

// ngp_step_frame's frame for a session: env.step + find_stuff of every running match; on a model-call frame the rows of the
// external seats go to obs[e][0] (left, x-mirrored) / obs[e][1] (right), those of genome seats to x (wide networks; x == null:
// the decide kernel runs the FP64 policies); flags[e] gets NEED on a model-call frame of a match with an external seat, DONE
// (and EMULATOR_ERROR) once the match has ended.
template <int CORE>
__global__ void __launch_bounds__(32) session_frame_kernel(RolloutParams p, StepEnv *envs, int total, float *__restrict__ x,
                                                           float *__restrict__ obs, uint8_t *__restrict__ flags)
{
    __shared__ a26::Tables T;
    __shared__ uint32_t ram_smem[32 * 32];
    load_tables_cta(T, p.tables);
    const int e = blockIdx.x * 32 + threadIdx.x;
    if (e >= total) return;
    StepEnv &v = envs[e];
    if (v.done) {
        flags[e] = NGP_SESSION_DONE | (v.emu_error ? NGP_SESSION_EMULATOR_ERROR : 0);
        return;
    }
    double loc[3][2], lb[2];
    uint8_t f = 0;
    if (step_env_frame<CORE>(p, v, T, &ram_smem[threadIdx.x], loc, lb)) {
        if (v.ext & EXT_RIGHT) write_inference_row(obs + (size_t)e * 12 + 6, loc[0], lb, loc[2][0], loc[1][0]);
        else if (x) write_inference_row(x + (size_t)v.right_row * 6, loc[0], lb, loc[2][0], loc[1][0]);
        if ((v.ext & EXT_LEFT) || (x && v.left_kind == pol::KIND_MLP)) {
            const double fball[2] = {loc[0][0], __dsub_rn(160.0, loc[0][1])}, flast[2] = {lb[0], __dsub_rn(160.0, lb[1])};
            write_inference_row(v.ext & EXT_LEFT ? obs + (size_t)e * 12 : x + (size_t)v.left_row * 6, fball, flast, loc[1][0], loc[2][0]);
        }
        f = v.ext ? NGP_SESSION_NEED : 0;
    }
    flags[e] = f;
}

}  // namespace

// env.step of every running match and, for wide networks, the MLP rows of the genome seats
static int session_frame(ngp_session *s, float *obs, uint8_t *flags, cudaStream_t st)
{
    ngp_handle *h = s->h;
    StepEnv *envs = reinterpret_cast<StepEnv *>(s->envs.p);
    float *x = s->C > 0 ? s->x.p : nullptr;
    if (s->p.core) session_frame_kernel<1><<<(s->n + 31) / 32, 32, 0, st>>>(s->p, envs, s->n, x, obs, flags);
    else session_frame_kernel<0><<<(s->n + 31) / 32, 32, 0, st>>>(s->p, envs, s->n, x, obs, flags);
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    if (s->C > 0) {
        if (h->prep_src != s->p.genomes || h->prep_n != s->n_genomes) {     // another call packed another table since the last step
            const int rc = ngp_mlp_prepare(h, s->p.genomes, s->n_genomes, st);
            if (rc != NGP_OK) return rc;
        }
        const int rc = ngp_mlp_forward_chunks(h, s->p.genomes, s->chunk.p, s->x.p, (int)s->C, s->T, s->act.p, st);
        if (rc != NGP_OK) return rc;
    }
    return NGP_OK;
}

// ngp_session_begin after the list check (play_match_list, ngp_core.cu): p and rec as ngp_play_matches_stepwise gets them, with
// the caller's lists, which may name NGP_PLAYER_EXTERNAL
int ngp_session_start(ngp_handle *h, const RolloutParams &p, const RecordArgs &rec, int n_genomes, bool wide, float *obs, uint8_t *flags,
                      cudaStream_t st, ngp_session **out)
{
    auto s = std::make_unique<ngp_session>();        // freed with everything it holds on an early return
    s->h = h; s->p = p; s->rec = rec; s->n = p.n; s->n_genomes = n_genomes; s->wide = wide;
    const int n = p.n;
    NGP_CUDA(s->counters.ensure(8));
    NGP_CUDA(s->h_counters.ensure(8));
    NGP_CUDA(s->lists.ensure(2 * (size_t)n));
    NGP_CUDA(s->ext.ensure((size_t)n));
    if (!p.frames) {
        NGP_CUDA(s->frames.ensure((size_t)n));
        s->p.frames = s->frames.p;
    }
    s->p.counters = s->counters.p;
    NGP_CUDA(cudaMemsetAsync(s->counters.p, 0, 8 * sizeof(unsigned long long), st));
    session_lists_kernel<<<(n + 127) / 128, 128, 0, st>>>(p.match_right, p.match_left, n, s->lists.p, s->ext.p);
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    s->p.match_right = s->lists.p; s->p.match_left = s->lists.p + n;
    int rc = ngp_list_begin(h, s->p, rec, n_genomes, wide, s->ext.p, s->envs, s->x, s->act, s->chunk, &s->T, &s->C, st);
    if (rc != NGP_OK) return rc;
    if (s->C > 0) {
        rc = ngp_mlp_prepare(h, p.genomes, n_genomes, st);
        if (rc != NGP_OK) return rc;
    }
    rc = session_frame(s.get(), obs, flags, st);
    if (rc != NGP_OK) return rc;
    h->sessions.push_back(s.get());
    *out = s.release();
    return NGP_OK;
}

extern "C" int ngp_session_step(ngp_session *s, const uint8_t *actions, float *obs, uint8_t *flags, ngp_game_state *capture, void *stream)
{
    NGP_REQUIRE(s && actions && obs && flags, "ngp_session_step: bad arguments (actions, obs and flags are required)");
    NGP_REQUIRE(((uintptr_t)obs & 3) == 0 && ((uintptr_t)capture & 15) == 0, "ngp_session_step: obs must be 4-byte and capture 16-byte aligned");
    ngp_handle *h = s->h;
    NGP_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    RecordArgs rec = s->rec;
    rec.capture_at = nullptr; rec.capture = capture;
    int rc = ngp_list_decide(h, s->p, rec, s->envs.p, s->n, s->C > 0 ? s->act.p : nullptr, SessionStep{actions, capture != nullptr}, st);
    if (rc != NGP_OK) return rc;
    return session_frame(s, obs, flags, st);
}

extern "C" int ngp_session_status(ngp_session *s, int32_t *running, uint64_t *frames_total, void *stream)
{
    NGP_REQUIRE(s, "ngp_session_status: null session");
    NGP_CUDA(cudaSetDevice(s->h->device));
    cudaStream_t st = (cudaStream_t)stream;
    NGP_CUDA(cudaMemcpyAsync(s->h_counters.p, s->counters.p, 5 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    NGP_CUDA(cudaStreamSynchronize(st));
    const unsigned long long *c = s->h_counters.p, run = (unsigned long long)s->n - c[3];
    if (running) *running = (int32_t)run;
    if (frames_total) *frames_total = c[1] + run;            // every running match has played one env.step not decided yet
    if (c[2]) {
        ngp_set_error("ngp_session_status: %llu matches stopped on an emulator error", c[2]);
        return NGP_ERR_EMULATOR;
    }
    if (c[4]) {
        ngp_set_error("ngp_session_status: %llu consumed actions were outside 0..2 and played as NGP_ACT_NONE", c[4]);
        return NGP_ERR_INVALID;
    }
    return NGP_OK;
}

extern "C" int ngp_session_end(ngp_session *s)
{
    if (!s) return NGP_OK;
    ngp_handle *h = s->h;
    cudaSetDevice(h->device);
    for (size_t i = 0; i < h->sessions.size(); ++i)
        if (h->sessions[i] == s) { h->sessions.erase(h->sessions.begin() + i); break; }
    delete s;                                                // cudaFree waits for the device's work, this session's included
    return NGP_OK;
}
