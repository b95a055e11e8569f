// ngp_ops.cu -- stand-alone operator kernels of libngp.so:
//   K2  frame -> observation          utils.find_stuff / get_rect_quickly  (utils.py:14-19, 60-68)
//   K3  per-genome grouped MLP        numpy_nn.NeuralNetwork.run           (numpy_nn.py:120-137)
//   K4  GA step                       DEAP selTournament / cxBlend / mutGaussian / varAnd as wired in
//                                     ga.py:85-94 and driven by eaSimple at main.py:165-170
#include <math.h>
#include <stdlib.h>

#include "ngp_internal.h"

// =================================================================================================
// K2: find_stuff.  HBM-bound: 76 800 B of cropped RGB per frame, read once with 16-byte loads.
// The crop [34,194) x 160 x 3 is one contiguous byte range of the frame; a 16-byte vector never
// straddles a row (480 = 30 * 16), and its channel phase is (vector index mod 3).
//
// 192-thread CTAs (a multiple of 3): thread t always sees vectors of phase t % 3, so its twelve
// comparison words (3 targets x 4 words) live in registers, and 4800 vectors per frame are exactly 25
// per thread.  The stream path only asks "does any byte of this vector equal its target byte?" with
// the exact zero-byte test ((z - 0x01010101) & ~z & 0x80808080 on z = data ^ pattern: 3 instructions per
// word and target) -- and only of vectors that differ from the last one found free of target bytes, which
// for the background of a frame is 5 instructions; the rare vectors that hold an object pixel (< 1 % of a
// frame) take the exact per-byte accounting.  One redux.sync per accumulator and frame.
// =================================================================================================
struct FindStuffPatterns {
    uint32_t w[3][3][4];     // [phase][target][word]: target bytes repeated with the phase
    uint32_t clean;          // a byte value that no target channel has, four times: a vector that is free of target bytes
};

constexpr int FS_THREADS = 192;
constexpr int FS_VEC_PER_FRAME = (a26::CROP_BOTTOM - a26::CROP_TOP) * 480 / 16;   // 4800
constexpr int FS_ROUNDS = FS_VEC_PER_FRAME / FS_THREADS;                           // 25
static_assert(FS_ROUNDS * FS_THREADS == FS_VEC_PER_FRAME && FS_THREADS % 3 == 0, "find_stuff tiling");

__device__ __forceinline__ uint32_t fs_zero_byte(uint32_t z) { return (z - 0x01010101u) & ~z & 0x80808080u; }

// Exact accounting of one target in one vector that contains at least one byte matching it.  Sums are kept linear so that
// no per-byte division is needed: a matching byte at offset B of its row with channel ch belongs to column (B - ch) / 3, so
// a target's column sum is (sum of B - sum of ch) / 3, divided once per frame.  Per word: exact zero-byte mask, popcount,
// and the two weighted byte sums as one multiply each (byte 3 of b * c is sum b_i * c_(3-i) for 0/1 bytes b_i).
__device__ __forceinline__ void fs_account(uint32_t &cnt, uint32_t &srow, uint32_t &scol, const uint32_t (&words)[4], const uint32_t (&pt)[4],
                                           uint32_t row, uint32_t byte0, int phase)
{
#pragma unroll
    for (int wi = 0; wi < 4; ++wi) {
        const uint32_t z = words[wi] ^ pt[wi];
        const uint32_t b = (~(((z & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | z) & 0x80808080u) >> 7;     // 1 in every matching byte
        const uint32_t c = __popc(b);
        const uint32_t p0 = (uint32_t)(phase + wi) % 3u, p1 = (p0 + 1u) % 3u, p2 = (p0 + 2u) % 3u;   // channels of bytes 0,1,2 (3 = 0)
        const uint32_t chc = p0 | (p2 << 8) | (p1 << 16) | (p0 << 24);
        const uint32_t sidx = (b * 0x00010203u) >> 24, sch = (b * chc) >> 24;
        cnt += c; srow += c * row; scol += c * (byte0 + 4u * wi) + sidx - sch;
    }
}

__global__ void __launch_bounds__(FS_THREADS, 4) find_stuff_kernel(const uint8_t *__restrict__ frames, int n, FindStuffPatterns pat,
                                                                float *__restrict__ loc, uint8_t *__restrict__ valid)
{
    constexpr int GROUP = 5, GROUPS = FS_ROUNDS / GROUP;      // 5 vectors per thread and step, 5 steps per frame
    __shared__ uint32_t red[2][FS_THREADS / 32][9];          // double-buffered: one barrier per frame
    const int tid = threadIdx.x, phase = tid % 3;
    uint32_t pt[3][4];
#pragma unroll
    for (int t = 0; t < 3; ++t)
#pragma unroll
        for (int wi = 0; wi < 4; ++wi) pt[t][wi] = pat.w[phase][t][wi];
    const int my_frames = blockIdx.x < n ? (n - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
    const int steps = my_frames * GROUPS;
    auto vec_ptr = [&](int step) {
        const size_t f = blockIdx.x + (size_t)(step / GROUPS) * gridDim.x;
        return reinterpret_cast<const uint4 *>(frames + f * (a26::FB_ROWS * 480) + a26::CROP_TOP * 480) + tid + (step % GROUPS) * GROUP * FS_THREADS;
    };
    uint4 cur[GROUP], nxt[GROUP];
    if (steps > 0) {
        const uint4 *p = vec_ptr(0);
#pragma unroll
        for (int j = 0; j < GROUP; ++j) cur[j] = __ldcs(&p[j * FS_THREADS]);
    }
    uint32_t acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};           // per target: count, sum row, sum of (row offset - channel)
    uint32_t clean[4] = {pat.clean, pat.clean, pat.clean, pat.clean};       // the last vector found free of target bytes
    int buf = 0;
#pragma unroll 1
    for (int step = 0; step < steps; ++step) {
        // the next step's 80 bytes are requested before this step's are looked at: loads are always in flight
        if (step + 1 < steps) {
            const uint4 *p = vec_ptr(step + 1);
#pragma unroll
            for (int j = 0; j < GROUP; ++j) nxt[j] = __ldcs(&p[j * FS_THREADS]);
        }
        uint32_t flagged = 0;                                // bit 3j+t: vector j holds a byte of target t
#pragma unroll
        for (int j = 0; j < GROUP; ++j) {
            const uint32_t words[4] = {cur[j].x, cur[j].y, cur[j].z, cur[j].w};
            // a vector equal to one already found free of target bytes needs no test (a thread always sees the same channel
            // phase, so the background of a frame is one and the same vector for it): 5 instructions instead of 40
            if (((words[0] ^ clean[0]) | (words[1] ^ clean[1]) | (words[2] ^ clean[2]) | (words[3] ^ clean[3])) == 0u) continue;
            uint32_t fl = 0;
#pragma unroll
            for (int t = 0; t < 3; ++t) {
                uint32_t any = 0;
#pragma unroll
                for (int wi = 0; wi < 4; ++wi) any |= fs_zero_byte(words[wi] ^ pt[t][wi]);
                if (any) fl |= 1u << t;
            }
            if (fl) flagged |= fl << (3 * j);
            else { clean[0] = words[0]; clean[1] = words[1]; clean[2] = words[2]; clean[3] = words[3]; }
        }
        // rare (< 1 % of the vectors): fetched again (L2) and accounted for exactly; kept out of the unrolled stream so that
        // the hot loop stays a few KB of straight-line code
        if (flagged) {
            const uint4 *p = vec_ptr(step);
            const int g = step % GROUPS;
#pragma unroll 1
            for (int j = 0; j < GROUP; ++j) {
                const uint32_t fl = (flagged >> (3 * j)) & 7u;
                if (!fl) continue;
                const uint4 v = p[j * FS_THREADS];
                const uint32_t words[4] = {v.x, v.y, v.z, v.w};
                const uint32_t k = (uint32_t)tid + (uint32_t)(g * GROUP + j) * FS_THREADS;
                const uint32_t row = k / 30u, byte0 = (k % 30u) * 16u;
                if (fl & 1u) fs_account(acc[0], acc[1], acc[2], words, pt[0], row, byte0, phase);
                if (fl & 2u) fs_account(acc[3], acc[4], acc[5], words, pt[1], row, byte0, phase);
                if (fl & 4u) fs_account(acc[6], acc[7], acc[8], words, pt[2], row, byte0, phase);
            }
        }
        if (step % GROUPS == GROUPS - 1) {                   // frame complete
            const int f = blockIdx.x + (step / GROUPS) * gridDim.x;
#pragma unroll
            for (int i = 0; i < 9; ++i) { acc[i] = __reduce_add_sync(0xFFFFFFFFu, acc[i]); }
            if ((tid & 31) == 0)
#pragma unroll
                for (int i = 0; i < 9; ++i) red[buf][tid >> 5][i] = acc[i];
#pragma unroll
            for (int i = 0; i < 9; ++i) acc[i] = 0;
            __syncthreads();
            if (tid < 3) {
                uint32_t c = 0, sr = 0, sc = 0;
#pragma unroll
                for (int w = 0; w < FS_THREADS / 32; ++w) { c += red[buf][w][3 * tid]; sr += red[buf][w][3 * tid + 1]; sc += red[buf][w][3 * tid + 2]; }
                valid[f * 3 + tid] = c > 0;
                loc[(f * 3 + tid) * 2 + 0] = c ? (float)((double)sr / (double)c) : 0.f;
                loc[(f * 3 + tid) * 2 + 1] = c ? (float)((double)(sc / 3u) / (double)c) : 0.f;
            }
            buf ^= 1;
        }
#pragma unroll
        for (int j = 0; j < GROUP; ++j) cur[j] = nxt[j];
    }
}

extern "C" int ngp_find_stuff(ngp_handle *h, const uint8_t *frames, int32_t n, float *loc, uint8_t *valid, void *stream)
{
    NGP_REQUIRE(h && frames && loc && valid && n > 0, "ngp_find_stuff: bad arguments");
    NGP_REQUIRE(((uintptr_t)frames & 15) == 0, "ngp_find_stuff: frames must be 16-byte aligned");
    NGP_CUDA(cudaSetDevice(h->device));
    FindStuffPatterns pat;
    const uint8_t *targets[3] = {h->cfg.ball_colour, h->cfg.left_colour, h->cfg.right_colour};
    for (int phase = 0; phase < 3; ++phase)
        for (int t = 0; t < 3; ++t)
            for (int w = 0; w < 4; ++w) {
                uint32_t v = 0;
                for (int j = 0; j < 4; ++j) v |= (uint32_t)targets[t][(phase + w * 4 + j) % 3] << (8 * j);
                pat.w[phase][t][w] = v;
            }
    {
        bool used[256] = {false};
        for (int t = 0; t < 3; ++t)
            for (int c = 0; c < 3; ++c) used[targets[t][c]] = true;
        uint32_t b = 0;
        while (used[b]) ++b;                                   // nine target bytes at most: some value is free
        pat.clean = b * 0x01010101u;
    }
    // persistent CTAs over frames, as many as are resident at once
    if (!h->fs_per_sm) {
        int per = 0;
        NGP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, find_stuff_kernel, FS_THREADS, 0));
        h->fs_per_sm = per < 1 ? 1 : per;
    }
    const int per_sm = h->fs_per_sm;
    int grid = n < h->sm_count * per_sm ? n : h->sm_count * per_sm;
    find_stuff_kernel<<<grid, FS_THREADS, 0, (cudaStream_t)stream>>>(frames, n, pat, loc, valid);
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    return NGP_OK;
}

// =================================================================================================
// K3: grouped MLP forward, FP32 FFMA.
//   small nets (every layer <= 32 wide): one thread per (genome, env); the genome's weights are read
//   through the read-only path and broadcast inside the warp.
//   larger nets: one launch per layer, a CTA computes a 64(env) x 64(out) tile for one genome from
//   K-chunks of activations and weights staged in shared memory (4x4 register tile per thread).
// The last layer's pre-activations are accumulated in FP64 and the action is decided on the FP64
// sigmoids so the reference's argmax (first maximum wins; both outputs saturating to 1.0 -> index 0)
// is reproduced (SURVEY hard part 4).
// =================================================================================================
__device__ __forceinline__ float sigmoid_f32(float z) { return 1.0f / (1.0f + expf(-z)); }

__global__ void __launch_bounds__(128) mlp_small_kernel(const float *__restrict__ genomes, const float *__restrict__ x, int n_genomes, int envs,
                                                        pol::Shape sh, int G, uint8_t *__restrict__ act, float *__restrict__ out)
{
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)n_genomes * envs) return;
    const int g = (int)(idx / envs);
    const float *w = genomes + (size_t)g * G;
    const int bias = sh.bias ? 1 : 0;
    float cur[pol::FUSED_MAX_WIDTH + 1], nxt[pol::FUSED_MAX_WIDTH + 1];
    const int n_in = sh.nodes[0];
    for (int i = 0; i < n_in; ++i) cur[i] = x[idx * n_in + i];
    const int L = sh.n_layers - 1;
    double zlast[pol::FUSED_MAX_WIDTH];
    for (int l = 0; l < L; ++l) {
        const int ni = sh.nodes[l], no = sh.nodes[l + 1];
        if (bias) cur[ni] = 1.0f;
        for (int o = 0; o < no; ++o) {
            if (l == L - 1) {
                double z = 0.0;
                for (int i = 0; i < ni + bias; ++i) z += (double)__ldg(&w[o * (ni + bias) + i]) * (double)cur[i];
                zlast[o] = z;
                nxt[o] = (float)pol::det_sigmoid(z);
            } else {
                float z = 0.f;
                for (int i = 0; i < ni + bias; ++i) z = fmaf(__ldg(&w[o * (ni + bias) + i]), cur[i], z);
                nxt[o] = sigmoid_f32(z);
            }
        }
        w += (ni + bias) * no;
        for (int o = 0; o < no; ++o) cur[o] = nxt[o];
    }
    const int n_out = sh.nodes[L];
    int best = 0;
    double sbest = pol::det_sigmoid(zlast[0]);
    for (int o = 1; o < n_out; ++o) {
        double s = pol::det_sigmoid(zlast[o]);
        if (s > sbest) { sbest = s; best = o; }
    }
    act[idx] = best == 0 ? pol::ACT_UP : pol::ACT_DOWN;
    if (out) for (int o = 0; o < n_out; ++o) out[idx * n_out + o] = cur[o];
}

// one layer: in[g][e][ni] (+ implicit bias 1) x W_g[no][ni+bias] -> out[g][e][no] (sigmoid), or for the
// last layer FP64 pre-activations zout[g][e][no]
template <bool LAST>
__global__ void __launch_bounds__(256) mlp_layer_kernel(const float *__restrict__ genomes, size_t w_off, int G, const float *__restrict__ in,
                                                        int envs, int ni, int no, int bias, float *__restrict__ outp, double *__restrict__ zout)
{
    constexpr int TE = 64, TO = 64, TK = 32;
    __shared__ float As[TK][TE + 1];     // activations, k-major
    __shared__ float Ws[TK][TO + 1];     // weights, k-major
    const int g = blockIdx.z, e0 = blockIdx.y * TE, o0 = blockIdx.x * TO;
    const float *W = genomes + (size_t)g * G + w_off;
    const float *A = in + (size_t)g * envs * ni;
    const int K = ni + bias;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;     // 16 x 16 threads, 4x4 outputs each
    float acc[4][4];
    double dacc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) { acc[i][j] = 0.f; dacc[i][j] = 0.0; }
    for (int k0 = 0; k0 < K; k0 += TK) {
        for (int i = threadIdx.x; i < TK * TE; i += 256) {
            const int e = i / TK, k = i % TK;
            float v = 0.f;
            if (e0 + e < envs && k0 + k < K) v = (k0 + k < ni) ? A[(size_t)(e0 + e) * ni + k0 + k] : 1.0f;
            As[k][e] = v;
        }
        for (int i = threadIdx.x; i < TK * TO; i += 256) {
            const int o = i / TK, k = i % TK;
            Ws[k][o] = (o0 + o < no && k0 + k < K) ? __ldg(&W[(size_t)(o0 + o) * K + k0 + k]) : 0.f;
        }
        __syncthreads();
#pragma unroll 8
        for (int k = 0; k < TK; ++k) {
            float a[4], w[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) { a[i] = As[k][ty * 4 + i]; w[i] = Ws[k][tx * 4 + i]; }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (LAST) dacc[i][j] += (double)a[i] * (double)w[j];
                    else acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
                }
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int e = e0 + ty * 4 + i, o = o0 + tx * 4 + j;
            if (e < envs && o < no) {
                if (LAST) zout[((size_t)g * envs + e) * no + o] = dacc[i][j];
                else outp[((size_t)g * envs + e) * no + o] = sigmoid_f32(acc[i][j]);
            }
        }
}

// hidden layer with a tiny fan-in (the first layer: 6 observation values + bias) and a wide fan-out: write-bound.
// Thread = one output unit with its weight row in registers, the genome's input rows in shared memory (broadcast
// reads), stores coalesced along the outputs.  Same accumulation order as mlp_layer_kernel (k ascending, bias last).
constexpr int NARROW_K = 8;
template <int NI>        // NI = compile-time fan-in (6: the observation vector), or 0 = run-time fan-in up to NARROW_K - bias
__global__ void __launch_bounds__(128) mlp_narrow_in_kernel(const float *__restrict__ genomes, size_t w_off, int G, const float *__restrict__ in,
                                                            int envs, int ni_rt, int no, int bias, float *__restrict__ outp)
{
    constexpr int TE = 64;
    __shared__ float xs[TE * NARROW_K];
    const int ni = NI ? NI : ni_rt;
    const int g = blockIdx.z, e0 = blockIdx.y * TE, o = blockIdx.x * 128 + threadIdx.x;
    const int K = ni + bias, ne = min(TE, envs - e0);
    const float *src = in + ((size_t)g * envs + e0) * ni;
    for (int i = threadIdx.x; i < ne * ni; i += 128) xs[i] = __ldg(&src[i]);
    float w[NARROW_K];
    const float *W = genomes + (size_t)g * G + w_off + (size_t)min(o, no - 1) * K;
#pragma unroll
    for (int k = 0; k < NARROW_K; ++k) w[k] = k < K ? __ldg(&W[k]) : 0.f;
    float wb = 0.f;
    if (bias) {
#pragma unroll
        for (int k = 0; k < NARROW_K; ++k) if (k == ni) { wb = w[k]; w[k] = 0.f; }
    }
    __syncthreads();
    if (o >= no) return;
    float *dst = outp + ((size_t)g * envs + e0) * no + o;
#pragma unroll 4
    for (int e = 0; e < ne; ++e) {
        const float *xe = xs + e * ni;
        float acc = 0.f;
#pragma unroll
        for (int k = 0; k < (NI ? NI : NARROW_K); ++k) if (NI || k < ni) acc = fmaf(xe[k], w[k], acc);
        if (bias) acc = fmaf(1.0f, wb, acc);
        // fast exponential and reciprocal (ex2.approx, rcp.approx: a few ulp), far inside the 1e-5 bar
        *dst = __fdividef(1.0f, 1.0f + __expf(-acc));
        dst += no;
    }
}

// last layer with few outputs (the action layer): one warp per (genome, env) row, lanes stride over k, FP64
// accumulation, decision on the FP64 sigmoids (reference argmax incl. the saturation tie rule)
__global__ void __launch_bounds__(256) mlp_last_small_kernel(const float *__restrict__ genomes, size_t w_off, int G, const float *__restrict__ in,
                                                             int envs, int ni, int no, int bias, uint8_t *__restrict__ act, float *__restrict__ out)
{
    extern __shared__ float w_s[];                     // [no][ni + bias]
    const int g = blockIdx.y, K = ni + bias;
    const float *W = genomes + (size_t)g * G + w_off;
    for (int i = threadIdx.x; i < no * K; i += blockDim.x) w_s[i] = __ldg(&W[i]);
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int e = blockIdx.x * (blockDim.x >> 5) + warp;
    if (e >= envs) return;
    const float *a = in + ((size_t)g * envs + e) * ni;
    double z[8];
#pragma unroll
    for (int o = 0; o < 8; ++o) z[o] = 0.0;
    for (int k = lane; k < K; k += 32) {
        const double x = k < ni ? (double)__ldg(&a[k]) : 1.0;
#pragma unroll
        for (int o = 0; o < 8; ++o)
            if (o < no) z[o] += (double)w_s[o * K + k] * x;
    }
#pragma unroll
    for (int o = 0; o < 8; ++o)
        for (int off = 16; off; off >>= 1) z[o] += __shfl_down_sync(0xFFFFFFFFu, z[o], off);
    if (lane == 0) {
        int best = 0;
        double sbest = 0.0;
        const size_t row = (size_t)g * envs + e;
        for (int o = 0; o < no; ++o) {
            const double s = pol::det_sigmoid(z[o]);
            if (out) out[row * no + o] = (float)s;
            if (o == 0 || s > sbest) { sbest = s; best = o; }
        }
        act[row] = best == 0 ? pol::ACT_UP : pol::ACT_DOWN;
    }
}

// Action layer on top of a wide hidden layer (fan-in a multiple of 128, up to 512; one or two outputs): CTA = one genome,
// warp w owns environments w, w+8, ..  Each lane keeps its 16 k-positions of every weight row in FP64 registers (loaded once
// per genome), streams the activation rows with 16-byte loads (two rows in flight) and accumulates in FP64; the decision
// is taken on the FP64 sigmoids like mlp_last_small_kernel.
template <int NO>
__global__ void __launch_bounds__(256) mlp_last_wide_kernel(const float *__restrict__ genomes, size_t w_off, int G, const float *__restrict__ in,
                                                            int envs, int ni, int bias, uint8_t *__restrict__ act, float *__restrict__ out)
{
    const int g = blockIdx.x, K = ni + bias, kj = ni >> 7;
    const float *W = genomes + (size_t)g * G + w_off;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double w[NO][16];
#pragma unroll
    for (int o = 0; o < NO; ++o)
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int i = 0; i < 4; ++i) w[o][4 * j + i] = j < kj ? (double)__ldg(&W[(size_t)o * K + 128 * j + 4 * lane + i]) : 0.0;
    double wb[NO];
#pragma unroll
    for (int o = 0; o < NO; ++o) wb[o] = bias ? (double)__ldg(&W[(size_t)o * K + ni]) : 0.0;
    for (int e = warp; e < envs; e += 16) {
        const int e2 = e + 8;
        const bool two = e2 < envs;
        const float4 *a0 = reinterpret_cast<const float4 *>(in + ((size_t)g * envs + e) * ni) + lane;
        const float4 *a1 = reinterpret_cast<const float4 *>(in + ((size_t)g * envs + (two ? e2 : e)) * ni) + lane;
        float4 x0[4], x1[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) if (j < kj) { x0[j] = __ldcs(&a0[32 * j]); x1[j] = __ldcs(&a1[32 * j]); }
        double z0[NO], z1[NO];
#pragma unroll
        for (int o = 0; o < NO; ++o) { z0[o] = 0.0; z1[o] = 0.0; }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (j >= kj) continue;
            const double d0[4] = {(double)x0[j].x, (double)x0[j].y, (double)x0[j].z, (double)x0[j].w};
            const double d1[4] = {(double)x1[j].x, (double)x1[j].y, (double)x1[j].z, (double)x1[j].w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int o = 0; o < NO; ++o) { z0[o] += w[o][4 * j + i] * d0[i]; z1[o] += w[o][4 * j + i] * d1[i]; }
        }
#pragma unroll
        for (int o = 0; o < NO; ++o)
            for (int off = 16; off; off >>= 1) {
                z0[o] += __shfl_down_sync(0xFFFFFFFFu, z0[o], off);
                z1[o] += __shfl_down_sync(0xFFFFFFFFu, z1[o], off);
            }
        // lanes 0 .. 2*NO-1 evaluate one FP64 sigmoid each (row r = lane / NO, output o = lane % NO)
        double zmine = 0.0;
#pragma unroll
        for (int r = 0; r < 2; ++r)
#pragma unroll
            for (int o = 0; o < NO; ++o) {
                const double zz = __shfl_sync(0xFFFFFFFFu, (r ? z1[o] : z0[o]) + wb[o], 0);
                if (lane == r * NO + o) zmine = zz;
            }
        const double sg = lane < 2 * NO ? pol::det_sigmoid(zmine) : 0.0;
        int best = 0;
        double sbest = 0.0;
#pragma unroll
        for (int o = 0; o < NO; ++o) {
            const double so = __shfl_sync(0xFFFFFFFFu, sg, (lane < NO ? 0 : NO) + o);     // lane 0 reads row 0, lane NO reads row 1
            if (o == 0 || so > sbest) { sbest = so; best = o; }
        }
        if (lane < 2 * NO && (lane < NO || two)) {
            const size_t row = (size_t)g * envs + (lane < NO ? e : e2);
            if (out) out[row * NO + (lane % NO)] = (float)sg;
            if (lane % NO == 0) act[row] = best == 0 ? pol::ACT_UP : pol::ACT_DOWN;
        }
    }
}

__global__ void mlp_decide_kernel(const double *__restrict__ z, long long rows, int n_out, uint8_t *__restrict__ act, float *__restrict__ out)
{
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    int best = 0;
    double sbest = 0.0;
    for (int o = 0; o < n_out; ++o) {
        double s = pol::det_sigmoid(z[r * n_out + o]);
        if (out) out[r * n_out + o] = (float)s;
        if (o == 0 || s > sbest) { sbest = s; best = o; }
    }
    act[r] = best == 0 ? pol::ACT_UP : pol::ACT_DOWN;
}

int ngp_mlp_layer_tf32(ngp_handle *h, const float *genomes, size_t w_off, const float *in, int n_genomes, int envs, int ni, int no, int bias,
                       float *out, cudaStream_t st);   // ngp_mlp_tf32.cu

int ngp_mlp_layer_tmem(ngp_handle *h, int l, size_t g0, const float *in, int n_genomes, int envs, float *out, cudaStream_t st);  // ngp_mlp_tmem.cu

static int mlp_forward_impl(ngp_handle *h, const float *genomes, const float *x, int32_t n_genomes, int32_t envs, uint8_t *act, float *out,
                            void *stream, bool prepared);
static int mlp_forward_slice(ngp_handle *h, const float *genomes, const float *x, size_t g0, int n_genomes, int envs, uint8_t *act,
                             float *out, cudaStream_t st, bool prepared);

extern "C" int ngp_mlp_forward(ngp_handle *h, const float *genomes, const float *x, int32_t n_genomes, int32_t envs, uint8_t *act,
                               float *out, void *stream)
{
    return mlp_forward_impl(h, genomes, x, n_genomes, envs, act, out, stream, false);
}

extern "C" int ngp_mlp_forward_prepared(ngp_handle *h, const float *genomes, const float *x, int32_t n_genomes, int32_t envs, uint8_t *act,
                                        float *out, void *stream)
{
    NGP_REQUIRE(h && h->prep_src == genomes && h->prep_n == n_genomes && n_genomes > 0,
                "ngp_mlp_forward_prepared: call ngp_mlp_prepare on these genomes first");
    return mlp_forward_impl(h, genomes, x, n_genomes, envs, act, out, stream, true);
}

static int mlp_forward_impl(ngp_handle *h, const float *genomes, const float *x, int32_t n_genomes, int32_t envs, uint8_t *act, float *out,
                            void *stream, bool prepared)
{
    NGP_REQUIRE(h && genomes && x && act && n_genomes > 0 && envs > 0, "ngp_mlp_forward: bad arguments");
    NGP_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    const pol::Shape &sh = h->shape;
    int widest = 0;
    for (int i = 0; i < sh.n_layers; ++i) widest = sh.nodes[i] > widest ? sh.nodes[i] : widest;
    const long long rows = (long long)n_genomes * envs;
    if (widest <= pol::FUSED_MAX_WIDTH) {
        mlp_small_kernel<<<(unsigned)((rows + 127) / 128), 128, 0, st>>>(genomes, x, n_genomes, envs, sh, h->gene_size, act, out);
        h->launches++;
        NGP_CUDA(cudaGetLastError());
        return NGP_OK;
    }
    const int n_in = sh.nodes[0], n_out = sh.nodes[sh.n_layers - 1];
    const size_t slice_rows = (size_t)(n_genomes < MLP_GENOME_SLICE ? n_genomes : MLP_GENOME_SLICE) * envs;
    NGP_CUDA(h->mlp_a.ensure(slice_rows * widest));
    NGP_CUDA(h->mlp_b.ensure(slice_rows * widest));
    NGP_CUDA(h->mlp_z.ensure(slice_rows * n_out));
    for (int g0 = 0; g0 < n_genomes; g0 += MLP_GENOME_SLICE) {
        const int gn = n_genomes - g0 < MLP_GENOME_SLICE ? n_genomes - g0 : MLP_GENOME_SLICE;
        const size_t r0 = (size_t)g0 * envs;
        const int rc = mlp_forward_slice(h, genomes + (size_t)g0 * h->gene_size, x + r0 * n_in, g0, gn, envs, act + r0,
                                         out ? out + r0 * n_out : nullptr, st, prepared);
        if (rc != NGP_OK) return rc;
    }
    return NGP_OK;
}

// the layers of the wide path for genomes [g0, g0 + n_genomes) of the call (pointers already offset to g0; g0 locates the
// genomes in the prepared packed copy)
static int mlp_forward_slice(ngp_handle *h, const float *genomes, const float *x, size_t g0, int n_genomes, int envs, uint8_t *act,
                             float *out, cudaStream_t st, bool prepared)
{
    const pol::Shape &sh = h->shape;
    const long long rows = (long long)n_genomes * envs;
    const float *in = x;
    float *bufs[2] = {h->mlp_a.p, h->mlp_b.p};
    size_t w_off = 0;
    const int bias = sh.bias ? 1 : 0, L = sh.n_layers - 1;
    for (int l = 0; l < L; ++l) {
        const int ni = sh.nodes[l], no = sh.nodes[l + 1];
        dim3 grid((no + 63) / 64, (envs + 63) / 64, n_genomes);
        bool launched = false;
        if (l == L - 1 && no <= 8 && (size_t)no * (ni + bias) * 4 <= 48 * 1024) {
            // action layer: warp-per-row dot products, decision fused (no intermediate buffer)
            if (no <= 2 && ni % 128 == 0 && ni <= 512 && l > 0) {      // on top of a wide hidden layer (our own 16-byte aligned scratch)
                if (no == 2) mlp_last_wide_kernel<2><<<n_genomes, 256, 0, st>>>(genomes, w_off, h->gene_size, in, envs, ni, bias, act, out);
                else mlp_last_wide_kernel<1><<<n_genomes, 256, 0, st>>>(genomes, w_off, h->gene_size, in, envs, ni, bias, act, out);
                h->launches++;
                NGP_CUDA(cudaGetLastError());
                return NGP_OK;
            }
            dim3 g2((envs + 7) / 8, n_genomes);
            mlp_last_small_kernel<<<g2, 256, (size_t)no * (ni + bias) * 4, st>>>(genomes, w_off, h->gene_size, in, envs, ni, no, bias, act, out);
            h->launches++;
            NGP_CUDA(cudaGetLastError());
            return NGP_OK;
        }
        if (l != L - 1 && ni + bias <= NARROW_K) {
            dim3 g3((no + 127) / 128, (envs + 63) / 64, n_genomes);
            if (ni == 6) mlp_narrow_in_kernel<6><<<g3, 128, 0, st>>>(genomes, w_off, h->gene_size, in, envs, ni, no, bias, bufs[l & 1]);
            else mlp_narrow_in_kernel<0><<<g3, 128, 0, st>>>(genomes, w_off, h->gene_size, in, envs, ni, no, bias, bufs[l & 1]);
            h->launches++;
            NGP_CUDA(cudaGetLastError());
            launched = true;
        }
        if (!launched && prepared && l != L - 1 && !h->opt_mlp_no_tf32) {
            // prepared genome set: weights stream from HBM straight into tensor memory (ngp_mlp_tmem.cu)
            const int rc = ngp_mlp_layer_tmem(h, l, g0, in, n_genomes, envs, bufs[l & 1], st);
            if (rc == NGP_OK) launched = true;
            else if (rc != NGP_ERR_UNSUPPORTED) return rc;
        }
        if (!launched && l != L - 1 && !h->opt_mlp_no_tf32) {
            // wide hidden layer with enough environments per genome: tensor cores (3xTF32, tcgen05 + TMEM)
            const int rc = ngp_mlp_layer_tf32(h, genomes, w_off, in, n_genomes, envs, ni, no, bias, bufs[l & 1], st);
            if (rc == NGP_OK) launched = true;
            else if (rc != NGP_ERR_UNSUPPORTED) return rc;
        }
        if (!launched) {
            if (l == L - 1) mlp_layer_kernel<true><<<grid, 256, 0, st>>>(genomes, w_off, h->gene_size, in, envs, ni, no, bias, nullptr, h->mlp_z.p);
            else mlp_layer_kernel<false><<<grid, 256, 0, st>>>(genomes, w_off, h->gene_size, in, envs, ni, no, bias, bufs[l & 1], nullptr);
            h->launches++;
            NGP_CUDA(cudaGetLastError());
        }
        in = bufs[l & 1];
        w_off += (size_t)(ni + bias) * no;
    }
    mlp_decide_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, st>>>(h->mlp_z.p, rows, sh.nodes[L], act, out);
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    return NGP_OK;
}

// =================================================================================================
// K4: GA step.  Counter-based RNG: Philox4x32-10 keyed by the seed; the counter encodes
// (slot, block-within-slot, generation, stream) so results do not depend on launch geometry.
// =================================================================================================
#include "ga_streams.cuh"

__global__ void init_population_kernel(float *__restrict__ genomes, long long total, uint64_t seed)
{
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;      // one Philox call -> 4 genes
    if (q * 4 >= total) return;
    uint32_t o[4];
    pol::philox4x32((uint32_t)q, (uint32_t)(q >> 32), 0, STREAM_INIT, (uint32_t)seed, (uint32_t)(seed >> 32), o);
    for (int j = 0; j < 4; ++j)
        if (q * 4 + j < total) genomes[q * 4 + j] = u01(o[j]);
}

// avg / std (population, ddof=0) / min / max of the fitness vector (main.py:158-162)
__global__ void __launch_bounds__(1024) fitness_stats_kernel(const double *__restrict__ fitness, int n, double *__restrict__ stats)
{
    __shared__ double s_sum[32], s_min[32], s_max[32];
    __shared__ double s_mean;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double sum = 0.0, mn = INFINITY, mx = -INFINITY;
    for (int i = threadIdx.x; i < n; i += blockDim.x) { double f = fitness[i]; sum += f; mn = fmin(mn, f); mx = fmax(mx, f); }
    for (int off = 16; off; off >>= 1) {
        sum += __shfl_down_sync(0xFFFFFFFFu, sum, off);
        mn = fmin(mn, __shfl_down_sync(0xFFFFFFFFu, mn, off));
        mx = fmax(mx, __shfl_down_sync(0xFFFFFFFFu, mx, off));
    }
    if (lane == 0) { s_sum[warp] = sum; s_min[warp] = mn; s_max[warp] = mx; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0, a = INFINITY, b = -INFINITY;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { t += s_sum[w]; a = fmin(a, s_min[w]); b = fmax(b, s_max[w]); }
        s_mean = t / n; stats[0] = s_mean; stats[2] = a; stats[3] = b;
    }
    __syncthreads();
    const double mean = s_mean;
    double sq = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) { double d = fitness[i] - mean; sq += d * d; }
    for (int off = 16; off; off >>= 1) sq += __shfl_down_sync(0xFFFFFFFFu, sq, off);
    __syncthreads();
    if (lane == 0) s_sum[warp] = sq;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += s_sum[w];
        stats[1] = sqrt(t / n);
    }
}

// selTournament: one warp per offspring slot; lanes split the T draws; winner = max fitness, first in
// draw order on ties.
__global__ void __launch_bounds__(256) select_tournament_kernel(const double *__restrict__ fitness, int n, int k, int T, const int32_t *__restrict__ draws,
                                                                uint64_t seed, uint64_t generation, int32_t *__restrict__ parent_idx)
{
    const int slot = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (slot >= k) return;
    double best_f = -INFINITY;
    int best_pos = 0x7FFFFFFF, best_idx = -1;
    if (draws) {
        for (int j = lane; j < T; j += 32) {
            const int idx = draws[(size_t)slot * T + j];
            const double f = fitness[idx];
            if (best_idx < 0 || f > best_f) { best_f = f; best_pos = j; best_idx = idx; }
        }
    } else {
        // draw j comes from Philox block j/4, word j%4; lanes take whole blocks
        for (int b = lane; b * 4 < T; b += 32) {
            uint32_t o[4];
            pol::philox4x32((uint32_t)slot, (uint32_t)b, (uint32_t)generation, STREAM_SELECT, (uint32_t)seed, (uint32_t)(seed >> 32), o);
            for (int w = 0; w < 4 && b * 4 + w < T; ++w) {
                const int idx = (int)(((uint64_t)o[w] * (uint64_t)n) >> 32);
                const double f = fitness[idx];
                if (best_idx < 0 || f > best_f) { best_f = f; best_pos = b * 4 + w; best_idx = idx; }
            }
        }
    }
    for (int off = 16; off; off >>= 1) {
        const double of = __shfl_down_sync(0xFFFFFFFFu, best_f, off);
        const int op = __shfl_down_sync(0xFFFFFFFFu, best_pos, off);
        const int oi = __shfl_down_sync(0xFFFFFFFFu, best_idx, off);
        if (oi >= 0 && (best_idx < 0 || of > best_f || (of == best_f && op < best_pos))) { best_f = of; best_pos = op; best_idx = oi; }
    }
    if (lane == 0) parent_idx[slot] = best_idx;
}

// ---- selTournament for large populations: order statistics instead of N/4 draws per slot ----
// The winner of a tournament of T independent uniform draws (with replacement) is the drawn individual of highest fitness.
// With the population sorted by fitness (descending) the best rank R among T draws has P(R >= r) = ((N - r) / N)^T, so
// R = floor(N * (1 - u^(1/T))) for one uniform u in (0, 1] has exactly the tournament's distribution; among individuals of
// EQUAL fitness DEAP keeps the first drawn one, which is uniform over the tie group (draws are exchangeable): a second
// uniform picks inside the group.  One Philox block per slot instead of T/4: O(N log^2 N) for the sort + O(N log N) for the
// picks instead of O(N^2 / 4).  Same distribution as the draw-by-draw kernel, not the same draws, so it is only used on the
// Philox path (never with injected draws) and only from `select_os_min_t` (default 8192) aspirants upwards.
constexpr uint32_t STREAM_SELECT_OS = 0x53454C32u;

__device__ __forceinline__ unsigned long long fitness_sort_key(double f)
{
    // monotone map of IEEE doubles to unsigned integers, then inverted: ascending key order = descending fitness
    unsigned long long b = (unsigned long long)__double_as_longlong(f);
    b = (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
    return ~b;
}

__global__ void rank_init_kernel(const double *__restrict__ fitness, int n, int n_pow2, unsigned long long *__restrict__ keys, int32_t *__restrict__ idx)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pow2) return;
    keys[i] = i < n ? fitness_sort_key(fitness[i]) : ~0ull;          // padding sorts last
    idx[i] = i < n ? i : 0x7FFFFFFF;
}

__device__ __forceinline__ bool rank_after(unsigned long long ka, int ia, unsigned long long kb, int ib)
{
    return ka > kb || (ka == kb && ia > ib);                         // ties: lower population index first
}

// bitonic sort, ascending in (key, index).  Steps with partner distance j < RANK_TILE run inside shared memory.
constexpr int RANK_TILE = 2048;
__global__ void __launch_bounds__(RANK_TILE / 2) rank_sort_tile_kernel(unsigned long long *__restrict__ keys, int32_t *__restrict__ idx, int k_first, int k_last)
{
    __shared__ unsigned long long sk[RANK_TILE];
    __shared__ int32_t si[RANK_TILE];
    const int base = blockIdx.x * RANK_TILE;
    for (int t = threadIdx.x; t < RANK_TILE; t += blockDim.x) { sk[t] = keys[base + t]; si[t] = idx[base + t]; }
    __syncthreads();
    for (int k = k_first; k <= k_last; k <<= 1) {
        for (int j = min(k >> 1, RANK_TILE >> 1); j > 0; j >>= 1) {
            const int t = threadIdx.x;
            const int a = 2 * t - (t & (j - 1)), b = a + j;          // the t-th pair with distance j
            const bool up = (((base + a) & k) == 0);
            const bool swap = rank_after(sk[a], si[a], sk[b], si[b]) == up;
            if (swap) {
                const unsigned long long tk = sk[a]; sk[a] = sk[b]; sk[b] = tk;
                const int32_t ti = si[a]; si[a] = si[b]; si[b] = ti;
            }
            __syncthreads();
        }
    }
    for (int t = threadIdx.x; t < RANK_TILE; t += blockDim.x) { keys[base + t] = sk[t]; idx[base + t] = si[t]; }
}

__global__ void rank_sort_global_kernel(unsigned long long *__restrict__ keys, int32_t *__restrict__ idx, int n_pow2, int k, int j)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_pow2 / 2) return;
    const int a = 2 * t - (t & (j - 1)), b = a + j;
    const bool up = ((a & k) == 0);
    const unsigned long long ka = keys[a], kb = keys[b];
    const int32_t ia = idx[a], ib = idx[b];
    if (rank_after(ka, ia, kb, ib) == up) { keys[a] = kb; keys[b] = ka; idx[a] = ib; idx[b] = ia; }
}

__global__ void select_order_stat_kernel(const unsigned long long *__restrict__ keys, const int32_t *__restrict__ idx, int n, int k, int T, uint64_t seed,
                                         uint64_t generation, int32_t *__restrict__ parent_idx)
{
    const int slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= k) return;
    uint32_t o[4];
    pol::philox4x32((uint32_t)slot, 0u, (uint32_t)generation, STREAM_SELECT_OS, (uint32_t)seed, (uint32_t)(seed >> 32), o);
    // u in (0, 1] with 53 bits; best rank among T uniform draws over n ranks
    const double u = ((double)((((unsigned long long)o[0] << 32) | o[1]) >> 11) + 1.0) * (1.0 / 9007199254740992.0);
    long long r = (long long)floor((double)n * -expm1(log(u) / (double)T));
    r = r < 0 ? 0 : (r > n - 1 ? n - 1 : r);
    // tie group [lo, hi) of rank r in the sorted keys
    const unsigned long long key = keys[r];
    int lo = 0, hi = (int)r;                                         // first position with keys[pos] == key
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (keys[mid] < key) lo = mid + 1; else hi = mid; }
    const int first = lo;
    lo = (int)r; hi = n;                                             // first position with keys[pos] > key
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (keys[mid] <= key) lo = mid + 1; else hi = mid; }
    const int count = lo - first;
    const int pick = first + (int)(((unsigned long long)o[2] * (unsigned long long)count) >> 32);
    parent_idx[slot] = idx[pick];
}

static int select_dispatch(ngp_handle *h, const double *fitness, int n, int k, int T, const int32_t *draws, uint64_t seed, uint64_t generation,
                           int32_t *parent_idx, cudaStream_t st)
{
    const int min_t = h->opt_select_os_min_t > 0 ? h->opt_select_os_min_t : 8192;
    if (draws || T < min_t) {
        select_tournament_kernel<<<(unsigned)(((long long)k * 32 + 255) / 256), 256, 0, st>>>(fitness, n, k, T, draws, seed, generation, parent_idx);
        h->launches++;
        NGP_CUDA(cudaGetLastError());
        return NGP_OK;
    }
    int n_pow2 = RANK_TILE;
    while (n_pow2 < n) n_pow2 <<= 1;
    NGP_CUDA(h->rank_keys.ensure(n_pow2));
    NGP_CUDA(h->rank_idx.ensure(n_pow2));
    unsigned long long *keys = h->rank_keys.p;
    int32_t *idx = h->rank_idx.p;
    rank_init_kernel<<<(n_pow2 + 255) / 256, 256, 0, st>>>(fitness, n, n_pow2, keys, idx);
    rank_sort_tile_kernel<<<n_pow2 / RANK_TILE, RANK_TILE / 2, 0, st>>>(keys, idx, 2, RANK_TILE);     // sorted tiles, alternating direction
    h->launches += 2;
    for (int kk = RANK_TILE * 2; kk <= n_pow2; kk <<= 1) {
        for (int j = kk >> 1; j >= RANK_TILE; j >>= 1) {
            rank_sort_global_kernel<<<(n_pow2 / 2 + 255) / 256, 256, 0, st>>>(keys, idx, n_pow2, kk, j);
            h->launches++;
        }
        rank_sort_tile_kernel<<<n_pow2 / RANK_TILE, RANK_TILE / 2, 0, st>>>(keys, idx, kk, kk);        // distances below the tile size
        h->launches++;
    }
    select_order_stat_kernel<<<(k + 255) / 256, 256, 0, st>>>(keys, idx, n, k, T, seed, generation, parent_idx);
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    return NGP_OK;
}

// varAnd: clone selected parents, blend-crossover pairs (0,1),(2,3).., then Gaussian mutation.
// One thread per (pair, gene).  Every FP32 operation is individually rounded (no FMA contraction) so
// that, given injected noise, the children match the numpy restatement bit-for-bit.
__global__ void __launch_bounds__(256) vary_kernel(const float *__restrict__ genomes, const int32_t *__restrict__ parent_idx, int n, int G,
                                                   ngp_noise noise, uint64_t seed, uint64_t generation, float cxpb, float alpha, float mutpb,
                                                   float mu, float sigma, float indpb, float *__restrict__ next, uint8_t *__restrict__ invalid)
{
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int pairs = (n + 1) / 2;
    if (tid >= (long long)pairs * G) return;
    const int pair = (int)(tid / G), gene = (int)(tid % G);
    const int i0 = 2 * pair, i1 = 2 * pair + 1;
    const bool has1 = i1 < n;
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32), gen = (uint32_t)generation;
    float x0 = genomes[(size_t)parent_idx[i0] * G + gene];
    float x1 = has1 ? genomes[(size_t)parent_idx[i1] * G + gene] : 0.f;
    uint32_t o[4];
    // ---- mate (ga.py:89, cxBlend) ----
    bool do_cx = false;
    if (has1) {
        if (noise.cx_do) do_cx = noise.cx_do[pair] != 0;
        else { pol::philox4x32((uint32_t)pair, 0, gen, STREAM_CXDO, k0, k1, o); do_cx = u01(o[0]) < cxpb; }
    }
    if (do_cx) {
        float u;
        if (noise.cx_u) u = noise.cx_u[(size_t)pair * G + gene];
        else { pol::philox4x32((uint32_t)pair, (uint32_t)(gene >> 2), gen, STREAM_CXU, k0, k1, o); u = u01(o[gene & 3]); }
        blend_gene(alpha, u, x0, x1);
    }
    // ---- mutate (ga.py:91-92, mutGaussian) ----
    bool do_mut[2];
    for (int s = 0; s < 2; ++s) {
        const int ind = s ? i1 : i0;
        if (s && !has1) { do_mut[s] = false; continue; }
        if (noise.mut_do) do_mut[s] = noise.mut_do[ind] != 0;
        else { pol::philox4x32((uint32_t)ind, 0, gen, STREAM_MUTDO, k0, k1, o); do_mut[s] = u01(o[0]) < mutpb; }
        if (do_mut[s]) {
            float u, z;
            if (noise.mut_u) u = noise.mut_u[(size_t)ind * G + gene];
            else { pol::philox4x32((uint32_t)ind, (uint32_t)(gene >> 2), gen, STREAM_MUTU, k0, k1, o); u = u01(o[gene & 3]); }
            if (noise.mut_z) z = noise.mut_z[(size_t)ind * G + gene];
            else z = mut_normal((uint32_t)ind, (uint32_t)gene, gen, k0, k1);
            if (u < indpb) {
                const float step = __fadd_rn(mu, __fmul_rn(sigma, z));
                if (s) x1 = __fadd_rn(x1, step); else x0 = __fadd_rn(x0, step);
            }
        }
    }
    next[(size_t)i0 * G + gene] = x0;
    if (has1) next[(size_t)i1 * G + gene] = x1;
    if (gene == 0) {
        invalid[i0] = (do_cx || do_mut[0]) ? 1 : 0;
        if (has1) invalid[i1] = (do_cx || do_mut[1]) ? 1 : 0;
    }
}

extern "C" int ngp_ga_step(ngp_handle *h, const float *genomes, const double *fitness, int32_t n, uint64_t seed, uint64_t generation,
                           const ngp_noise *noise, float *next, int32_t *parent_idx, uint8_t *invalid, double *stats, void *stream)
{
    NGP_REQUIRE(h && genomes && fitness && next && invalid && n > 0, "ngp_ga_step: bad arguments");
    NGP_REQUIRE(genomes != next, "ngp_ga_step: next must not alias genomes");
    NGP_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    ngp_noise nz;
    memset(&nz, 0, sizeof(nz));
    if (noise) nz = *noise;
    int T = h->cfg.tournament_size;
    if (T < 1) T = 1;
    if (!parent_idx) {
        NGP_CUDA(h->d_parent.ensure(n));
        parent_idx = h->d_parent.p;
    }
    if (stats) {
        fitness_stats_kernel<<<1, 1024, 0, st>>>(fitness, n, stats);
        h->launches++;
        NGP_CUDA(cudaGetLastError());
    }
    {
        const int rc = select_dispatch(h, fitness, n, n, T, nz.sel_draws, seed, generation, parent_idx, st);
        if (rc != NGP_OK) return rc;
    }
    const long long work = (long long)((n + 1) / 2) * h->gene_size;
    vary_kernel<<<(unsigned)((work + 255) / 256), 256, 0, st>>>(genomes, parent_idx, n, h->gene_size, nz, seed, generation, h->cfg.cxpb,
                                                               h->cfg.cx_alpha, h->cfg.mutpb, h->cfg.mut_mu, h->cfg.mut_sigma,
                                                               h->cfg.mut_indpb, next, invalid);
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    return NGP_OK;
}

extern "C" int ngp_select(ngp_handle *h, const double *fitness, int32_t n, int32_t k, const int32_t *draws, uint64_t seed,
                          uint64_t generation, int32_t *parent_idx, void *stream)
{
    NGP_REQUIRE(h && fitness && parent_idx && n > 0 && k > 0, "ngp_select: bad arguments");
    NGP_CUDA(cudaSetDevice(h->device));
    int T = h->cfg.tournament_size;
    if (T < 1) T = 1;
    return select_dispatch(h, fitness, n, k, T, draws, seed, generation, parent_idx, (cudaStream_t)stream);
}

extern "C" int ngp_init_population(ngp_handle *h, float *genomes, int32_t n, uint64_t seed, void *stream)
{
    NGP_REQUIRE(h && genomes && n > 0, "ngp_init_population: bad arguments");
    NGP_CUDA(cudaSetDevice(h->device));
    const long long total = (long long)n * h->gene_size, calls = (total + 3) / 4;
    init_population_kernel<<<(unsigned)((calls + 255) / 256), 256, 0, (cudaStream_t)stream>>>(genomes, total, seed);
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    return NGP_OK;
}
