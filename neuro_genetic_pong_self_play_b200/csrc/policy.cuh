// policy.cuh -- device-side policy pieces used inside the fused rollout:
//   deterministic FP64 sigmoid MLP  (numpy_nn.NeuralNetwork.run, /root/reference/numpy_nn.py:120-137)
//   scripted bots                    (/root/reference/dumb_ais.py:1-25)
//   bounds clamp                     (/root/reference/utils.py:71-77)
//   Philox4x32-10 counter RNG        (stands in for np.random.choice, /root/reference/utils.py:112-113)
// All double arithmetic uses explicitly rounded intrinsics (no FMA contraction) so the result is
// bit-identical to the CPU oracle's restatement compiled with -ffp-contract=off.
#pragma once
#include <stdint.h>

namespace pol {

enum { ACT_NONE = 0, ACT_UP = 1, ACT_DOWN = 2 };
enum { KIND_HARDCODED = 0, KIND_SCORE_HARDCODED = 1, KIND_MLP = 2 };
constexpr int FUSED_MAX_WIDTH = 32;     // widest layer the fused (thread-per-env) MLP supports

struct Shape {
    int n_layers;
    int nodes[8];
    int bias;
};

// genes of one network: a (nodes[l] + bias) x nodes[l + 1] weight matrix per layer, in reference gene order
inline int gene_size(const Shape &sh)
{
    int total = 0;
    for (int i = 0; i + 1 < sh.n_layers; ++i) total += (sh.nodes[i] + (sh.bias ? 1 : 0)) * sh.nodes[i + 1];
    return total;
}

#ifdef __CUDACC__

__device__ __forceinline__ void philox4x32(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t out[4])
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        uint32_t n0 = h1 ^ c1 ^ k0, n2 = h0 ^ c3 ^ k1;
        c0 = n0; c1 = l1; c2 = n2; c3 = l0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// the per-frame random action bit of get_actions (main.py:139-140): fresh for every (generation, environment, frame, player)
__device__ __forceinline__ uint32_t random_action_bit(uint64_t seed, uint64_t generation, uint32_t env_id, uint32_t frame, uint32_t stream)
{
    uint32_t o[4];
    philox4x32(env_id, frame, ((uint32_t)generation << 1) | stream, 0x504F4E47u, (uint32_t)seed, (uint32_t)(seed >> 32), o);
    return o[0] & 1u;
}

// exp() from IEEE +,*,floor only: identical bits on host and device
__device__ __forceinline__ double det_exp(double x)
{
    const double LN2_HI = 6.93147180369123816490e-01, LN2_LO = 1.90821492927058770002e-10, INV_LN2 = 1.44269504088896338700e+00;
    if (x != x) return x;
    if (x > 709.0) return __longlong_as_double(0x7FF0000000000000LL);
    if (x < -708.0) return 0.0;
    double k = floor(__dadd_rn(__dmul_rn(x, INV_LN2), 0.5));
    double r = __dsub_rn(__dsub_rn(x, __dmul_rn(k, LN2_HI)), __dmul_rn(k, LN2_LO));
    double p = 1.0 / 6227020800.0;
    p = __dadd_rn(__dmul_rn(p, r), 1.0 / 479001600.0);
    p = __dadd_rn(__dmul_rn(p, r), 1.0 / 39916800.0);
    p = __dadd_rn(__dmul_rn(p, r), 1.0 / 3628800.0);
    p = __dadd_rn(__dmul_rn(p, r), 1.0 / 362880.0);
    p = __dadd_rn(__dmul_rn(p, r), 1.0 / 40320.0);
    p = __dadd_rn(__dmul_rn(p, r), 1.0 / 5040.0);
    p = __dadd_rn(__dmul_rn(p, r), 1.0 / 720.0);
    p = __dadd_rn(__dmul_rn(p, r), 1.0 / 120.0);
    p = __dadd_rn(__dmul_rn(p, r), 1.0 / 24.0);
    p = __dadd_rn(__dmul_rn(p, r), 1.0 / 6.0);
    p = __dadd_rn(__dmul_rn(p, r), 0.5);
    p = __dadd_rn(__dmul_rn(p, r), 1.0);
    p = __dadd_rn(__dmul_rn(p, r), 1.0);
    long long ki = (long long)k;
    double scale = __longlong_as_double((ki + 1023) << 52);
    return __dmul_rn(p, scale);
}

__device__ __forceinline__ double det_sigmoid(double z)
{
    return __ddiv_rn(1.0, __dadd_rn(1.0, det_exp(-z)));
}

// The same network with its three layer widths known at compile time (the reference's default NETWORK_SHAPE [6,2,2] with
// bias, config.py:30-32): identical operations in identical order -- so identical bits -- but the activations live in registers
// instead of two 33-entry local arrays and the loops are straight-line code.
template <int N0, int N1, int N2>
__device__ __forceinline__ int mlp_fixed_f64(const float *__restrict__ genome, const double *x)
{
    double h[N1], out[N2];
#pragma unroll
    for (int o = 0; o < N1; ++o) {
        double z = 0.0;
#pragma unroll
        for (int i = 0; i < N0; ++i) z = __dadd_rn(z, __dmul_rn((double)__ldg(&genome[o * (N0 + 1) + i]), x[i]));
        z = __dadd_rn(z, __dmul_rn((double)__ldg(&genome[o * (N0 + 1) + N0]), 1.0));
        h[o] = det_sigmoid(z);
    }
    const float *w = genome + (N0 + 1) * N1;
#pragma unroll
    for (int o = 0; o < N2; ++o) {
        double z = 0.0;
#pragma unroll
        for (int i = 0; i < N1; ++i) z = __dadd_rn(z, __dmul_rn((double)__ldg(&w[o * (N1 + 1) + i]), h[i]));
        z = __dadd_rn(z, __dmul_rn((double)__ldg(&w[o * (N1 + 1) + N1]), 1.0));
        out[o] = det_sigmoid(z);
    }
    int best = 0;
#pragma unroll
    for (int o = 1; o < N2; ++o)
        if (out[o] > out[best]) best = o;
    return best == 0 ? ACT_UP : ACT_DOWN;
}

// NeuralNetwork.run in FP64: weights f32 in reference gene order (row-major (out, in+bias), bias
// weight = last column); returns ACT_UP when argmax == 0 (first maximum wins), else ACT_DOWN.
static __device__ __noinline__ int mlp_small_f64(const Shape &sh, const float *__restrict__ genome, const double x[6], double *out_opt)
{
#ifdef __CUDA_ARCH__
    __builtin_assume(__isLocal(x));                 // the caller's observation vector: LDL instead of generic loads
#endif
    if (!out_opt && sh.bias && sh.n_layers == 3 && sh.nodes[0] == 6 && sh.nodes[1] == 2 && sh.nodes[2] == 2) return mlp_fixed_f64<6, 2, 2>(genome, x);
    double cur[FUSED_MAX_WIDTH + 1], nxt[FUSED_MAX_WIDTH + 1];
    const int bias = sh.bias ? 1 : 0;
    for (int i = 0; i < sh.nodes[0]; ++i) cur[i] = x[i];
    const float *w = genome;
    for (int l = 0; l + 1 < sh.n_layers; ++l) {
        const int ni = sh.nodes[l], no = sh.nodes[l + 1];
        if (bias) cur[ni] = 1.0;
        for (int o = 0; o < no; ++o) {
            double z = 0.0;
            for (int i = 0; i < ni + bias; ++i) z = __dadd_rn(z, __dmul_rn((double)__ldg(&w[o * (ni + bias) + i]), cur[i]));
            nxt[o] = det_sigmoid(z);
        }
        w += (ni + bias) * no;
        for (int o = 0; o < no; ++o) cur[o] = nxt[o];
    }
    const int n_out = sh.nodes[sh.n_layers - 1];
    int best = 0;
    for (int o = 0; o < n_out; ++o) {
        if (out_opt) out_opt[o] = cur[o];
        if (cur[o] > cur[best]) best = o;
    }
    return best == 0 ? ACT_UP : ACT_DOWN;
}

__device__ __forceinline__ int hardcoded_ai(const double x[6])
{
    if (x[1] < x[4]) return ACT_UP;
    if (x[1] > x[4]) return ACT_DOWN;
    return ACT_NONE;
}

__device__ __forceinline__ int clamp_action(bool valid, double paddle_row, int action, double paddle_height)
{
    if (valid) {
        if (paddle_row < paddle_height) return ACT_DOWN;
        else if (paddle_row > __dsub_rn(160.0, paddle_height)) return ACT_UP;
    }
    return action;
}

#endif
}  // namespace pol
