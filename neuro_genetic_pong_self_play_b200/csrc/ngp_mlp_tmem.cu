// ngp_mlp_tmem.cu -- K3 wide hidden layers, second generation: weights prepared once per genome set (the reference's
// NeuralNetwork.__init__/populate_weights, /root/reference/numpy_nn.py:35-69, runs once per individual and `run` many times
// per episode, main.py:29,84-90), then streamed straight from HBM into TENSOR MEMORY as the A operand of tcgen05.mma.
//
// Why: the first-generation layer (ngp_mlp_tf32.cu) stages raw FP32 weight tiles in shared memory, reads them back, writes
// hi/lo tiles and lets the tensor core read those three times: ~10 bytes of shared-memory traffic per weight byte, which is
// the SM's shared-memory bandwidth at 2.3 TB/s of weights (profiles/README.md).  Here a weight never touches shared memory:
//
//   ngp_mlp_prepare   packs every wide layer of every genome into 128-output x 16-k tiles  [tile][q][row][4 floats]  (one
//                     coalesced 16-byte load per thread and quarter-chunk) and the bias weights into their own vector
//   copy warp         one thread: each 128 x 16 tile is 8 KB of CONTIGUOUS packed memory -> one cp.async.bulk (TMA, 1-D) per chunk
//                     into a deep ring of raw tiles in shared memory (up to 64 KB in flight per CTA, no registers held)
//   A producers       4 warps, thread = output row (= TMEM lane): 4 x LDS.128 of its row (conflict-free), split  w = hi + lo
//                     (hi = tf32-truncated), tcgen05.st hi and lo into a 4-stage ring of TMEM columns
//   B producers       8 warps (4 for 128-environment tiles), one chunk each at a time: activations [env][k] (L2-resident,
//                     16-byte aligned rows) -> registers -> hi/lo tiles in one of four shared-memory stages in the canonical
//                     no-swizzle K-major core-matrix layout; the warps are the prefetch depth of the activations
//   MMA warp          per chunk and k-step of 8:  D += A_lo*B_hi + A_hi*B_lo + A_hi*B_hi  ("3xTF32", error ~2^-21) with A from
//                     TMEM and B from shared memory; tcgen05.commit hands the stage back to both producer groups
//   epilogue          the A producers (their warp owns the TMEM lanes of its rows): tcgen05.ld, + bias, sigmoid, coalesced stores
//
// D^T form as before: M = 128 outputs, N = TN environments (64 or 128: with 128 a genome's weights are streamed once for the
// 2 x 64 rows of the round-robin stepwise evaluation), K = fan-in (bias handled in the epilogue, so K = 512 exactly for the
// flagship net).  TMEM: accumulator columns (TN = 64: two accumulators, main and small terms) + 4 stages x (16 hi + 16 lo)
// columns = 256 -> two CTAs per SM.  Who paces the pipeline was measured with clock64 in every role:
// profiles/r02zb_mlp_tmem_role_timing.txt.
// Shared-memory traffic per weight byte: one bulk write + one read (2 B/B) instead of ~10 B/B; the tensor core reads only B.
#include "ngp_internal.h"

namespace tmm {

constexpr int TM = 128, KC = 16, STAGES = 4;
constexpr uint32_t SBO = 128;
constexpr uint32_t TMEM_COLS = 256;
constexpr int A_THREADS = 256;
// B side: the activations of a chunk take ~4 000 cycles from the first load to the published tile (L2 latency behind the weight
// stream; nothing may be in flight across the warp's fence.proxy.async).  Measured with clock64 in every role
// (profiles/README.md): four B warps deliver a chunk every ~1 000 cycles and the MMA thread waits for them 36 % of its time.
// With 64-environment tiles eight B warps hold eight chunks of activations in registers (the prefetch depth) and take turns on the
// four stages; 128-environment tiles need twice the registers per chunk and stay with four.
__host__ __device__ constexpr int b_warps(int TN) { return TN > 64 ? 4 : 8; }
__host__ __device__ constexpr int threads(int TN) { return A_THREADS + 32 * b_warps(TN) + 64; }      // + MMA warp + copy warp
constexpr uint32_t RAW_TILE = KC * TM * 4;                                                 // 8 KB: one packed 128 x 16 weight tile

// B stage layout.  TN = 128: two tiles (hi, lo) of 128 rows each.  TN = 64: hi and lo form ONE 128-row tile (rows 64..127 = lo), so
// that A_hi x [B_hi; B_lo] is a single N = 128 MMA.
__host__ __device__ constexpr bool folded(int TN) { return TN <= 64; }
__host__ __device__ constexpr uint32_t lbo(int TN) { return (folded(TN) ? 128u : (uint32_t)TN) * 16u + 16u; }     // +16 B: conflict-free stores
__host__ __device__ constexpr uint32_t tile_b(int TN) { return folded(TN) ? (64u / 8u) * SBO : (KC / 4) * lbo(TN); }        // byte offset of the lo part
__host__ __device__ constexpr uint32_t stage_b(int TN) { return folded(TN) ? (KC / 4) * lbo(TN) : 2 * (KC / 4) * lbo(TN); }
__host__ __device__ constexpr int raw_stages(int TN) { return TN > 64 ? 5 : 8; }           // two CTAs per SM must fit 227 KB
__host__ __device__ constexpr uint32_t smem_bytes(int TN) { return STAGES * stage_b(TN) + raw_stages(TN) * RAW_TILE + 512; }
__host__ __device__ constexpr uint32_t idesc(int TN)
{
    // cute::UMMA::InstrDescriptor: D=F32 (bit 4), A=B=TF32 (2 at bits 7, 10), both K-major, N>>3 at 17, M>>4 at 24
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(TN >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);
}

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t lbo_bytes)
{
    return (uint64_t)((smem_addr & 0x3FFFF) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(SBO >> 4) << 32) | (1ull << 46);
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count)); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    uint32_t ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    } while (!ok);
}
// D[tmem] (+)= A[tmem] * B[smem]
__device__ __forceinline__ void umma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t db, uint32_t id, uint32_t accumulate)
{
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, {%5, %5, %5, %5}, p;\n\t}"
                 ::"r"(tmem_d), "r"(tmem_a), "l"(db), "r"(id), "r"(accumulate), "r"(0u) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16])
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
                 ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
                   "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(bar), "r"(bytes) : "memory");
}
// 1-D bulk copy global -> shared (TMA engine), completion counted in bytes on an mbarrier
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t tf32_hi(float v) { return __float_as_uint(v) & 0xFFFFE000u; }

// packed layout of one genome's layer: tiles[ob][c][q][row][4]  (ob = 128-output block, c = 16-k chunk, q = quarter of the chunk)
// followed by bias[ob * 128 + row]; rows / k beyond the layer are zero
__host__ __device__ inline size_t packed_floats(int ni, int no)
{
    const size_t OB = (no + TM - 1) / TM, NC = (ni + KC - 1) / KC;
    return OB * NC * (size_t)(KC * TM) + OB * TM;
}

__global__ void __launch_bounds__(256) mlp_pack_layer_kernel(const float *__restrict__ genomes, size_t w_off, int G, int ni, int no, int bias,
                                                             float *__restrict__ packed, size_t per_genome, size_t layer_off)
{
    const int OB = (no + TM - 1) / TM, NC = (ni + KC - 1) / KC, K = ni + bias;
    const int g = blockIdx.y;
    const float *W = genomes + (size_t)g * G + w_off;
    float *dst = packed + (size_t)g * per_genome + layer_off;
    const long long units = (long long)OB * NC * 4 * TM;
    for (long long u = (long long)blockIdx.x * blockDim.x + threadIdx.x; u < units + (long long)OB * TM; u += (long long)gridDim.x * blockDim.x) {
        if (u < units) {
            const int row = (int)(u % TM), q = (int)((u / TM) % 4), c = (int)((u / (TM * 4)) % NC), ob = (int)(u / ((long long)TM * 4 * NC));
            const int o = ob * TM + row, k0 = c * KC + q * 4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (o < no) {
                const float *src = W + (size_t)o * K + k0;
                if (k0 + 0 < ni) v.x = __ldg(src + 0);
                if (k0 + 1 < ni) v.y = __ldg(src + 1);
                if (k0 + 2 < ni) v.z = __ldg(src + 2);
                if (k0 + 3 < ni) v.w = __ldg(src + 3);
            }
            reinterpret_cast<float4 *>(dst)[u] = v;
        } else {
            const int o = (int)(u - units);
            dst[units * 4 + o] = (bias && o < no) ? __ldg(W + (size_t)o * K + ni) : 0.f;
        }
    }
}

template <int TN>
__global__ void __launch_bounds__(threads(TN), 2)
mlp_layer_tmem_kernel(const float *__restrict__ packed, size_t per_genome, size_t layer_off, const float *__restrict__ in, int envs, int ni, int no,
                      float *__restrict__ out)
{
    constexpr uint32_t LBO = lbo(TN), TILE_B = tile_b(TN), STAGE_B = stage_b(TN), IDESC = idesc(TN);
    constexpr int B_WARPS = b_warps(TN), B_THREADS = 32 * B_WARPS;
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint32_t tmem_base_slot;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = blockIdx.z, e0 = blockIdx.y * TN, ob = blockIdx.x;
    const int NC = (ni + KC - 1) / KC;
    const uint32_t smem_base = smem_u32(smem);
    constexpr int NA = raw_stages(TN);
    const uint32_t raw_base = smem_base + STAGES * STAGE_B;               // NA raw weight tiles (bulk-copy destinations, 128-byte aligned)
    // barriers: a_full[s] (4 warps), b_full[s] (4 warps), free[s] (one commit), raw_full[r] (copy thread + bytes), raw_free[r] (4 warps), done
    const uint32_t bar_a = raw_base + NA * RAW_TILE, bar_b = bar_a + 8 * STAGES, bar_free = bar_b + 8 * STAGES, bar_done = bar_free + 8 * STAGES;
    const uint32_t bar_rfull = bar_done + 8, bar_rfree = bar_rfull + 8 * NA;
    const uint32_t bar_bnext = bar_rfree + 8 * NA;                        // [B_WARPS]: "the stage of your next chunk is free" (one commit)

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    const float *tiles = packed + (size_t)g * per_genome + layer_off + (size_t)ob * NC * (KC * TM);       // this CTA's NC contiguous 8 KB tiles
    constexpr int COPY_WARP = (A_THREADS + B_THREADS) / 32 + 1;
    if (warp == COPY_WARP && lane == 0) {
        // the copy thread sets the barriers up itself and has the first NA weight tiles under way while warp 0 allocates tensor
        // memory: the ~2 000 cycles a bulk copy takes to arrive are the first thing a CTA waits for
        for (int s = 0; s < STAGES; ++s) { mbar_init(bar_a + 8 * s, 4); mbar_init(bar_b + 8 * s, 1); mbar_init(bar_free + 8 * s, 1); }
        for (int r = 0; r < NA; ++r) { mbar_init(bar_rfull + 8 * r, 1); mbar_init(bar_rfree + 8 * r, 4); }
        for (int w = 0; w < B_WARPS; ++w) mbar_init(bar_bnext + 8 * w, 1);
        mbar_init(bar_done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        for (int c = 0; c < NA && c < NC; ++c) {
            mbar_expect_tx(bar_rfull + 8 * c, RAW_TILE);
            bulk_g2s(raw_base + c * RAW_TILE, tiles + (size_t)c * (KC * TM), RAW_TILE, bar_rfull + 8 * c);
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    constexpr bool TWO_ACC = TN <= 64;
    const uint32_t tmem_d = tmem_base_slot;                              // columns [0, TN): accumulator (TWO_ACC: of the hi*hi terms)
    const uint32_t tmem_d2 = TWO_ACC ? tmem_d + 64 : tmem_d;             // columns [64, 128): accumulator of the lo*hi + hi*lo terms
    const uint32_t tmem_a = tmem_d + 128;                                // columns [128, 256): 4 stages x (16 hi + 16 lo)

    if (warp == COPY_WARP) {
        // ------------------------------- copy warp: one bulk copy per chunk, NA chunks ahead -------------------------------
        if (lane == 0) {
            for (int c = NA; c < NC; ++c) {                              // the first NA are on their way (above)
                const int r = c % NA;
                mbar_wait(bar_rfree + 8 * r, ((c / NA) - 1) & 1);
                mbar_expect_tx(bar_rfull + 8 * r, RAW_TILE);
                bulk_g2s(raw_base + r * RAW_TILE, tiles + (size_t)c * (KC * TM), RAW_TILE, bar_rfull + 8 * r);
            }
        }
        __syncwarp();
    } else if (warp < A_THREADS / 32) {
        // ------------------------------- A producers: thread = output row = TMEM lane -------------------------------
        // Eight warps: warp w serves TMEM lane quadrant w & 3 (the lanes a warp may access) and the chunks of parity w >> 2.
        // The completion of a chunk's tcgen05.st is only awaited after the next chunk of this warp has been loaded and split.
        const int quad = warp & 3, par = warp >> 2, row = quad * 32 + lane;
        const uint32_t lane_addr = tmem_a + ((uint32_t)(quad * 32) << 16);
        int pending = -1;                                                // chunk whose stores have been issued but not yet published
        auto publish = [&](int c) {
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(bar_a + 8 * (c % STAGES));
                mbar_arrive(bar_rfree + 8 * (c % NA));                   // every lane's loads of the raw tile have been consumed by its stores
            }
        };
#pragma unroll 1
        for (int c = par; c < NC; c += 2) {
            const int r = c % NA, s = c % STAGES;
            mbar_wait(bar_rfull + 8 * r, (c / NA) & 1);
            const float4 *raw = reinterpret_cast<const float4 *>(smem + STAGES * STAGE_B + r * RAW_TILE) + row;       // [q][row] float4
            uint32_t hi[16], lo[16];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float4 v = raw[q * TM];
                hi[4 * q + 0] = tf32_hi(v.x); lo[4 * q + 0] = __float_as_uint(v.x - __uint_as_float(hi[4 * q + 0]));
                hi[4 * q + 1] = tf32_hi(v.y); lo[4 * q + 1] = __float_as_uint(v.y - __uint_as_float(hi[4 * q + 1]));
                hi[4 * q + 2] = tf32_hi(v.z); lo[4 * q + 2] = __float_as_uint(v.z - __uint_as_float(hi[4 * q + 2]));
                hi[4 * q + 3] = tf32_hi(v.w); lo[4 * q + 3] = __float_as_uint(v.w - __uint_as_float(hi[4 * q + 3]));
            }
            if (pending >= 0) publish(pending);
            if (c >= STAGES) {                                           // the MMAs that read this TMEM stage STAGES chunks ago are done
                mbar_wait(bar_free + 8 * s, ((c / STAGES) - 1) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            }
            tmem_st16(lane_addr + (uint32_t)(s * 32), hi);
            tmem_st16(lane_addr + (uint32_t)(s * 32 + 16), lo);
            pending = c;
        }
        if (pending >= 0) publish(pending);
    } else if (warp < (A_THREADS + B_THREADS) / 32) {
        // ------------------------------- B producers: activations -> hi/lo tiles in shared memory -------------------------------
        // A warp loads a whole chunk (TN rows x 64 bytes), waits for it, splits and stores it, and only then fences:
        // fence.proxy.async compiles to a MEMBAR that also waits for the thread's outstanding global loads, so nothing may be in
        // flight across it; the latency is hidden by the other warps' chunks instead.
        const int wb = warp - A_THREADS / 32;
        constexpr int UNITS = TN * (KC / 4) / 32;                        // 16-byte units per lane and chunk (8 or 16)
        const float *A = in + (size_t)g * envs * ni;
        // unit u = lane + 32 j: 8 consecutive lanes = 8 consecutive rows of one k-unit (conflict-free 128-byte store rows);
        // k-unit = (lane >> 3) & 3, row = (lane & 7) + 8 j
        const int cu = (lane >> 3) & 3, rl = lane & 7;
        // Warp wb takes chunks wb, wb + B_WARPS, ...; they all use stage sb = wb % STAGES, which it shares with the warps wb +- STAGES.
        // A parity wait is only sound for a waiter that sees every completion of its barrier in turn, so "stage free" is not
        // waited for on the stage's barrier (two warps share it and each would miss every other completion) but on the warp's
        // own: the MMA thread commits chunk c also to the barrier of the warp that fills this stage next, for chunk c + STAGES.
        const int sb = wb % STAGES;
        uint32_t waits = 0;
#pragma unroll 1
        for (int c = wb; c < NC; c += B_WARPS) {
            float4 v[UNITS];
#pragma unroll
            for (int j = 0; j < UNITS; ++j) {
                const int row = e0 + rl + 8 * j, k = c * KC + cu * 4;
                v[j] = (row < envs && k < ni) ? __ldg(reinterpret_cast<const float4 *>(A + (size_t)row * ni + k)) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            if (c >= STAGES) { mbar_wait(bar_bnext + 8 * wb, waits & 1u); ++waits; }
            uint8_t *stage = smem + sb * STAGE_B;
#pragma unroll
            for (int j = 0; j < UNITS; ++j) {
                const int r = rl + 8 * j;
                float4 h, l;
                h.x = __uint_as_float(tf32_hi(v[j].x)); l.x = v[j].x - h.x;
                h.y = __uint_as_float(tf32_hi(v[j].y)); l.y = v[j].y - h.y;
                h.z = __uint_as_float(tf32_hi(v[j].z)); l.z = v[j].z - h.z;
                h.w = __uint_as_float(tf32_hi(v[j].w)); l.w = v[j].w - h.w;
                uint8_t *dst = stage + cu * LBO + (r >> 3) * SBO + (r & 7) * 16;
                *reinterpret_cast<float4 *>(dst) = h;
                *reinterpret_cast<float4 *>(dst + TILE_B) = l;
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_b + 8 * sb);
        }
    } else if (warp == (A_THREADS + B_THREADS) / 32) {
        // ------------------------------- MMA warp -------------------------------
        // One thread issues everything, so its own instruction latency paces the tensor pipe (measured: 90 cycles per MMA with
        // the descriptors rebuilt each time): the stage loop is unrolled so that every descriptor and TMEM address is the base
        // plus a compile-time constant.
        if (lane == 0) {
            const uint64_t desc0 = make_desc(smem_base, LBO);            // + (byte offset >> 4): shared addresses stay below 2^18
            static_assert(B_WARPS % STAGES == 0, "the unrolled period covers whole turns of the stage ring");
#pragma unroll 1
            for (int c0 = 0; c0 < NC; c0 += B_WARPS) {
#pragma unroll
                for (int t = 0; t < B_WARPS; ++t) {
                    const int c = c0 + t, s = t % STAGES;
                    const uint32_t ph = (uint32_t)((c0 / STAGES + t / STAGES) & 1);
                    if (c < NC) {
                        mbar_wait(bar_a + 8 * s, ph);
                        mbar_wait(bar_b + 8 * s, ph);
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        const uint32_t a_hi = tmem_a + (uint32_t)(s * 32), a_lo = a_hi + 16;
#pragma unroll
                        for (int j = 0; j < KC / 8; ++j) {
                            const uint64_t d_hi = desc0 + (uint64_t)((s * STAGE_B + 2 * j * LBO) >> 4), d_lo = d_hi + (uint64_t)(TILE_B >> 4);
                            if (TWO_ACC) {
                                // folded: A_hi x [B_hi; B_lo] is one N = 128 MMA into columns [0, 128) (hi*hi | hi*lo); A_lo x B_hi goes
                                // on top of the hi*lo half; the epilogue adds the halves
                                umma_ts(tmem_d, a_hi + 8 * j, d_hi, idesc(128), (c | j) ? 1u : 0u);
                                umma_ts(tmem_d2, a_lo + 8 * j, d_hi, idesc(64), 1u);
                            } else {
                                umma_ts(tmem_d, a_lo + 8 * j, d_hi, IDESC, (c | j) ? 1u : 0u);       // small terms first
                                umma_ts(tmem_d, a_hi + 8 * j, d_lo, IDESC, 1u);
                                umma_ts(tmem_d, a_hi + 8 * j, d_hi, IDESC, 1u);
                            }
                        }
                        umma_commit(bar_free + 8 * s);
                        umma_commit(bar_bnext + 8 * ((t + STAGES) % B_WARPS));
                        if (c == NC - 1) umma_commit(bar_done);
                    }
                }
            }
        }
        __syncwarp();
    }
    // ------------------------------- epilogue: the A producers (warp w: lane quadrant w & 3, column half w >> 2) -------------------------------
    if (warp < A_THREADS / 32) {
        mbar_wait(bar_done, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int quad = warp & 3, colh = warp >> 2;
        const int o = ob * TM + quad * 32 + lane;
        const float b = packed[(size_t)g * per_genome + layer_off + (size_t)((no + TM - 1) / TM) * NC * (KC * TM) + o];
#pragma unroll 1
        for (int part = 0; part < TN / 64; ++part) {
            const int col0 = colh * (TN / 2) + part * 32;
            uint32_t v[32];
            const uint32_t taddr = tmem_d + ((uint32_t)(quad * 32) << 16) + (uint32_t)col0;
            asm volatile(
                "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
                  "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
                  "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
                  "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                : "r"(taddr) : "memory");
            if (!TWO_ACC) asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");       // two accumulators: both loads in flight, one wait
            if (TWO_ACC) {
                uint32_t w[32];
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                    "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                    "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                    : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7]), "=r"(w[8]), "=r"(w[9]),
                      "=r"(w[10]), "=r"(w[11]), "=r"(w[12]), "=r"(w[13]), "=r"(w[14]), "=r"(w[15]), "=r"(w[16]), "=r"(w[17]), "=r"(w[18]),
                      "=r"(w[19]), "=r"(w[20]), "=r"(w[21]), "=r"(w[22]), "=r"(w[23]), "=r"(w[24]), "=r"(w[25]), "=r"(w[26]), "=r"(w[27]),
                      "=r"(w[28]), "=r"(w[29]), "=r"(w[30]), "=r"(w[31])
                    : "r"(taddr + 64) : "memory");
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(w[j]));
            }
            if (o < no) {
                float *dst = out + ((size_t)g * envs + e0 + col0) * no + o;
                const int e_left = envs - (e0 + col0);
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    // fast exponential and reciprocal (ex2.approx, rcp.approx: a few ulp), far inside the 1e-5 bar
                    if (j < e_left) *dst = __fdividef(1.0f, 1.0f + __expf(-(__uint_as_float(v[j]) + b)));
                    dst += no;
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"(TMEM_COLS) : "memory");
}

}  // namespace tmm

// which layers of the handle's network run on the prepared (packed) path
static bool layer_is_packed(const pol::Shape &sh, int l)
{
    const int L = sh.n_layers - 1;              // hidden layers with a real contraction and 16-byte aligned activation rows
    return l != L - 1 && sh.nodes[l] >= 64 && sh.nodes[l + 1] >= 64 && sh.nodes[l] % 4 == 0;
}

// ngp_mlp_prepare: see include/ngp.h
extern "C" int ngp_mlp_prepare(ngp_handle *h, const float *genomes, int32_t n_genomes, void *stream)
{
    NGP_REQUIRE(h && genomes && n_genomes > 0, "ngp_mlp_prepare: bad arguments");
    NGP_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    const pol::Shape &sh = h->shape;
    const int bias = sh.bias ? 1 : 0, L = sh.n_layers - 1;
    size_t per_genome = 0;
    for (int l = 0; l < L; ++l)
        if (layer_is_packed(sh, l)) per_genome += tmm::packed_floats(sh.nodes[l], sh.nodes[l + 1]);
    h->prep_n = 0; h->prep_src = nullptr; h->prep_per_genome = per_genome;
    if (per_genome == 0) { h->prep_n = n_genomes; h->prep_src = genomes; return NGP_OK; }      // nothing to pack for this network
    NGP_CUDA(h->prep_packed.ensure(per_genome * (size_t)n_genomes));
    size_t w_off = 0, layer_off = 0;
    for (int l = 0; l < L; ++l) {
        const int ni = sh.nodes[l], no = sh.nodes[l + 1];
        if (layer_is_packed(sh, l)) {
            for (int g0 = 0; g0 < n_genomes; g0 += MLP_GENOME_SLICE) {
                dim3 grid(128, n_genomes - g0 < MLP_GENOME_SLICE ? n_genomes - g0 : MLP_GENOME_SLICE);
                tmm::mlp_pack_layer_kernel<<<grid, 256, 0, st>>>(genomes + (size_t)g0 * h->gene_size, w_off, h->gene_size, ni, no, bias,
                                                                 h->prep_packed.p + (size_t)g0 * per_genome, per_genome, layer_off);
                h->launches++;
                NGP_CUDA(cudaGetLastError());
            }
            layer_off += tmm::packed_floats(ni, no);
        }
        w_off += (size_t)(ni + bias) * no;
    }
    h->prep_n = n_genomes; h->prep_src = genomes;
    return NGP_OK;
}

// one prepared wide hidden layer (called by ngp_mlp_forward_prepared) for the prepared genomes [g0, g0 + n_genomes);
// NGP_ERR_UNSUPPORTED -> the caller uses the unprepared path
int ngp_mlp_layer_tmem(ngp_handle *h, int l, size_t g0, const float *in, int n_genomes, int envs, float *out, cudaStream_t st)
{
    const pol::Shape &sh = h->shape;
    if (!layer_is_packed(sh, l) || envs < 16 || !h->prep_packed.p) return NGP_ERR_UNSUPPORTED;
    size_t layer_off = 0;
    for (int i = 0; i < l; ++i)
        if (layer_is_packed(sh, i)) layer_off += tmm::packed_floats(sh.nodes[i], sh.nodes[i + 1]);
    const int ni = sh.nodes[l], no = sh.nodes[l + 1];
    const float *packed = h->prep_packed.p + g0 * h->prep_per_genome;
    if (!h->tmem_attr_set) {
        NGP_CUDA(cudaFuncSetAttribute(tmm::mlp_layer_tmem_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tmm::smem_bytes(64)));
        NGP_CUDA(cudaFuncSetAttribute(tmm::mlp_layer_tmem_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tmm::smem_bytes(128)));
        h->tmem_attr_set = 1;
    }
    if (envs > 64) {
        dim3 grid((no + tmm::TM - 1) / tmm::TM, (envs + 127) / 128, n_genomes);
        tmm::mlp_layer_tmem_kernel<128><<<grid, tmm::threads(128), tmm::smem_bytes(128), st>>>(packed, h->prep_per_genome, layer_off, in, envs, ni, no, out);
    } else {
        dim3 grid((no + tmm::TM - 1) / tmm::TM, 1, n_genomes);
        tmm::mlp_layer_tmem_kernel<64><<<grid, tmm::threads(64), tmm::smem_bytes(64), st>>>(packed, h->prep_per_genome, layer_off, in, envs, ni, no, out);
    }
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    return NGP_OK;
}
