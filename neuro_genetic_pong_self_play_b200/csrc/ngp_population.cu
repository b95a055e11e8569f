// ngp_population.cu -- population-level pieces around the fused evaluation: the hall of fame (DEAP tools.HallOfFame as the
// reference uses it, ga.py:78, main.py:165-168, utils.py:90-101), toolbox.mate / toolbox.mutate as separate callables
// (ga.py:89-92) and the device side of the per-generation multi-GPU exchange (ga.py:83's gather of every fitness on the master).
#include <string.h>

#include "ngp_internal.h"
#include "ga_streams.cuh"

// =================================================================================================
// hall of fame
// =================================================================================================
// 64-bit FNV-1a over the gene bit patterns (-0.0 == 0.0 and NaN != NaN under Python's ==; both are folded so that equal
// genomes always hash equal: -0.0 hashes as 0.0, and the full compare below uses float ==).
__global__ void genome_hash_kernel(const float *__restrict__ genomes, int rows, int G, uint64_t *__restrict__ hash)
{
    const int row = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (row >= rows) return;
    // 32 interleaved FNV streams (lane l hashes genes l, l+32, ...), combined in lane order
    uint64_t hsh = 1469598103934665603ull ^ (uint64_t)lane;
    for (int g = lane; g < G; g += 32) {
        float v = genomes[(size_t)row * G + g];
        uint32_t b = v == 0.0f ? 0u : __float_as_uint(v);
        hsh = (hsh ^ b) * 1099511628211ull;
    }
    uint64_t acc = 0;
    for (int l = 0; l < 32; ++l) {
        const uint64_t o = __shfl_sync(0xFFFFFFFFu, hsh, l);
        acc = (acc ^ o) * 1099511628211ull + 0x9E3779B97F4A7C15ull;
    }
    if (lane == 0) hash[row] = acc;
}

// Sequential HallOfFame.update in one CTA.  Members are referred to by *virtual row*: v < maxsize = row v of the old hall,
// v >= maxsize = individual v - maxsize of the population.  order[0..cur) is the hall, best first.
struct HofArgs {
    const float *hof_genomes; const double *hof_fitness; const uint64_t *hof_hash;
    const float *genomes; const double *fitness; const uint64_t *hash;
    int n_hof, maxsize, n, G;
    int32_t *order;            // [maxsize + 1]
    int32_t *out_count;        // [1]
};

__device__ __forceinline__ double hof_fit(const HofArgs &a, int v) { return v < a.maxsize ? a.hof_fitness[v] : a.fitness[v - a.maxsize]; }
__device__ __forceinline__ uint64_t hof_hash_of(const HofArgs &a, int v) { return v < a.maxsize ? a.hof_hash[v] : a.hash[v - a.maxsize]; }
__device__ __forceinline__ const float *hof_row(const HofArgs &a, int v)
{
    return v < a.maxsize ? a.hof_genomes + (size_t)v * a.G : a.genomes + (size_t)(v - a.maxsize) * a.G;
}

__global__ void __launch_bounds__(1024) hof_update_kernel(HofArgs a)
{
    __shared__ int s_cur, s_flag, s_pos;
    const int tid = threadIdx.x, nt = blockDim.x;
    for (int i = tid; i < a.n_hof; i += nt) a.order[i] = i;
    if (tid == 0) s_cur = a.n_hof;
    __syncthreads();
    for (int c = 0; c < a.n; ++c) {
        const int cur = s_cur;
        const double f = a.fitness[c];
        // DEAP: `if len(self) == 0 and maxsize != 0: insert` / `if ind.fitness > self[-1].fitness or len(self) < maxsize`
        if (cur > 0 && !(cur < a.maxsize || f > hof_fit(a, a.order[cur - 1]))) continue;       // uniform across the CTA
        if (tid == 0) { s_flag = 0; s_pos = 0; }
        __syncthreads();
        // similar to any member?  (operator.eq on the gene lists)
        const uint64_t hc = a.hash[c];
        const float *gc = a.genomes + (size_t)c * a.G;
        int greater = 0;
        for (int i = tid; i < cur; i += nt) {
            const int v = a.order[i];
            if (hof_fit(a, v) > f) greater++;
            if (hof_hash_of(a, v) == hc) {
                const float *gm = hof_row(a, v);
                bool same = true;
                for (int g = 0; g < a.G && same; ++g) same = gm[g] == gc[g];
                if (same) s_flag = 1;
            }
        }
        if (greater) atomicAdd(&s_pos, greater);
        __syncthreads();
        if (s_flag) { __syncthreads(); continue; }
        int len = cur;
        if (len >= a.maxsize) len--;                       // self.remove(-1): the worst leaves
        const int pos = s_pos < len ? s_pos : len;         // number of members strictly better: the newcomer goes before equals
        // shift order[pos..len) one to the right, back to front in chunks so that no element is overwritten before it is read
        for (int hi = len; hi > pos; hi -= nt) {
            const int i = hi - 1 - tid;
            int v = 0;
            if (i >= pos) v = a.order[i];
            __syncthreads();
            if (i >= pos) a.order[i + 1] = v;
            __syncthreads();
        }
        if (tid == 0) { a.order[pos] = a.maxsize + c; s_cur = len + 1; }
        __syncthreads();
    }
    if (tid == 0) *a.out_count = s_cur;
}

__global__ void hof_gather_kernel(HofArgs a, const int32_t *__restrict__ count, float *__restrict__ out_genomes, double *__restrict__ out_fitness,
                                  uint64_t *__restrict__ out_hash)
{
    const int m = blockIdx.x;
    if (m >= *count) return;
    const int v = a.order[m];
    const float *src = hof_row(a, v);
    for (int g = threadIdx.x; g < a.G; g += blockDim.x) out_genomes[(size_t)m * a.G + g] = src[g];
    if (threadIdx.x == 0) { out_fitness[m] = hof_fit(a, v); out_hash[m] = hof_hash_of(a, v); }
}

extern "C" int ngp_hof_update(ngp_handle *h, float *hof_genomes, double *hof_fitness, int32_t *n_hof, int32_t maxsize,
                              const float *genomes, const double *fitness, int32_t n, void *stream)
{
    NGP_REQUIRE(h && n_hof && maxsize >= 0 && n >= 0, "ngp_hof_update: bad arguments");
    NGP_REQUIRE(*n_hof >= 0 && *n_hof <= maxsize, "ngp_hof_update: n_hof out of range");
    if (maxsize == 0 || n == 0) return NGP_OK;
    NGP_REQUIRE(hof_genomes && hof_fitness && genomes && fitness, "ngp_hof_update: null pointer");
    NGP_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int G = h->gene_size;
    NGP_CUDA(h->hof_hash_old.ensure(maxsize));
    NGP_CUDA(h->hof_hash_new.ensure(n));
    NGP_CUDA(h->hof_order.ensure((size_t)maxsize + 2));
    NGP_CUDA(h->hof_tmp_genomes.ensure((size_t)maxsize * G));
    NGP_CUDA(h->hof_tmp_fitness.ensure((size_t)maxsize * 2));          // fitness, then the hashes as 64-bit words
    if (*n_hof > 0) {
        genome_hash_kernel<<<(unsigned)(((long long)*n_hof * 32 + 255) / 256), 256, 0, st>>>(hof_genomes, *n_hof, G, h->hof_hash_old.p);
        h->launches++;
    }
    genome_hash_kernel<<<(unsigned)(((long long)n * 32 + 255) / 256), 256, 0, st>>>(genomes, n, G, h->hof_hash_new.p);
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    HofArgs a;
    a.hof_genomes = hof_genomes; a.hof_fitness = hof_fitness; a.hof_hash = h->hof_hash_old.p;
    a.genomes = genomes; a.fitness = fitness; a.hash = h->hof_hash_new.p;
    a.n_hof = *n_hof; a.maxsize = maxsize; a.n = n; a.G = G;
    a.order = h->hof_order.p; a.out_count = h->hof_order.p + maxsize + 1;
    hof_update_kernel<<<1, 1024, 0, st>>>(a);
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    double *tmp_fit = h->hof_tmp_fitness.p;
    uint64_t *tmp_hash = reinterpret_cast<uint64_t *>(tmp_fit + maxsize);
    hof_gather_kernel<<<maxsize, 128, 0, st>>>(a, a.out_count, h->hof_tmp_genomes.p, tmp_fit, tmp_hash);
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    NGP_CUDA(cudaMemcpyAsync(h->h_counters.p + 3, a.out_count, 4, cudaMemcpyDeviceToHost, st));
    NGP_CUDA(cudaStreamSynchronize(st));
    const int count = (int)(h->h_counters.p[3] & 0xFFFFFFFFull);
    NGP_CUDA(cudaMemcpyAsync(hof_genomes, h->hof_tmp_genomes.p, (size_t)count * G * 4, cudaMemcpyDeviceToDevice, st));
    NGP_CUDA(cudaMemcpyAsync(hof_fitness, tmp_fit, (size_t)count * 8, cudaMemcpyDeviceToDevice, st));
    NGP_CUDA(cudaStreamSynchronize(st));
    *n_hof = count;
    return NGP_OK;
}

// =================================================================================================
// toolbox.mate / toolbox.mutate on single individuals (ga.py:89-92)
// =================================================================================================
__global__ void mate_kernel(float *__restrict__ x0, float *__restrict__ x1, int G, const float *__restrict__ u_in, uint32_t pair, uint64_t seed,
                            uint64_t generation, float alpha)
{
    const int gene = blockIdx.x * blockDim.x + threadIdx.x;
    if (gene >= G) return;
    float u;
    if (u_in) u = u_in[gene];
    else {
        uint32_t o[4];
        pol::philox4x32(pair, (uint32_t)(gene >> 2), (uint32_t)generation, STREAM_CXU, (uint32_t)seed, (uint32_t)(seed >> 32), o);
        u = u01(o[gene & 3]);
    }
    float a = x0[gene], b = x1[gene];
    blend_gene(alpha, u, a, b);
    x0[gene] = a; x1[gene] = b;
}

__global__ void mutate_kernel(float *__restrict__ x, int G, const float *__restrict__ u_in, const float *__restrict__ z_in, uint32_t slot, uint64_t seed,
                              uint64_t generation, float mu, float sigma, float indpb)
{
    const int gene = blockIdx.x * blockDim.x + threadIdx.x;
    if (gene >= G) return;
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32), gen = (uint32_t)generation;
    float u, z;
    if (u_in) u = u_in[gene];
    else {
        uint32_t o[4];
        pol::philox4x32(slot, (uint32_t)(gene >> 2), gen, STREAM_MUTU, k0, k1, o);
        u = u01(o[gene & 3]);
    }
    z = z_in ? z_in[gene] : mut_normal(slot, (uint32_t)gene, gen, k0, k1);
    if (u < indpb) x[gene] = __fadd_rn(x[gene], __fadd_rn(mu, __fmul_rn(sigma, z)));
}

extern "C" int ngp_mate(ngp_handle *h, float *ind1, float *ind2, const float *u, int32_t pair, uint64_t seed, uint64_t generation,
                        void *stream)
{
    NGP_REQUIRE(h && ind1 && ind2 && ind1 != ind2, "ngp_mate: bad arguments");
    NGP_CUDA(cudaSetDevice(h->device));
    const int G = h->gene_size;
    mate_kernel<<<(G + 255) / 256, 256, 0, (cudaStream_t)stream>>>(ind1, ind2, G, u, (uint32_t)pair, seed, generation, h->cfg.cx_alpha);
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    return NGP_OK;
}

extern "C" int ngp_mutate(ngp_handle *h, float *ind, const float *u, const float *z, int32_t slot, uint64_t seed, uint64_t generation,
                          void *stream)
{
    NGP_REQUIRE(h && ind, "ngp_mutate: bad arguments");
    NGP_CUDA(cudaSetDevice(h->device));
    const int G = h->gene_size;
    mutate_kernel<<<(G + 255) / 256, 256, 0, (cudaStream_t)stream>>>(ind, G, u, z, (uint32_t)slot, seed, generation, h->cfg.mut_mu,
                                                                     h->cfg.mut_sigma, h->cfg.mut_indpb);
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    return NGP_OK;
}

// =================================================================================================
// multi-GPU exchange record (one per rank, all ranks the same size):
//   [ n_local i32 | k_local i32 | 8 bytes pad | fitness f64[n_max] | elite_fitness f64[k_max] | elite_genomes f32[k_max][G] ]
// padded to a multiple of 16 bytes.  Shards may differ by one genome when the population does not divide by the world size.
// =================================================================================================
extern "C" int64_t ngp_exchange_bytes(const ngp_handle *h, int32_t n_max, int32_t k_max)
{
    if (!h || n_max < 0 || k_max < 0) return -1;
    const int64_t raw = 16 + (int64_t)n_max * 8 + (int64_t)k_max * 8 + (int64_t)k_max * h->gene_size * 4;
    return (raw + 15) & ~(int64_t)15;
}

// rank by counting: position of individual i among the shard sorted by fitness descending, ties by index.
// One warp per individual; the k best copy themselves into the record.
__global__ void __launch_bounds__(256) pack_elites_kernel(const float *__restrict__ genomes, const double *__restrict__ fitness, int n, int k, int G,
                                                          int32_t *__restrict__ header, double *__restrict__ rec_fitness,
                                                          double *__restrict__ rec_elite_fitness, float *__restrict__ rec_elite_genomes)
{
    const int i = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (i >= n) return;
    if (i == 0 && lane == 0) { header[0] = n; header[1] = k; header[2] = 0; header[3] = 0; }
    const double f = fitness[i];
    int better = 0;
    for (int j = lane; j < n; j += 32) {
        const double o = fitness[j];
        better += (o > f || (o == f && j < i)) ? 1 : 0;
    }
    for (int off = 16; off; off >>= 1) better += __shfl_xor_sync(0xFFFFFFFFu, better, off);
    if (lane == 0) rec_fitness[i] = f;
    if (better < k) {
        if (lane == 0) rec_elite_fitness[better] = f;
        for (int g = lane; g < G; g += 32) rec_elite_genomes[(size_t)better * G + g] = genomes[(size_t)i * G + g];
    }
}

extern "C" int ngp_pack_elites(ngp_handle *h, const float *genomes, const double *fitness, int32_t n, int32_t k, int32_t n_max,
                               int32_t k_max, void *out, void *stream)
{
    NGP_REQUIRE(h && genomes && fitness && out && n > 0 && k >= 0 && k <= n && n <= n_max && k <= k_max, "ngp_pack_elites: bad arguments");
    NGP_REQUIRE(((uintptr_t)out & 15) == 0, "ngp_pack_elites: record must be 16-byte aligned");
    NGP_CUDA(cudaSetDevice(h->device));
    int32_t *hdr = reinterpret_cast<int32_t *>(out);
    double *rf = reinterpret_cast<double *>(hdr + 4);
    double *ref = rf + n_max;
    float *reg = reinterpret_cast<float *>(ref + k_max);
    pack_elites_kernel<<<(unsigned)(((long long)n * 32 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(genomes, fitness, n, k, h->gene_size, hdr, rf, ref,
                                                                                               reg);
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    return NGP_OK;
}

// Gathered records -> compact global arrays in rank order: fitness_all f64[sum n_r], elites (genomes f32[sum k_r][G],
// fitness f64[sum k_r]); each rank's elites best first.
__global__ void unpack_elites_kernel(const uint8_t *__restrict__ gathered, long long rec_bytes, int world, int n_max, int k_max, int G,
                                     double *__restrict__ fitness_all, float *__restrict__ elite_genomes, double *__restrict__ elite_fitness)
{
    const int r = blockIdx.y;
    const uint8_t *rec = gathered + (size_t)r * rec_bytes;
    const int32_t *hdr = reinterpret_cast<const int32_t *>(rec);
    const int n = hdr[0], k = hdr[1];
    long long n_off = 0, k_off = 0;
    for (int q = 0; q < r; ++q) {
        const int32_t *hq = reinterpret_cast<const int32_t *>(gathered + (size_t)q * rec_bytes);
        n_off += hq[0]; k_off += hq[1];
    }
    const double *rf = reinterpret_cast<const double *>(hdr + 4);
    const double *ref = rf + n_max;
    const float *reg = reinterpret_cast<const float *>(ref + k_max);
    const long long total = (long long)n + k + (long long)k * G;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        if (t < n) { if (fitness_all) fitness_all[n_off + t] = rf[t]; }
        else if (t < n + k) { if (elite_fitness) elite_fitness[k_off + (t - n)] = ref[t - n]; }
        else if (elite_genomes) elite_genomes[k_off * G + (t - n - k)] = reg[t - n - k];
    }
}

extern "C" int ngp_unpack_elites(ngp_handle *h, const void *gathered, int32_t world, int32_t n_max, int32_t k_max, double *fitness_all,
                                 float *elite_genomes, double *elite_fitness, void *stream)
{
    NGP_REQUIRE(h && gathered && world > 0 && n_max > 0 && k_max >= 0, "ngp_unpack_elites: bad arguments");
    NGP_CUDA(cudaSetDevice(h->device));
    const long long rec = ngp_exchange_bytes(h, n_max, k_max);
    const long long total = (long long)n_max + k_max + (long long)k_max * h->gene_size;
    long long bx = (total + 255) / 256;
    if (bx > 64) bx = 64;
    unpack_elites_kernel<<<dim3((unsigned)bx, (unsigned)world), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const uint8_t *>(gathered), rec, world,
                                                                                              n_max, k_max, h->gene_size, fitness_all, elite_genomes,
                                                                                              elite_fitness);
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    return NGP_OK;
}
