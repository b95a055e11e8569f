// ngp_internal.h -- handle layout and helpers shared by the translation units of libngp.so
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <utility>
#include <vector>

#include "../../include/ngp.h"
#include "a26_core.cuh"
#include "policy.cuh"

// Memory owned by a handle: a grow-only array of T in device memory, or pinned host memory with HOST.  ensure() keeps the
// allocation while `count` elements fit; otherwise it frees before allocating (the peak footprint is the new size alone) and
// after a refused allocation holds nothing.
template <typename T, bool HOST = false>
struct Buffer {
    T *p = nullptr;
    size_t cap = 0;               // elements

    Buffer() = default;
    Buffer(const Buffer &) = delete;
    Buffer &operator=(const Buffer &) = delete;
    ~Buffer() { release(); }

    cudaError_t ensure(size_t count)
    {
        if (count <= cap) return cudaSuccess;
        release();
        const cudaError_t e = HOST ? cudaMallocHost((void **)&p, count * sizeof(T)) : cudaMalloc((void **)&p, count * sizeof(T));
        if (e != cudaSuccess) p = nullptr;
        else cap = count;
        return e;
    }

private:
    void release()
    {
        if (p) { if (HOST) cudaFreeHost(p); else cudaFree(p); }
        p = nullptr; cap = 0;
    }
};
template <typename T> using HostBuffer = Buffer<T, true>;

// Created value-initialised (every scalar zero) by ngp_create; the device must be current when it is destroyed.
struct ngp_handle {
    ngp_config cfg;
    int device;
    int sm_count;
    int gene_size;
    pol::Shape shape;
    int rom_translated;           // the ROM is the cartridge the statically translated core was generated from
    uint64_t cart_hash;           // fnv1a64 of the cartridge image: the header of every ngp_game_state of this handle
    // device tables
    Buffer<a26::Tables> d_tables;         // rom + decode + colour-match weights
    Buffer<uint32_t> d_needed;            // paddle charge -> cycles table [4097]
    Buffer<uint32_t> d_palette;           // NTSC palette [128]
    Buffer<a26::Snapshot> d_start;        // [2]: 'Start' (1P) and 'Start.2P'
    // stepwise (explicit action) environments
    Buffer<a26::Snapshot> d_envs;
    Buffer<uint8_t> d_fb;                 // palette-index frames [n_envs][210][160]
    int n_envs;
    int env_players;              // gym-retro `players` of the state the stepwise environments were reset to (1 for 'Start')
    // fused evaluation scratch
    Buffer<double> d_rewards;
    Buffer<int32_t> d_frames;
    Buffer<unsigned long long> d_counters;    // [0] next env, [1] frames, [2] emulator errors, [3] bad list entries / finished
                                              // environments, [8, 14) ngp_play_matches_stepwise's chunk counts
    // host staging (pinned) for the *_host entry points
    HostBuffer<float> h_genomes; HostBuffer<double> h_fitness; Buffer<float> d_genomes_stage; Buffer<double> d_fitness_stage;
    Buffer<float> d_hof_stage; Buffer<double> d_hof_fit_stage;
    HostBuffer<unsigned long long> h_counters;
    uint64_t launches;
    // per-handle scratch of the operator entry points (nothing here is shared between handles)
    Buffer<float> mlp_a, mlp_b; Buffer<double> mlp_z;                                         // ngp_mlp_forward activations
    Buffer<int32_t> d_parent;                                                                 // ngp_ga_step selection winners
    Buffer<unsigned long long> rank_keys; Buffer<int32_t> rank_idx;                           // fitness ranking of the order-statistics tournament
    Buffer<uint64_t> hof_hash_old, hof_hash_new; Buffer<int32_t> hof_order; Buffer<float> hof_tmp_genomes; Buffer<double> hof_tmp_fitness;   // ngp_hof_update
    // ngp_evaluate for nets wider than the fused rollout (ngp_stepwise.cu): per-environment state (bytes of StepEnv), MLP
    // input rows, actions, gathered hall-of-fame opponents
    Buffer<uint8_t> step_envs; Buffer<float> step_x; Buffer<uint8_t> step_act; Buffer<float> step_opp;
    // ngp_play_matches_stepwise's chunk layout: per genome rows | chunks | first chunk, the genome of every chunk, CUB scan scratch
    Buffer<int32_t> list_genome; Buffer<int32_t> list_chunk; Buffer<uint8_t> list_scan_tmp;
    // ngp_mlp_prepare: packed wide layers of the prepared genome set (ngp_mlp_tmem.cu)
    Buffer<float> prep_packed; size_t prep_per_genome; const float *prep_src; int prep_n; int tmem_attr_set;
    int fs_per_sm;                                                          // resident find_stuff CTAs per SM
    int tf32_attr_set;                                                      // dynamic shared memory opt-in done
    // ngp_set_option (tuning experiments; 0 = automatic)
    int opt_rollout_block, opt_rollout_nosync, opt_rollout_lean, opt_rollout_blocks_per_sm, opt_mlp_no_tf32, opt_select_os_min_t;
    // profiling of the rollout kernel
    int profile_on;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof_events;
    int prof_used;
    // match sessions open on this handle (ngp_session.cu); ngp_destroy ends them
    std::vector<ngp_session *> sessions;

    ~ngp_handle()
    {
        for (auto &e : prof_events) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
    }
};

// The wide MLP layer kernels take the genome from grid.y or grid.z, which CUDA caps at 65 535: ngp_mlp_forward and
// ngp_mlp_prepare run larger genome sets in slices of at most this many genomes.
constexpr int MLP_GENOME_SLICE = 65535;

// ngp_ops.cu: the wide MLP over x[n_chunks][T][6] with the prepared weights of genome chunk_genome[c] for chunk c
int ngp_mlp_forward_chunks(ngp_handle *h, const float *genomes, const int32_t *chunk_genome, const float *x, int n_chunks, int T,
                           uint8_t *act, cudaStream_t st);

void ngp_set_error(const char *fmt, ...);
#define NGP_CUDA(expr)                                                                           \
    do {                                                                                         \
        cudaError_t e_ = (expr);                                                                 \
        if (e_ != cudaSuccess) {                                                                 \
            ngp_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
            cudaGetLastError();   /* reported once: the next call's launch check must not see it */ \
            return NGP_ERR_CUDA;                                                                 \
        }                                                                                        \
    } while (0)
#define NGP_REQUIRE(cond, msg)                                      \
    do {                                                            \
        if (!(cond)) { ngp_set_error("%s", msg); return NGP_ERR_INVALID; } \
    } while (0)
