// rollout_kernel.cuh -- the fused rollout kernel template.  ngp_core.cu instantiates the flavours ngp_evaluate and
// ngp_play_matches run; ngp_record.cu instantiates their recording twins (REC = true, ngp_record_matches) in a translation
// unit of their own, so the parallel build compiles both sets side by side.
#pragma once
#include "game_state.cuh"

__device__ __forceinline__ void load_tables(a26::Tables &dst, const a26::Tables *__restrict__ src)
{
    const uint32_t *s = reinterpret_cast<const uint32_t *>(src);
    uint32_t *d = reinterpret_cast<uint32_t *>(&dst);
    for (unsigned i = threadIdx.x; i < sizeof(a26::Tables) / 4; i += blockDim.x) d[i] = s[i];
    __syncthreads();
}

// Fused rollout: one environment (= one game of one genome) per thread.  Lanes are persistent and
// pull the next environment from a global counter at frame boundaries, so a warp stays in
// scanline lock-step whatever episode each of its lanes is in.
// `rec` is read by the REC twins only (ngp_record_matches, ngp_play_matches_states): they store every frame below
// rec.max_record with roll::record_frame when there is a record, key the fall-back actions by rec.key, start matches from
// rec.states with roll::resume_state and write rec.capture with roll::capture_state.
template <int CORE, bool SYNC, int MAXT, bool REC = false>
__global__ void __launch_bounds__(MAXT, 1) rollout_kernel(roll::RolloutParams p, roll::RecordArgs rec)
{
    __shared__ a26::Tables T;
    extern __shared__ uint32_t ram_smem[];
    load_tables(T, p.tables);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    a26::Ram ram{&ram_smem[warp * 1024 + lane]};
    const int total = p.n * p.games;
    a26::Chip s; a26::CpuRegs r;
    roll::Episode ep;
    ep.env = -1;
    bool exhausted = false;
    unsigned long long my_frames = 0;
    int capture_at = -1;                // REC: capture the episode after this many env.steps
    for (;;) {
        if (ep.env < 0 && !exhausted) {
            int e = (int)atomicAdd(&p.counters[0], 1ull);
            if (e < total) {
                roll::episode_begin(ep, p, e, s, r, ram);
                if (REC && rec.start && rec.start[e] >= 0) roll::resume_state(rec, rec.start[e], ep, s, r, ram);
                if (REC && rec.capture_at) {
                    capture_at = rec.capture_at[e];
                    if (capture_at == ep.frame) roll::capture_state(rec, ep, s, r, ram);
                }
            } else exhausted = true;
        }
        const bool active = ep.env >= 0;
        // SYNC: the CTA walks through frames together (CTA-wide barriers inside the frame), so it also stops together
        if (SYNC) { if (!__syncthreads_or(active)) break; }
        else if (__all_sync(0xFFFFFFFFu, !active)) break;
        if (SYNC || active) {
            double reward;
            const bool done = roll::episode_frame<CORE, SYNC, REC>(ep, p, s, r, T, ram, &reward, active, &rec);
            if (active) my_frames++;
            if (REC && active && rec.record && ep.frame <= rec.max_record) roll::record_frame(rec, ep, s, ep.last_s1, ep.last_s2);
            if (REC && active && !done && ep.frame == capture_at) roll::capture_state(rec, ep, s, r, ram);
            if (done) {
                p.rewards[ep.env] = reward;
                p.frames[ep.env] = ep.frame;
                if (p.scores) { p.scores[2 * ep.env] = ep.last_s1; p.scores[2 * ep.env + 1] = ep.last_s2; }
                if (s.error) atomicAdd(&p.counters[2], 1ull);
                ep.env = -1;
            }
        }
    }
    // one atomic per warp for the frame counter
    for (int off = 16; off; off >>= 1) my_frames += __shfl_down_sync(0xFFFFFFFFu, my_frames, off);
    if (lane == 0 && my_frames) atomicAdd(&p.counters[1], my_frames);
}

using RolloutKernel = void (*)(roll::RolloutParams, roll::RecordArgs);

// The recording twin of flavour f (ngp_record.cu): 0 = <0,false,384>, 1 = <1,false,256>, 2 = <1,true,256>, 3 = <1,true,384>,
// 4 = <1,true,512>.
RolloutKernel rollout_record_kernel(int flavour);
