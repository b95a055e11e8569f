// stepwise.cuh -- the per-environment state of the per-frame driver (ngp_stepwise.cu: wide ngp_evaluate;
// ngp_stepwise_lists.cu: ngp_play_matches_stepwise), kept in HBM between its kernels.
#pragma once
#include "ngp_internal.h"
#include "rollout.cuh"

namespace {

constexpr int CHECK_EVERY = 8;       // frames between two reads of the finished-environment count

struct StepEnv {
    a26::Snapshot snap;
    // perform_episode's locals (main.py:70-75)
    int32_t done, frame, timeout, total_frames, last_s1, last_s2;
    uint8_t have_last_score, have_last_ball, left_act, right_act;
    double last_ball[2];
    // what the frame kernel saw (consumed by the decide kernel)
    double loc[3][2];
    uint8_t valid[3], s1, s2, emu_error, pad_[2];
    // plan (main.py:33-58 / round-robin)
    int32_t state, left_kind, left_row, right_row;      // rows of the batched MLP input / action arrays (-1: no MLP on the left)
    double mult;
};

}  // namespace

// ngp_stepwise.cu: one frame of every running environment of `envs` (StepEnv[total]; step_frame_kernel, p.core picks the core); the
// inference rows of model-call frames go to x[right_row], and x_hof[left_row] (reference schedule) or x[left_row]
int ngp_step_frame(ngp_handle *h, const roll::RolloutParams &p, void *envs, int total, float *x, float *x_hof, cudaStream_t st);
