// mixed_internal.h — launch interface of mixed_kernels.cu used by ocb_api.cu (not part of the C ABI)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace ocb {

struct MixSelectParams {
    const int32_t* a_main;     // [P][N] actions of the policy being trained
    const int32_t* a_partner;  // [P][N] actions of the partner convention
    int32_t* act;              // [P][N] the action that is played
    const unsigned long long* step_counter;  // device: the env's global step count (counter of the mask stream)
    unsigned long long mix_seed;
    int P, N, L, s;
};

struct MixRecordParams {
    const int8_t* obs_cur;     // [P][N][SC] observation the actions of this step were computed on
    const int32_t* a_main;     // [P][N]
    const float* logp_main;    // [P][N]
    const float* v_main;       // [P][N]
    const int32_t* rew_cur;    // [P][N] reward of this step
    const int32_t* done_cur;   // [N]
    int8_t* obs_buf;           // [L+1][P][N][SC]
    int32_t* actions;          // [L][P][N]
    float* logp;               // [L][P][N] or nullptr
    float* values;             // [L+1][P][N] or nullptr
    int32_t* reward;           // [L][P][N] or nullptr
    int32_t* done;             // [L][N] or nullptr
    int P, N, SC, L, s;
};

cudaError_t launch_mix_select(const MixSelectParams& p, cudaStream_t stream);
cudaError_t launch_mix_record(const MixRecordParams& p, cudaStream_t stream);
// a[0 .. n) = *v, read when the kernel runs (v is a DEVICE address)
cudaError_t launch_fill_f32(float* a, size_t n, const float* v, cudaStream_t stream);
cudaError_t launch_fill2_i32(int32_t* a, int n0, int v0, int32_t* b, int n1, int v1, cudaStream_t stream);

}  // namespace ocb
