// mixed_kernels.cu — the two small kernels of the mixed-play ("MP") collection (SURVEY §8f row 3).
//
// Reference: XDPlayer.collect_mp_episode / next_mp_step (train/XD/xd_player.py:232-356), MixedAgent
// (train/partner_agents.py:151-244) and SharedReplayBuffer.diaginsert / partinsert
// (train/MAPPO/utils/shared_buffer.py:150-220).  There every env step draws a fresh per-world mask per
// seat (rand < 0.5 -> the partner convention acts), forces a growing block of worlds back to the policy
// being trained, and copies exactly the forced worlds of the turn scratch onto a diagonal (phase 1) or a
// row prefix (phase 2) of the [L+1, G, 2] buffer with a dozen strided torch copies per step.
//
// Here the env holds R replicas of the G = L-1 worlds.  Per env step:
//   mix_select_kernel  one thread per agent row: forced / drawn mask -> the action that is played;
//   mix_record_kernel  one warp per RECORDED agent row: observation (int8, in place), action, log-prob,
//                      value of the main policy, reward and done of this step -> buffer slot t.
// Both are HBM-bound byte movers: select touches 12 B per agent row, record 2*S*C + 20 B per recorded row.
#include <cuda_runtime.h>
#include <stdint.h>

#include "mixed_internal.h"
#include "mixed_schedule.h"

namespace ocb {

namespace {

constexpr int kSelThreads = 256;
constexpr int kRecWarps = 8;

__global__ void __launch_bounds__(kSelThreads) mix_select_kernel(const MixSelectParams p) {
    const int row = blockIdx.x * kSelThreads + threadIdx.x;
    if (row >= p.P * p.N) return;
    const int n = row % p.N;
    int act = p.a_main[row];
    if (!mix_forced_main(p.L, p.s, n % (p.L - 1)) && mix_draw_partner(p.mix_seed, (uint32_t)row, *p.step_counter))
        act = p.a_partner[row];
    p.act[row] = act;
}

__global__ void __launch_bounds__(kRecWarps * 32) mix_record_kernel(const MixRecordParams p) {
    const int lane = threadIdx.x & 31;
    const long long item = (long long)blockIdx.x * kRecWarps + (threadIdx.x >> 5);
    int seat, n, t;
    if (!mix_record_item(p.L, p.s, p.N, p.P, item, &seat, &n, &t)) return;
    const size_t src = (size_t)seat * p.N + n, dst = ((size_t)t * p.P + seat) * p.N + n;

    // observation the action was computed on (SC is a multiple of 4: C = 20)
    const int8_t* so = p.obs_cur + src * p.SC;
    int8_t* d_o = p.obs_buf + dst * p.SC;
    if ((p.SC & 15) == 0) {
        const uint4* s16 = reinterpret_cast<const uint4*>(so);
        uint4* d16 = reinterpret_cast<uint4*>(d_o);
        for (int c = lane; c < (p.SC >> 4); c += 32) __stcs(d16 + c, __ldcs(s16 + c));
    } else {
        const uint32_t* s4 = reinterpret_cast<const uint32_t*>(so);
        uint32_t* d4 = reinterpret_cast<uint32_t*>(d_o);
        for (int c = lane; c < (p.SC >> 2); c += 32) __stcs(d4 + c, __ldcs(s4 + c));
    }
    if (lane == 0) {
        p.actions[dst] = p.a_main[src];  // a recorded row is a forced row: the main policy acted
        if (p.logp) p.logp[dst] = p.logp_main[src];
        if (p.values) p.values[dst] = p.v_main[src];
        if (p.reward) p.reward[dst] = p.rew_cur[src];
        if (p.done && seat == 0) p.done[(size_t)t * p.N + n] = p.done_cur[n];
    }
}

__global__ void fill_i32_kernel(int32_t* a, int n0, int v0, int32_t* b, int n1, int v1) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n0) a[i] = v0;
    if (i < n1) b[i] = v1;
}

__global__ void fill_f32_kernel(float* a, size_t n, const float* v) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = *v;
}

}  // namespace

cudaError_t launch_fill_f32(float* a, size_t n, const float* v, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    fill_f32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(a, n, v);
    return cudaGetLastError();
}

cudaError_t launch_mix_select(const MixSelectParams& p, cudaStream_t stream) {
    const int rows = p.P * p.N;
    mix_select_kernel<<<(rows + kSelThreads - 1) / kSelThreads, kSelThreads, 0, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_mix_record(const MixRecordParams& p, cudaStream_t stream) {
    const int G = p.L - 1, R = p.N / G;
    const int cnt = p.s < p.L ? p.s : p.s - p.L;
    const long long items = (long long)R * cnt * p.P;
    if (items == 0) return cudaSuccess;
    mix_record_kernel<<<(unsigned)((items + kRecWarps - 1) / kRecWarps), kRecWarps * 32, 0, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_fill2_i32(int32_t* a, int n0, int v0, int32_t* b, int n1, int v1, cudaStream_t stream) {
    const int n = n0 > n1 ? n0 : n1;
    if (n == 0) return cudaSuccess;
    fill_i32_kernel<<<(n + 255) / 256, 256, 0, stream>>>(a, n0, v0, b, n1, v1);
    return cudaGetLastError();
}

}  // namespace ocb
