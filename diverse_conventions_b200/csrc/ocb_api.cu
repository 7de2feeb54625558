// ocb_api.cu — the C ABI of include/ocb.h (Overcooked part).
// Plain CUDA runtime; no torch, no C++ types in any signature.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include <new>

#include "api_common.h"
#include "oc_core.cuh"
#include "oc_kernels.h"
#include "oc_tables.h"
#include "policy_internal.h"
#include "mixed_internal.h"
#include "ocb.h"

using namespace ocb;

namespace ocb {
thread_local char g_err[512] = "";
int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
}  // namespace ocb

struct ocb_env {
    int device;
    int N, P, S, C, SC, L;
    uint64_t seed;
    uint64_t step_count;   // host mirror of *d_step_counter
    bool count_stale;      // launches were captured into a CUDA graph: replays advance only the device counter
    uint32_t world0;
    int lanes_per_world;  // G of the fused K-step launches
    int step_lanes;       // G of single-step / observe launches (load + full rebuild dominate there)
    int use_tma;
    int sm_count;
    Tables h_tables;
    // device
    Tables* d_tables;
    uint8_t* d_tmpl;
    uint32_t* d_players;
    uint16_t* d_objs;
    int32_t* d_timestep;
    int32_t* d_cur_return;
    long long* d_ret_sum;
    int32_t* d_episodes;
    unsigned long long* d_step_counter;  // device mirror of step_count
    // scratch for the host-buffer entry points
    // double-buffered device staging + streams of the host-buffer pipeline (ocb_step_host / ocb_step_host_async)
    int32_t* d_h_actions[2];
    int8_t* d_h_obs[2];
    int32_t* d_h_rew[2];
    int32_t* d_h_done[2];
    cudaStream_t own_stream;   // H2D of the actions + the step kernel
    cudaStream_t copy_stream;  // D2H of reward / done / observations
    cudaEvent_t ev_kernel[2], ev_done[2], ev_order;
    uint64_t host_issued, host_completed;
};

static int build_tables_or_fail(const ocb_config* cfg, Tables* tb, uint8_t* tmpl) {
    char msg[400];
    const int rc = build_tables(cfg, tb, tmpl, msg, sizeof(msg));
    return rc == OCB_OK ? OCB_OK : fail(rc, "%s", msg);
}

// lanes per world: few worlds -> more (redundant) lanes so that every SM scheduler still has
// several warps to hide the latency of the sequential transition; many worlds -> fewer lanes,
// less redundant issue.  From tools/sweep.py on B200 over world counts 1,024..32,768 and the 400 / 500 / 900-byte
// layouts (profiles/r1_sweep_layouts.jsonl): below 8,192 worlds G=4 wins everywhere; from 16,384 worlds G=1 for the
// small planes (0.99-1.03 of the HBM peak, 128 CTAs) and G=2 for planes >= 800 bytes (0.94); in between 4 resp. 2.
static int default_lanes(int N, int SC) {
    const bool big = SC >= 800;
    if (N < 8192) return 4;
    if (N < 16384) return big ? 2 : 4;
    return big ? 2 : 1;
}
// ... unless the role-split kernel serves the env (two players, at most two pots): below 16,384 worlds a launch is bound
// by the latency of a world's step, and the split kernel's step is the transition alone.  tools/gpu_split_defaults.sh
// (profiles/r2g_split_defaults.jsonl), ms per 100 steps, split against the best one-warp shape: cramped_room 1,024 / 4,096
// / 8,192 / 12,288 worlds 0.105 / 0.106 / 0.113 / 0.174 against 0.154 / 0.157 / 0.158 / 0.174; coordination_ring 0.109 /
// 0.109 / 0.148 / 0.217 against 0.162 / 0.166 / 0.166 / 0.215; asymmetric_advantages (900-byte planes) 0.142 / 0.134
// against 0.172 / 0.173 up to 4,096 worlds and a tie (0.257 / 0.253) at 8,192.  From 16,384 worlds on the one-warp shapes
// stay (cramped_room 0.199 against 0.227-0.235).
static bool split_is_default(int N, int SC) { return SC >= 800 ? N <= 4096 : N < 16384; }

// lanes per world of single-step / observe launches.  The planes of a tile are rebuilt by one bulk copy per view
// (tile_fill_begin), so what is left per world is the state load and the sequential transition: from a few thousand worlds
// on two lanes per world win (tools/step_single.py on B200: 262,144 worlds of coordination_ring 113 us at G = 2 against
// 144 / 160 / 190 at 4 / 8 / 1; 32,768 worlds 21.1 against 23.3 / 27.4 / 23.4; 8,192 worlds of cramped_room 10.3 against
// 10.9 / 11.4 / 13.0); below that the launch is latency-bound (10 us) and more lanes hide the transition better.
static int default_step_lanes(int N) { return N >= 4096 ? 2 : 8; }

// lanes_per_world == kLanesSplit selects the role-split K-step kernel (oc_rollout_split_kernel: a transition warp and GE
// encoder warps per 32 worlds).  It serves two players and at most two pots and only launches that write observations;
// every other launch of such an env falls back to the one-warp-does-all kernel with `fallback_lanes`.
constexpr int kLanesSplit = 16;
static bool split_supported(const ocb_env* e) { return e->P == 2 && e->h_tables.n_pots <= 2; }
static int fallback_lanes(const ocb_env* e) { return default_lanes(e->N, e->SC); }
static int default_lanes_env(const ocb_env* e) {
    if (split_supported(e) && split_is_default(e->N, e->SC) && rollout_split_smem_bytes(e->S, e->C, 1, 32) <= 200 * 1024)
        return kLanesSplit;
    return default_lanes(e->N, e->SC);
}
// Worlds per tile of a K-step launch: full tiles (32 / G worlds per warp; 32 per group of the role-split kernel).
// Narrower tiles would spread a launch more evenly over the SMs (16,384 worlds in 32-world groups are four CTAs on some
// SMs and three on others) and the kernels take any width (`RolloutParams::tile_worlds`), but measured (tools/gpu_tile.sh,
// profiles/r2g_tile_sweep.jsonl) they do not pay: widths whose planes are not a whole number of 128-byte lines lose 15 %
// (a tile starting inside a line shares it with a neighbour that another SM writes at another time), 8-world groups halve
// the throughput, and 16-world groups gain 3 % at 16,384 worlds while losing 1 % at 8,192.  OCB_TILE_WORLDS narrows the
// tiles for the parity tests of that code path and for experiments.
static int tile_worlds_for(int full) {
    if (const char* ev = getenv("OCB_TILE_WORLDS")) {
        const int v = atoi(ev);
        if (v >= 1) return v < full ? v : full;
    }
    return full;
}

static void split_shape(const ocb_env* e, int* GE, int* TW) {
    *GE = e->SC >= 800 ? 4 : 2, *TW = 1;  // encoder lanes per world (tools/gpu_split_defaults.sh)
    if (const char* ev = getenv("OCB_SPLIT_GE")) {  // tuning experiments only
        const int v = atoi(ev);
        if (v == 2 || v == 4) *GE = v;
    }
    (void)e;
}

static int pick_launch_shape(const ocb_env* e, int G, int* warps, size_t* smem) {
    // 4 warps per CTA measured best on B200 even when that leaves some SMs without a CTA
    // (16,384 worlds, G=1: 128 CTAs; 1- and 2-warp CTAs were 6% / 3% slower, profiles/README.md)
    int wmax = 4;
    if (const char* ev = getenv("OCB_WARPS_PER_CTA")) {  // tuning experiments only
        const int v = atoi(ev);
        if (v >= 1 && v <= 4) wmax = v;
    }
    for (int w = wmax; w >= 1; --w) {
        const size_t b = rollout_smem_bytes(e->P, e->S, e->C, G, w);
        if (b <= 200 * 1024) {
            *warps = w, *smem = b;
            return OCB_OK;
        }
    }
    return fail(OCB_ERR_UNSUPPORTED, "layout needs more shared memory than one SM has (S=%d, P=%d, lanes_per_world=%d)",
                e->S, e->P, G);
}

// ------------------------------------------------------------------ misc
extern "C" int ocb_abi_version(void) { return OCB_ABI_VERSION; }
extern "C" const char* ocb_last_error(void) { return g_err; }
extern "C" int ocb_device_count(void) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(OCB_ERR_NO_DEVICE, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    }
    return n;
}

// ------------------------------------------------------------------ life-cycle
extern "C" int ocb_destroy(ocb_env* e) {
    if (e == nullptr) return OCB_OK;
    DeviceGuard guard(e->device);
    CaptureRelaxed relaxed;  // safe while another stream is being captured
    cudaFree(e->d_tables);
    cudaFree(e->d_tmpl);
    cudaFree(e->d_players);
    cudaFree(e->d_objs);
    cudaFree(e->d_timestep);
    cudaFree(e->d_cur_return);
    cudaFree(e->d_ret_sum);
    cudaFree(e->d_episodes);
    cudaFree(e->d_step_counter);
    for (int b = 0; b < 2; ++b) {
        cudaFree(e->d_h_actions[b]);
        cudaFree(e->d_h_obs[b]);
        cudaFree(e->d_h_rew[b]);
        cudaFree(e->d_h_done[b]);
        if (e->ev_kernel[b]) cudaEventDestroy(e->ev_kernel[b]);
        if (e->ev_done[b]) cudaEventDestroy(e->ev_done[b]);
    }
    if (e->ev_order) cudaEventDestroy(e->ev_order);
    if (e->own_stream) cudaStreamDestroy(e->own_stream);
    if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
    delete e;
    return OCB_OK;
}

extern "C" int ocb_create(const ocb_config* cfg, int device, uint32_t num_worlds, uint64_t seed, ocb_env** out) {
    if (out == nullptr) return fail(OCB_ERR_INVALID_ARG, "out is NULL");
    *out = nullptr;
    if (num_worlds < 1 || num_worlds > (1u << 30)) return fail(OCB_ERR_INVALID_ARG, "num_worlds out of range");
    const int ndev = ocb_device_count();
    if (ndev <= 0) return fail(OCB_ERR_NO_DEVICE, "no CUDA device available (this library has no CPU path)");
    if (device < 0 || device >= ndev) return fail(OCB_ERR_INVALID_ARG, "device %d not in 0..%d", device, ndev - 1);

    ocb_env* e = new (std::nothrow) ocb_env();
    if (e == nullptr) return fail(OCB_ERR_INVALID_ARG, "out of host memory");
    memset(e, 0, sizeof(*e));
    uint8_t tmpl[OCB_MAX_CELLS * (5 * OCB_MAX_PLAYERS + 10)];
    int rc = build_tables_or_fail(cfg, &e->h_tables, tmpl);
    if (rc != OCB_OK) {
        delete e;
        return rc;
    }
    e->device = device;
    e->N = (int)num_worlds;
    e->P = e->h_tables.P, e->S = e->h_tables.S, e->C = e->h_tables.C, e->SC = e->h_tables.SC;
    e->L = 1 + 6 * e->P + 4 * e->S;
    e->seed = seed;
    e->lanes_per_world = default_lanes_env(e);
    e->step_lanes = default_step_lanes(e->N);
    e->use_tma = 1;
    if (cudaDeviceGetAttribute(&e->sm_count, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || e->sm_count < 1) {
        cudaGetLastError();
        e->sm_count = 148;
    }

    DeviceGuard guard(device);
    const size_t N = num_worlds;
#define OCB_TRY(call)                                                                         \
    do {                                                                                      \
        cudaError_t err__ = (call);                                                           \
        if (err__ != cudaSuccess) {                                                           \
            rc = fail(OCB_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(err__));              \
            cudaGetLastError();                                                               \
            ocb_destroy(e);                                                                   \
            return rc;                                                                        \
        }                                                                                     \
    } while (0)
    OCB_TRY(cudaMalloc(&e->d_tables, sizeof(Tables)));
    OCB_TRY(cudaMalloc(&e->d_tmpl, align16((size_t)32 * e->SC)));
    OCB_TRY(cudaMalloc(&e->d_players, sizeof(uint32_t) * e->P * N));
    OCB_TRY(cudaMalloc(&e->d_objs, sizeof(uint16_t) * e->S * N));
    OCB_TRY(cudaMalloc(&e->d_timestep, sizeof(int32_t) * N));
    OCB_TRY(cudaMalloc(&e->d_cur_return, sizeof(int32_t) * N));
    OCB_TRY(cudaMalloc(&e->d_ret_sum, sizeof(long long) * N));
    OCB_TRY(cudaMalloc(&e->d_episodes, sizeof(int32_t) * N));
    OCB_TRY(cudaMalloc(&e->d_step_counter, sizeof(unsigned long long)));
    OCB_TRY(cudaMemset(e->d_step_counter, 0, sizeof(unsigned long long)));
    OCB_TRY(cudaMemcpy(e->d_tables, &e->h_tables, sizeof(Tables), cudaMemcpyHostToDevice));
    {   // 32 copies: one bulk copy rebuilds the planes of a whole warp tile (oc_kernels.cu: tile_fill_begin)
        std::vector<uint8_t> tile((size_t)32 * e->SC);
        for (int r = 0; r < 32; ++r) memcpy(tile.data() + (size_t)r * e->SC, tmpl, (size_t)e->SC);
        OCB_TRY(cudaMemcpy(e->d_tmpl, tile.data(), tile.size(), cudaMemcpyHostToDevice));
    }
    OCB_TRY(cudaMemset(e->d_ret_sum, 0, sizeof(long long) * N));
    OCB_TRY(cudaMemset(e->d_episodes, 0, sizeof(int32_t) * N));
    OCB_TRY(launch_reset(e->d_tables, e->d_players, e->d_objs, e->d_timestep, e->d_cur_return, e->N,
                         e->S > e->P ? e->S : e->P, 0));
    OCB_TRY(cudaDeviceSynchronize());
#undef OCB_TRY
    int warps;
    size_t smem;
    rc = pick_launch_shape(e, e->lanes_per_world == kLanesSplit ? fallback_lanes(e) : e->lanes_per_world, &warps, &smem);
    if (rc != OCB_OK) {
        ocb_destroy(e);
        return rc;
    }
    *out = e;
    return OCB_OK;
}

extern "C" int ocb_num_worlds(const ocb_env* e) { return e ? e->N : fail(OCB_ERR_INVALID_ARG, "env is NULL"); }
extern "C" int ocb_num_players(const ocb_env* e) { return e ? e->P : fail(OCB_ERR_INVALID_ARG, "env is NULL"); }
extern "C" int ocb_obs_channels(const ocb_env* e) { return e ? e->C : fail(OCB_ERR_INVALID_ARG, "env is NULL"); }
extern "C" int ocb_obs_bytes_per_agent(const ocb_env* e) { return e ? e->SC : fail(OCB_ERR_INVALID_ARG, "env is NULL"); }
extern "C" int ocb_state_ints_per_world(const ocb_env* e) { return e ? e->L : fail(OCB_ERR_INVALID_ARG, "env is NULL"); }
// host mirror <- device counter after graph replays (synchronises the device once; no-op otherwise)
static int resync_step_count(ocb_env* e) {
    if (!e->count_stale) return OCB_OK;
    DeviceGuard guard(e->device);
    unsigned long long v = 0;
    cudaError_t err = cudaDeviceSynchronize();
    if (err == cudaSuccess) err = cudaMemcpy(&v, e->d_step_counter, sizeof(v), cudaMemcpyDeviceToHost);
    if (err != cudaSuccess) {
        cudaGetLastError();
        return fail(OCB_ERR_CUDA, "step counter resync: %s", cudaGetErrorString(err));
    }
    e->step_count = v;
    e->count_stale = false;
    return OCB_OK;
}
static bool stream_capturing(void* stream) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing((cudaStream_t)stream, &cs) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return cs != cudaStreamCaptureStatusNone;
}

extern "C" uint64_t ocb_step_count(const ocb_env* e) {
    if (e == nullptr) return 0;
    if (e->count_stale) resync_step_count(const_cast<ocb_env*>(e));  // the device counter is the source of truth
    return e->step_count;
}

extern "C" int ocb_set_tuning(ocb_env* e, int lanes_per_world, int use_tma) {
    if (e == nullptr) return fail(OCB_ERR_INVALID_ARG, "env is NULL");
    const bool explicit_lanes = lanes_per_world != 0;
    if (lanes_per_world == 0) lanes_per_world = default_lanes_env(e);
    if (lanes_per_world != 1 && lanes_per_world != 2 && lanes_per_world != 4 && lanes_per_world != 8 &&
        lanes_per_world != kLanesSplit)
        return fail(OCB_ERR_INVALID_ARG, "lanes_per_world must be 1, 2, 4, 8 or 16 (role-split kernel)");
    if (lanes_per_world == kLanesSplit) {
        if (!split_supported(e))
            return fail(OCB_ERR_UNSUPPORTED, "the role-split kernel serves 2 players and at most 2 pots (P=%d, pots=%d)", e->P,
                        e->h_tables.n_pots);
        if (rollout_split_smem_bytes(e->S, e->C, 1, 32) > 200 * 1024)
            return fail(OCB_ERR_UNSUPPORTED, "layout needs more shared memory than one SM has (S=%d, role-split kernel)", e->S);
    }
    int warps;
    size_t smem;
    int rc = pick_launch_shape(e, lanes_per_world == kLanesSplit ? fallback_lanes(e) : lanes_per_world, &warps, &smem);
    if (rc != OCB_OK) return rc;
    e->lanes_per_world = lanes_per_world;
    e->step_lanes = (explicit_lanes && lanes_per_world != kLanesSplit) ? lanes_per_world : default_step_lanes(e->N);
    e->use_tma = use_tma ? 1 : 0;
    return OCB_OK;
}

extern "C" int ocb_get_tuning(const ocb_env* e, int* lanes_per_world, int* use_tma, int* warps_per_cta) {
    if (e == nullptr) return fail(OCB_ERR_INVALID_ARG, "env is NULL");
    int warps = 0;
    size_t smem = 0;
    int rc = pick_launch_shape(e, e->lanes_per_world == kLanesSplit ? fallback_lanes(e) : e->lanes_per_world, &warps, &smem);
    if (rc != OCB_OK) return rc;
    if (e->lanes_per_world == kLanesSplit) {  // warps of one CTA of the split kernel
        int GE, TW;
        split_shape(e, &GE, &TW);
        warps = TW * (1 + GE);
    }
    if (lanes_per_world) *lanes_per_world = e->lanes_per_world;
    if (use_tma) *use_tma = e->use_tma;
    if (warps_per_cta) *warps_per_cta = warps;
    return OCB_OK;
}

// world offset used by the action RNG (multi-GPU shards use rank*N); not in the
// reference API, exported for the sharded rollout driver
extern "C" int ocb_set_world_offset(ocb_env* e, uint32_t world0) {
    if (e == nullptr) return fail(OCB_ERR_INVALID_ARG, "env is NULL");
    e->world0 = world0;
    return OCB_OK;
}

// ------------------------------------------------------------------ hot path
static RolloutParams base_params(ocb_env* e) {
    RolloutParams p;
    memset(&p, 0, sizeof(p));
    p.tables = e->d_tables, p.tmpl = e->d_tmpl;
    p.players = e->d_players, p.objs = e->d_objs, p.timestep = e->d_timestep;
    p.cur_return = e->d_cur_return, p.ret_sum = e->d_ret_sum, p.episodes = e->d_episodes;
    p.N = e->N, p.seed = e->seed, p.world0 = e->world0, p.step0 = e->step_count;
    p.use_tma = e->use_tma;
    p.step_counter = e->d_step_counter;
    return p;
}

static int run_rollout(ocb_env* e, int K, const void* actions, int act_dtype, int8_t* obs, int32_t* rew, int32_t* done,
                       uint8_t* actions_out, bool observe_only, void* stream) {
    if (e == nullptr) return fail(OCB_ERR_INVALID_ARG, "env is NULL");
    if (K < 0) return fail(OCB_ERR_INVALID_ARG, "K must be >= 0");
    if (act_dtype < OCB_ACT_I32 || act_dtype > OCB_ACT_U8) return fail(OCB_ERR_INVALID_ARG, "unknown action dtype %d", act_dtype);
    DeviceGuard guard(e->device);
    // The first step of the launch keys the action RNG.  Normally it comes from the host mirror; a launch that is being
    // captured into a CUDA graph reads it from the device counter instead (every replay continues the stream) and the
    // counter is advanced by a launch of its own; the host mirror is resynchronised at the next uncaptured call.
    const bool capturing = !observe_only && stream_capturing(stream);
    if (!capturing && !observe_only && e->count_stale) {
        const int src = resync_step_count(e);
        if (src != OCB_OK) return src;
    }
    RolloutParams p = base_params(e);
    if (capturing) p.step0_dev = e->d_step_counter, p.step_counter = nullptr;
    p.K = K, p.actions = actions, p.act_dtype = act_dtype, p.actions_out = actions_out;
    p.obs = obs, p.rew = rew, p.done = done;
    int warps;
    size_t smem;
    // single steps are dominated by the state load and the full plane rebuild: spread each world over
    // more lanes there (tools/step_latency.py); fused launches use the throughput-tuned shape
    int G = (observe_only || K <= 2) ? e->step_lanes : e->lanes_per_world;
    const bool split = G == kLanesSplit && obs != nullptr;
    if (G == kLanesSplit) G = fallback_lanes(e);
    cudaError_t err;
    if (split) {
        int GE, TW;
        split_shape(e, &GE, &TW);
        p.tile_worlds = tile_worlds_for(32);
        err = launch_rollout_split(p, GE, TW, rollout_split_smem_bytes(e->S, e->C, TW, p.tile_worlds), (cudaStream_t)stream);
    } else {
        int rc = pick_launch_shape(e, G, &warps, &smem);
        if (rc != OCB_OK) return rc;
        if (!observe_only && K > 2) p.tile_worlds = tile_worlds_for(32 / G);
        err = launch_rollout(p, e->P, G, warps, smem, observe_only, (cudaStream_t)stream);
    }
    if (err != cudaSuccess) {
        cudaGetLastError();
        return fail(OCB_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(err));
    }
    if (capturing) {
        err = launch_counter_add(e->d_step_counter, (unsigned long long)K, (cudaStream_t)stream);
        if (err != cudaSuccess) {
            cudaGetLastError();
            return fail(OCB_ERR_CUDA, "counter launch failed: %s", cudaGetErrorString(err));
        }
        e->count_stale = true;  // the capture itself executes nothing
    } else if (!observe_only) {
        e->step_count += (uint64_t)K;
    }
    return OCB_OK;
}

extern "C" int ocb_observe(ocb_env* e, int8_t* obs, void* stream) {
    if (obs == nullptr) return fail(OCB_ERR_INVALID_ARG, "obs is NULL");
    return run_rollout(e, 0, nullptr, OCB_ACT_I32, obs, nullptr, nullptr, nullptr, true, stream);
}

extern "C" int ocb_reset(ocb_env* e, int8_t* obs, void* stream) {
    if (e == nullptr) return fail(OCB_ERR_INVALID_ARG, "env is NULL");
    {
        DeviceGuard guard(e->device);
        cudaError_t err = launch_reset(e->d_tables, e->d_players, e->d_objs, e->d_timestep, e->d_cur_return, e->N,
                                       e->S > e->P ? e->S : e->P, (cudaStream_t)stream);
        if (err != cudaSuccess) {
            cudaGetLastError();
            return fail(OCB_ERR_CUDA, "reset launch failed: %s", cudaGetErrorString(err));
        }
    }
    return obs ? ocb_observe(e, obs, stream) : OCB_OK;
}

extern "C" int ocb_step_ex(ocb_env* e, const void* actions, int act_dtype, int8_t* obs, int32_t* reward, int32_t* done,
                           void* stream) {
    if (actions == nullptr) return fail(OCB_ERR_INVALID_ARG, "actions is NULL");
    return run_rollout(e, 1, actions, act_dtype, obs, reward, done, nullptr, false, stream);
}

extern "C" int ocb_step(ocb_env* e, const int32_t* actions, int8_t* obs, int32_t* reward, int32_t* done, void* stream) {
    return ocb_step_ex(e, actions, OCB_ACT_I32, obs, reward, done, stream);
}

extern "C" int ocb_rollout_actions(ocb_env* e, int K, const void* actions, int act_dtype, int8_t* obs_slab,
                                   int32_t* reward, int32_t* done, void* stream) {
    if (actions == nullptr) return fail(OCB_ERR_INVALID_ARG, "actions is NULL");
    return run_rollout(e, K, actions, act_dtype, obs_slab, reward, done, nullptr, false, stream);
}

extern "C" int ocb_rollout_random(ocb_env* e, int K, int8_t* obs_slab, int32_t* reward, int32_t* done,
                                  uint8_t* actions_out, void* stream) {
    return run_rollout(e, K, nullptr, OCB_ACT_I32, obs_slab, reward, done, actions_out, false, stream);
}

extern "C" int ocb_step_host_wait(ocb_env* e);

// Host-buffer stepping as a two-deep pipeline on the env's own (non-blocking) streams: step t's observation copy
// (13 MB at config 3, PCIe-bound) overlaps the H2D + kernel of step t + 1 when the caller already has the next actions.
//   own_stream : [wait ev_done[slot]] H2D actions -> step kernel -> record ev_kernel[slot]
//   copy_stream: wait ev_kernel[slot] -> D2H reward, done (small, first) -> D2H observations -> record ev_done[slot]
// Ordering with work the caller issued earlier on blocking streams (torch's default stream) is kept through an event on
// the legacy default stream, as the previous implementation on stream 0 did implicitly.
extern "C" int ocb_step_host_async(ocb_env* e, const int32_t* h_actions, int8_t* h_obs, int32_t* h_reward, int32_t* h_done) {
    if (e == nullptr) return fail(OCB_ERR_INVALID_ARG, "env is NULL");
    if (h_actions == nullptr) return fail(OCB_ERR_INVALID_ARG, "actions is NULL");
    DeviceGuard guard(e->device);
    const size_t N = e->N, P = e->P;
#define OCB_TRY(call)                                                            \
    do {                                                                         \
        cudaError_t err__ = (call);                                              \
        if (err__ != cudaSuccess) {                                              \
            cudaGetLastError();                                                  \
            return fail(OCB_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(err__)); \
        }                                                                        \
    } while (0)
    if (e->own_stream == nullptr) OCB_TRY(cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking));
    if (e->copy_stream == nullptr) OCB_TRY(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
    if (e->ev_order == nullptr) OCB_TRY(cudaEventCreateWithFlags(&e->ev_order, cudaEventDisableTiming));
    if (e->host_issued - e->host_completed >= 2) {  // pipeline full: retire the oldest step first
        const int rc = ocb_step_host_wait(e);
        if (rc < 0) return rc;
    }
    const int b = (int)(e->host_issued & 1);
    if (e->ev_kernel[b] == nullptr) OCB_TRY(cudaEventCreateWithFlags(&e->ev_kernel[b], cudaEventDisableTiming));
    if (e->ev_done[b] == nullptr) OCB_TRY(cudaEventCreateWithFlags(&e->ev_done[b], cudaEventDisableTiming));
    if (e->d_h_actions[b] == nullptr) OCB_TRY(cudaMalloc(&e->d_h_actions[b], sizeof(int32_t) * P * N));
    if (h_obs && e->d_h_obs[b] == nullptr) OCB_TRY(cudaMalloc(&e->d_h_obs[b], P * N * (size_t)e->SC));
    if (h_reward && e->d_h_rew[b] == nullptr) OCB_TRY(cudaMalloc(&e->d_h_rew[b], sizeof(int32_t) * P * N));
    if (h_done && e->d_h_done[b] == nullptr) OCB_TRY(cudaMalloc(&e->d_h_done[b], sizeof(int32_t) * N));
    cudaStream_t sc = e->own_stream, sd = e->copy_stream;
    if (e->host_issued == e->host_completed) {  // pipeline empty: order after the caller's earlier (blocking-stream) work
        OCB_TRY(cudaEventRecord(e->ev_order, 0));
        OCB_TRY(cudaStreamWaitEvent(sc, e->ev_order, 0));
    }
    OCB_TRY(cudaStreamWaitEvent(sc, e->ev_done[b], 0));  // the staging buffers of this slot have been copied out
    OCB_TRY(cudaMemcpyAsync(e->d_h_actions[b], h_actions, sizeof(int32_t) * P * N, cudaMemcpyHostToDevice, sc));
    int rc = ocb_step(e, e->d_h_actions[b], h_obs ? e->d_h_obs[b] : nullptr, h_reward ? e->d_h_rew[b] : nullptr,
                      h_done ? e->d_h_done[b] : nullptr, sc);
    if (rc != OCB_OK) return rc;
    OCB_TRY(cudaEventRecord(e->ev_kernel[b], sc));
    OCB_TRY(cudaStreamWaitEvent(sd, e->ev_kernel[b], 0));
    if (h_reward) OCB_TRY(cudaMemcpyAsync(h_reward, e->d_h_rew[b], sizeof(int32_t) * P * N, cudaMemcpyDeviceToHost, sd));
    if (h_done) OCB_TRY(cudaMemcpyAsync(h_done, e->d_h_done[b], sizeof(int32_t) * N, cudaMemcpyDeviceToHost, sd));
    if (h_obs) OCB_TRY(cudaMemcpyAsync(h_obs, e->d_h_obs[b], P * N * (size_t)e->SC, cudaMemcpyDeviceToHost, sd));
    OCB_TRY(cudaEventRecord(e->ev_done[b], sd));
    e->host_issued += 1;
    return OCB_OK;
}

// blocks until the OLDEST step enqueued by ocb_step_host_async has delivered its host buffers; returns the number of
// steps still in flight (0 or 1), or a negative error code
extern "C" int ocb_step_host_wait(ocb_env* e) {
    if (e == nullptr) return fail(OCB_ERR_INVALID_ARG, "env is NULL");
    if (e->host_issued == e->host_completed) return 0;
    DeviceGuard guard(e->device);
    OCB_TRY(cudaEventSynchronize(e->ev_done[e->host_completed & 1]));
    e->host_completed += 1;
    return (int)(e->host_issued - e->host_completed);
}

extern "C" int ocb_step_host(ocb_env* e, const int32_t* h_actions, int8_t* h_obs, int32_t* h_reward, int32_t* h_done) {
    int rc = ocb_step_host_async(e, h_actions, h_obs, h_reward, h_done);
    if (rc != OCB_OK) return rc;
    do {
        rc = ocb_step_host_wait(e);
    } while (rc > 0);
    return rc < 0 ? rc : OCB_OK;
}
#undef OCB_TRY

// ------------------------------------------------------------------ state I/O
extern "C" int ocb_get_state(ocb_env* e, int32_t* h_state, size_t n_ints) {
    if (e == nullptr || h_state == nullptr) return fail(OCB_ERR_INVALID_ARG, "NULL argument");
    const size_t need = (size_t)e->N * e->L;
    if (n_ints != need) return fail(OCB_ERR_INVALID_ARG, "state buffer has %zu ints, expected %zu", n_ints, need);
    DeviceGuard guard(e->device);
    int32_t* d = nullptr;
    cudaError_t err = cudaMalloc(&d, need * sizeof(int32_t));
    if (err == cudaSuccess) err = cudaDeviceSynchronize();
    if (err == cudaSuccess) err = launch_export_state(e->d_tables, e->d_players, e->d_objs, e->d_timestep, d, e->N, 0);
    if (err == cudaSuccess) err = cudaMemcpy(h_state, d, need * sizeof(int32_t), cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (err != cudaSuccess) {
        cudaGetLastError();
        return fail(OCB_ERR_CUDA, "get_state: %s", cudaGetErrorString(err));
    }
    return OCB_OK;
}

extern "C" int ocb_set_state(ocb_env* e, const int32_t* h_state, size_t n_ints) {
    if (e == nullptr || h_state == nullptr) return fail(OCB_ERR_INVALID_ARG, "NULL argument");
    const size_t need = (size_t)e->N * e->L;
    if (n_ints != need) return fail(OCB_ERR_INVALID_ARG, "state buffer has %zu ints, expected %zu", n_ints, need);
    DeviceGuard guard(e->device);
    int32_t* d = nullptr;
    int* d_bad = nullptr;
    int bad = 0;
    // validate into scratch copies first so that a rejected state leaves the env untouched
    uint32_t* t_players = nullptr;
    uint16_t* t_objs = nullptr;
    int32_t *t_time = nullptr, *t_ret = nullptr;
    const size_t N = e->N;
    cudaError_t err = cudaDeviceSynchronize();
    if (err == cudaSuccess) err = cudaMalloc(&d, need * sizeof(int32_t));
    if (err == cudaSuccess) err = cudaMalloc(&d_bad, sizeof(int));
    if (err == cudaSuccess) err = cudaMalloc(&t_players, sizeof(uint32_t) * e->P * N);
    if (err == cudaSuccess) err = cudaMalloc(&t_objs, sizeof(uint16_t) * e->S * N);
    if (err == cudaSuccess) err = cudaMalloc(&t_time, sizeof(int32_t) * N);
    if (err == cudaSuccess) err = cudaMalloc(&t_ret, sizeof(int32_t) * N);
    if (err == cudaSuccess) err = cudaMemset(d_bad, 0, sizeof(int));
    if (err == cudaSuccess) err = cudaMemcpy(d, h_state, need * sizeof(int32_t), cudaMemcpyHostToDevice);
    if (err == cudaSuccess) err = launch_import_state(e->d_tables, d, t_players, t_objs, t_time, t_ret, e->N, d_bad, 0);
    if (err == cudaSuccess) err = cudaMemcpy(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost);
    if (err == cudaSuccess && bad == 0) {
        err = cudaMemcpy(e->d_players, t_players, sizeof(uint32_t) * e->P * N, cudaMemcpyDeviceToDevice);
        if (err == cudaSuccess) err = cudaMemcpy(e->d_objs, t_objs, sizeof(uint16_t) * e->S * N, cudaMemcpyDeviceToDevice);
        if (err == cudaSuccess) err = cudaMemcpy(e->d_timestep, t_time, sizeof(int32_t) * N, cudaMemcpyDeviceToDevice);
        if (err == cudaSuccess) err = cudaMemcpy(e->d_cur_return, t_ret, sizeof(int32_t) * N, cudaMemcpyDeviceToDevice);
    }
    cudaFree(d), cudaFree(d_bad), cudaFree(t_players), cudaFree(t_objs), cudaFree(t_time), cudaFree(t_ret);
    if (err != cudaSuccess) {
        cudaGetLastError();
        return fail(OCB_ERR_CUDA, "set_state: %s", cudaGetErrorString(err));
    }
    if (bad) return fail(OCB_ERR_BAD_STATE, "%d world(s) hold a state the simulator cannot represent", bad);
    return OCB_OK;
}

extern "C" int ocb_read_episode_stats(ocb_env* e, int64_t* return_sum, int32_t* episodes, void* stream) {
    if (e == nullptr) return fail(OCB_ERR_INVALID_ARG, "env is NULL");
    DeviceGuard guard(e->device);
    cudaError_t err = cudaSuccess;
    if (return_sum)
        err = cudaMemcpyAsync(return_sum, e->d_ret_sum, sizeof(long long) * (size_t)e->N, cudaMemcpyDeviceToDevice,
                              (cudaStream_t)stream);
    if (err == cudaSuccess && episodes)
        err = cudaMemcpyAsync(episodes, e->d_episodes, sizeof(int32_t) * (size_t)e->N, cudaMemcpyDeviceToDevice,
                              (cudaStream_t)stream);
    if (err != cudaSuccess) {
        cudaGetLastError();
        return fail(OCB_ERR_CUDA, "read_episode_stats: %s", cudaGetErrorString(err));
    }
    return OCB_OK;
}

extern "C" int ocb_clear_episode_stats(ocb_env* e, void* stream) {
    if (e == nullptr) return fail(OCB_ERR_INVALID_ARG, "env is NULL");
    DeviceGuard guard(e->device);
    cudaError_t err = cudaMemsetAsync(e->d_ret_sum, 0, sizeof(long long) * (size_t)e->N, (cudaStream_t)stream);
    if (err == cudaSuccess) err = cudaMemsetAsync(e->d_episodes, 0, sizeof(int32_t) * (size_t)e->N, (cudaStream_t)stream);
    if (err == cudaSuccess) err = cudaMemsetAsync(e->d_cur_return, 0, sizeof(int32_t) * (size_t)e->N, (cudaStream_t)stream);
    if (err != cudaSuccess) {
        cudaGetLastError();
        return fail(OCB_ERR_CUDA, "clear_episode_stats: %s", cudaGetErrorString(err));
    }
    return OCB_OK;
}

// ------------------------------------------------------------------ device-resident policy rollout
extern "C" const uint64_t* ocb_step_counter_device(const ocb_env* e) {
    return e ? reinterpret_cast<const uint64_t*>(e->d_step_counter) : nullptr;
}

// T x (fused actor+critic forward on the current observations -> one env step), all launches on
// `stream`, nothing synchronises; graph-capturable (the sampling offset is read from the device-side
// step counter, so a replayed graph draws fresh actions).  Writes the PPO rollout buffer in place.
extern "C" int ocb_rollout_policy(ocb_env* e, ocb_policy* pol, int T, const int32_t* tile_policy, int8_t* obs_slab,
                                  int32_t* actions, float* logp, float* values, int32_t* reward, int32_t* done,
                                  int deterministic, uint64_t seed, void* stream) {
    if (e == nullptr || pol == nullptr) return fail(OCB_ERR_INVALID_ARG, "NULL handle");
    if (obs_slab == nullptr || actions == nullptr) return fail(OCB_ERR_INVALID_ARG, "obs_slab and actions are required");
    if (T < 1) return fail(OCB_ERR_INVALID_ARG, "T must be >= 1");
    if (ocb_policy_obs_bytes(pol) != e->SC) return fail(OCB_ERR_INVALID_ARG, "env and policy were built for different layouts");
    const size_t PN = (size_t)e->P * e->N, obs_step = PN * (size_t)e->SC;
    const int M = (int)PN;
    const uint64_t* ctr = reinterpret_cast<const uint64_t*>(e->d_step_counter);
    for (int t = 0; t < T; ++t) {
        int rc;
        if (values != nullptr)
            rc = ocb_policy_forward(pol, obs_slab + t * obs_step, M, tile_policy, actions + t * PN,
                                    logp ? logp + t * PN : nullptr, nullptr, values + t * PN, deterministic, seed, 0, ctr,
                                    stream);
        else  // evaluation rollouts (train/testing.py:39-59, cross-play scoring) need no critic
            rc = ocb_policy_act_ex(pol, obs_slab + t * obs_step, M, tile_policy, actions + t * PN,
                                   logp ? logp + t * PN : nullptr, nullptr, deterministic, seed, 0, ctr, stream);
        if (rc != OCB_OK) return rc;
        rc = ocb_step(e, actions + t * PN, obs_slab + (t + 1) * obs_step, reward ? reward + t * PN : nullptr,
                      done ? done + (size_t)t * e->N : nullptr, stream);
        if (rc != OCB_OK) return rc;
    }
    if (values == nullptr) return OCB_OK;
    // bootstrap value of the observation after the last step (MainPlayer.compute_one,
    // train/MAPPO/main_player.py:293-307)
    // (through the same fused actor+critic kernel as the steps above, so that the value head sums in the same order
    // everywhere and ocb_rollout_policy_fused can reproduce the buffer bit for bit)
    return ocb_policy_forward(pol, obs_slab + (size_t)T * obs_step, M, tile_policy, nullptr, nullptr, nullptr,
                              values + (size_t)T * PN, 1, 0, 0, nullptr, stream);
}

// The same rollout as ocb_rollout_policy (self-play of ONE policy, critic required) in one persistent
// launch (csrc/rollout_fused.cuh): bit-identical buffers, no per-step launches.  Also writes obs_slab[0].
extern "C" int ocb_rollout_policy_fused(ocb_env* e, ocb_policy* pol, int T, int policy_index, int8_t* obs_slab,
                                        int32_t* actions, float* logp, float* values, int32_t* reward, int32_t* done,
                                        int deterministic, uint64_t seed, void* stream) {
    if (e == nullptr || pol == nullptr) return fail(OCB_ERR_INVALID_ARG, "NULL handle");
    if (e->P != 2) return fail(OCB_ERR_UNSUPPORTED, "the policy rollout supports 2 players");
    DeviceGuard guard(e->device);
    RolloutParams p = base_params(e);
    const int rc = ocb_policy_rollout_fused_launch(pol, policy_index, nullptr, false, p, e->h_tables.W, e->h_tables.H, T, obs_slab, actions,
                                                   logp, values, reward, done, deterministic, seed,
                                                   reinterpret_cast<const uint64_t*>(e->d_step_counter),
                                                   reinterpret_cast<uint64_t*>(e->d_step_counter), stream);
    if (rc != OCB_OK) return rc;
    if (stream_capturing(stream))
        e->count_stale = true;
    else
        e->step_count += (uint64_t)T;
    return OCB_OK;
}

// Cross-play in one persistent launch: the rollout of ocb_rollout_policy(values = NULL) with a tile_policy table — seat-0 rows
// act with the actor of tile_policy[seat-0 tile], seat-1 rows with that of tile_policy[seat-1 tile] — bit-identical actions
// (same sampling counters).  Evaluation keeps no trajectory: every buffer is optional; the env's episode statistics
// (ocb_episode_stats) carry the result.
extern "C" int ocb_rollout_crossplay_fused(ocb_env* e, ocb_policy* pol, int T, const int32_t* tile_policy, int8_t* obs_slab,
                                           int32_t* actions, float* logp, int32_t* reward, int32_t* done, int deterministic,
                                           uint64_t seed, void* stream) {
    if (e == nullptr || pol == nullptr || tile_policy == nullptr) return fail(OCB_ERR_INVALID_ARG, "NULL handle / tile_policy");
    if (e->P != 2) return fail(OCB_ERR_UNSUPPORTED, "the policy rollout supports 2 players");
    DeviceGuard guard(e->device);
    RolloutParams p = base_params(e);
    const int rc = ocb_policy_rollout_fused_launch(pol, 0, tile_policy, false, p, e->h_tables.W, e->h_tables.H, T, obs_slab, actions,
                                                   logp, nullptr, reward, done, deterministic, seed,
                                                   reinterpret_cast<const uint64_t*>(e->d_step_counter),
                                                   reinterpret_cast<uint64_t*>(e->d_step_counter), stream);
    if (rc != OCB_OK) return rc;
    if (stream_capturing(stream))
        e->count_stale = true;
    else
        e->step_count += (uint64_t)T;
    return OCB_OK;
}

// Self-play of a population in one persistent launch: the worlds [128 s, 128 s + 128) are played by weight set
// slice_policy[s] on both seats, actor + critic — the buffers of ocb_rollout_policy(tile_policy = slice_policy ++
// slice_policy, values != NULL), bit for bit.  Also writes obs_slab[0].
extern "C" int ocb_rollout_population_fused(ocb_env* e, ocb_policy* pol, int T, const int32_t* slice_policy, int8_t* obs_slab,
                                            int32_t* actions, float* logp, float* values, int32_t* reward, int32_t* done,
                                            int deterministic, uint64_t seed, void* stream) {
    if (e == nullptr || pol == nullptr) return fail(OCB_ERR_INVALID_ARG, "NULL handle");
    if (e->P != 2) return fail(OCB_ERR_UNSUPPORTED, "the policy rollout supports 2 players");
    DeviceGuard guard(e->device);
    RolloutParams p = base_params(e);
    const int rc = ocb_policy_rollout_fused_launch(pol, 0, slice_policy, true, p, e->h_tables.W, e->h_tables.H, T, obs_slab, actions,
                                                   logp, values, reward, done, deterministic, seed,
                                                   reinterpret_cast<const uint64_t*>(e->d_step_counter),
                                                   reinterpret_cast<uint64_t*>(e->d_step_counter), stream);
    if (rc != OCB_OK) return rc;
    if (stream_capturing(stream))
        e->count_stale = true;
    else
        e->step_count += (uint64_t)T;
    return OCB_OK;
}

// Diagnostic twin of ocb_rollout_policy_fused: the same launch with the instrumented build of the kernel.  h_trace
// (HOST int64 [n_steps][64]) receives clock64 stamps of CTA 0 for steps u0 .. u0 + n_steps - 1 (event indices: see
// trace_ev in policy_kernels.cu).  Synchronous.
extern "C" int ocb_rollout_fused_debug_trace(ocb_env* e, ocb_policy* pol, int T, int policy_index, int8_t* obs_slab,
                                             int32_t* actions, float* logp, float* values, int32_t* reward, int32_t* done,
                                             uint64_t seed, int64_t* h_trace, int u0, int n_steps) {
    if (e == nullptr || pol == nullptr || h_trace == nullptr || n_steps < 1) return fail(OCB_ERR_INVALID_ARG, "NULL handle / trace");
    if (e->P != 2) return fail(OCB_ERR_UNSUPPORTED, "the policy rollout supports 2 players");
    DeviceGuard guard(e->device);
    long long* d_trace = nullptr;
    const size_t bytes = (size_t)n_steps * 64 * sizeof(long long);
    cudaError_t err = cudaMalloc(&d_trace, bytes);
    if (err == cudaSuccess) err = cudaMemset(d_trace, 0, bytes);
    if (err != cudaSuccess) {
        cudaGetLastError();
        return fail(OCB_ERR_CUDA, "ocb_rollout_fused_debug_trace: %s", cudaGetErrorString(err));
    }
    RolloutParams p = base_params(e);
    const int rc = ocb_policy_rollout_fused_launch(pol, policy_index, nullptr, false, p, e->h_tables.W, e->h_tables.H, T, obs_slab, actions,
                                                   logp, values, reward, done, 0, seed,
                                                   reinterpret_cast<const uint64_t*>(e->d_step_counter),
                                                   reinterpret_cast<uint64_t*>(e->d_step_counter), nullptr, d_trace, u0, n_steps);
    if (rc == OCB_OK) {
        e->step_count += (uint64_t)T;
        err = cudaDeviceSynchronize();
        if (err == cudaSuccess) err = cudaMemcpy(h_trace, d_trace, bytes, cudaMemcpyDeviceToHost);
    }
    cudaFree(d_trace);
    if (rc != OCB_OK) return rc;
    if (err != cudaSuccess) {
        cudaGetLastError();
        return fail(OCB_ERR_CUDA, "ocb_rollout_fused_debug_trace: %s", cudaGetErrorString(err));
    }
    return OCB_OK;
}

// ------------------------------------------------------------------ mixed-play collection (SURVEY §8f row 3)
// scratch layout: two ping-pong observations [P,N,SC] | a_main, a_partner, act [P,N] i32 | logp, v [P,N] f32 |
// reward [P,N] i32 | done [N] i32 | two constant tile tables
namespace {
struct MixScratch {
    int8_t* obs[2];
    int32_t *a_main, *a_partner, *act, *rew, *done, *tiles_main, *tiles_partner;
    float *logp, *v;
    size_t bytes;
    int n_tiles;
};
MixScratch mix_scratch(const ocb_env* e, void* base) {
    MixScratch m;
    const size_t PN = (size_t)e->P * e->N;
    char* b = static_cast<char*>(base);
    size_t off = 0;
    auto take = [&](size_t bytes) {
        char* r = b ? b + off : nullptr;
        off += (bytes + 255) & ~(size_t)255;
        return r;
    };
    m.obs[0] = reinterpret_cast<int8_t*>(take(PN * e->SC));
    m.obs[1] = reinterpret_cast<int8_t*>(take(PN * e->SC));
    m.a_main = reinterpret_cast<int32_t*>(take(PN * 4));
    m.a_partner = reinterpret_cast<int32_t*>(take(PN * 4));
    m.act = reinterpret_cast<int32_t*>(take(PN * 4));
    m.logp = reinterpret_cast<float*>(take(PN * 4));
    m.v = reinterpret_cast<float*>(take(PN * 4));
    m.rew = reinterpret_cast<int32_t*>(take(PN * 4));
    m.done = reinterpret_cast<int32_t*>(take((size_t)e->N * 4));
    m.n_tiles = (int)((PN + 127) / 128);
    m.tiles_main = reinterpret_cast<int32_t*>(take((size_t)m.n_tiles * 4));
    m.tiles_partner = reinterpret_cast<int32_t*>(take((size_t)m.n_tiles * 4));
    m.bytes = off;
    return m;
}
}  // namespace

extern "C" size_t ocb_rollout_mixed_scratch_bytes(const ocb_env* e) { return e ? mix_scratch(e, nullptr).bytes : 0; }

// 2L x { main actor+critic forward, partner actor forward, per-row select, env step, record of the forced
// worlds } + the value of the never-written slot L; every launch on `stream`, nothing synchronises,
// graph-capturable (the mask stream and the sampling offsets read the device-side step counter).
extern "C" int ocb_rollout_mixed(ocb_env* e, ocb_policy* pol, int L, int main_policy, int partner_policy, int8_t* obs_buf,
                                 int32_t* actions, float* logp, float* values, int32_t* reward, int32_t* done,
                                 int deterministic, uint64_t seed, uint64_t mix_seed, void* scratch, size_t scratch_bytes,
                                 void* stream) {
    if (e == nullptr || pol == nullptr) return fail(OCB_ERR_INVALID_ARG, "NULL handle");
    if (obs_buf == nullptr || actions == nullptr) return fail(OCB_ERR_INVALID_ARG, "obs_buf and actions are required");
    if (e->P != 2) return fail(OCB_ERR_UNSUPPORTED, "the policy rollout supports 2 players");
    if (L < 2) return fail(OCB_ERR_INVALID_ARG, "L must be >= 2");
    if (e->N % (L - 1) != 0)
        return fail(OCB_ERR_INVALID_ARG, "the env must hold a multiple of L - 1 = %d worlds (got %d)", L - 1, e->N);
    const int sets = ocb_policy_num_sets(pol);
    if (main_policy < 0 || main_policy >= sets || partner_policy < 0 || partner_policy >= sets)
        return fail(OCB_ERR_INVALID_ARG, "policy index out of range (the handle holds %d sets)", sets);
    const MixScratch m = mix_scratch(e, scratch);
    if (scratch == nullptr || scratch_bytes < m.bytes)
        return fail(OCB_ERR_INVALID_ARG, "scratch must hold ocb_rollout_mixed_scratch_bytes() = %zu bytes", m.bytes);
    if ((reinterpret_cast<uintptr_t>(scratch) & 255u) != 0) return fail(OCB_ERR_INVALID_ARG, "scratch must be 256-byte aligned");
    DeviceGuard guard(e->device);
    cudaStream_t st = (cudaStream_t)stream;
    const size_t PN = (size_t)e->P * e->N, obs_step = PN * (size_t)e->SC;
    const int M = (int)PN;
    const uint64_t* ctr = reinterpret_cast<const uint64_t*>(e->d_step_counter);
#define OCB_CU(call)                                                             \
    do {                                                                         \
        cudaError_t err__ = (call);                                              \
        if (err__ != cudaSuccess) {                                              \
            cudaGetLastError();                                                  \
            return fail(OCB_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(err__)); \
        }                                                                        \
    } while (0)
    OCB_CU(launch_fill2_i32(m.tiles_main, m.n_tiles, main_policy, m.tiles_partner, m.n_tiles, partner_policy, st));
    int rc = ocb_observe(e, m.obs[0], stream);
    if (rc != OCB_OK) return rc;
    // the partner samples from its own stream (same counters, different key)
    const uint64_t partner_seed = seed ^ 0x9E3779B97F4A7C15ull;
    for (int s = 0; s < 2 * L; ++s) {
        const int8_t* cur = m.obs[s & 1];
        rc = values ? ocb_policy_forward(pol, cur, M, m.tiles_main, m.a_main, m.logp, nullptr, m.v, deterministic, seed, 0,
                                         ctr, stream)
                    : ocb_policy_act_ex(pol, cur, M, m.tiles_main, m.a_main, m.logp, nullptr, deterministic, seed, 0, ctr,
                                        stream);
        if (rc != OCB_OK) return rc;
        rc = ocb_policy_act_ex(pol, cur, M, m.tiles_partner, m.a_partner, nullptr, nullptr, deterministic, partner_seed, 0,
                               ctr, stream);
        if (rc != OCB_OK) return rc;
        MixSelectParams sp;
        sp.a_main = m.a_main, sp.a_partner = m.a_partner, sp.act = m.act;
        sp.step_counter = e->d_step_counter, sp.mix_seed = mix_seed;
        sp.P = e->P, sp.N = e->N, sp.L = L, sp.s = s;
        OCB_CU(launch_mix_select(sp, st));
        rc = ocb_step(e, m.act, m.obs[(s + 1) & 1], m.rew, m.done, stream);
        if (rc != OCB_OK) return rc;
        MixRecordParams rp;
        rp.obs_cur = cur, rp.a_main = m.a_main, rp.logp_main = m.logp, rp.v_main = m.v, rp.rew_cur = m.rew,
        rp.done_cur = m.done;
        rp.obs_buf = obs_buf, rp.actions = actions, rp.logp = logp, rp.values = values, rp.reward = reward, rp.done = done;
        rp.P = e->P, rp.N = e->N, rp.SC = e->SC, rp.L = L, rp.s = s;
        OCB_CU(launch_mix_record(rp, st));
    }
    // slot L is never written by the collection (diaginsert / partinsert stop at L-1): the reference bootstraps from
    // the all-zero observation the buffer was created with (MainPlayer.compute_one on mp_buf.share_obs[-1]); the
    // critic's value of it is a constant of the weights (the tensor-core forward folds the terrain planes of real
    // observations into its bias, so it is evaluated on the host when the weights are set)
    OCB_CU(cudaMemsetAsync(obs_buf + (size_t)L * obs_step, 0, obs_step, st));
    if (values != nullptr) OCB_CU(launch_fill_f32(values + (size_t)L * PN, PN, ocb_policy_zero_obs_value(pol, main_policy), st));
    return OCB_OK;
#undef OCB_CU
}

// The collection of ocb_rollout_mixed in one persistent launch (rollout_fused.cuh, kMix): both actors in the pipeline, the
// per-row switch and the record of the forced worlds on the device.  Then main's critic over obs_buf[:L] in one value launch
// (every (t < L, seat, world) cell is recorded exactly once, so that is the per-step path's values[:L], bit for bit), and
// slot L as ocb_rollout_mixed leaves it.
extern "C" int ocb_rollout_mixed_fused(ocb_env* e, ocb_policy* pol, int L, int main_policy, int partner_policy, int8_t* obs_buf,
                                       int32_t* actions, float* logp, float* values, int32_t* reward, int32_t* done,
                                       int deterministic, uint64_t seed, uint64_t mix_seed, void* stream) {
    if (e == nullptr || pol == nullptr) return fail(OCB_ERR_INVALID_ARG, "NULL handle");
    if (obs_buf == nullptr || actions == nullptr) return fail(OCB_ERR_INVALID_ARG, "obs_buf and actions are required");
    if (e->P != 2) return fail(OCB_ERR_UNSUPPORTED, "the policy rollout supports 2 players");
    if (L < 2) return fail(OCB_ERR_INVALID_ARG, "L must be >= 2");
    if (e->N % (L - 1) != 0)
        return fail(OCB_ERR_INVALID_ARG, "the env must hold a multiple of L - 1 = %d worlds (got %d)", L - 1, e->N);
    const int sets = ocb_policy_num_sets(pol);
    if (main_policy < 0 || main_policy >= sets || partner_policy < 0 || partner_policy >= sets)
        return fail(OCB_ERR_INVALID_ARG, "policy index out of range (the handle holds %d sets)", sets);
    // the kernel stores observation rows as 4-byte words and the value pass reads them so: reject before anything runs
    if ((reinterpret_cast<uintptr_t>(obs_buf) & 3u) != 0) return fail(OCB_ERR_INVALID_ARG, "obs_buf must be 4-byte aligned");
    DeviceGuard guard(e->device);
    cudaStream_t st = (cudaStream_t)stream;
    const size_t PN = (size_t)e->P * e->N, obs_step = PN * (size_t)e->SC;
    RolloutParams p = base_params(e);
    FusedMixArgs mix;
    mix.L = L, mix.partner_policy = partner_policy, mix.mix_seed = mix_seed;
    mix.partner_seed = seed ^ 0x9E3779B97F4A7C15ull;  // the partner's sampling key of ocb_rollout_mixed
    int rc = ocb_policy_rollout_fused_launch(pol, main_policy, nullptr, false, p, e->h_tables.W, e->h_tables.H, 2 * L, obs_buf, actions,
                                             logp, nullptr, reward, done, deterministic, seed,
                                             reinterpret_cast<const uint64_t*>(e->d_step_counter),
                                             reinterpret_cast<uint64_t*>(e->d_step_counter), stream, nullptr, 0, 0, &mix);
    if (rc != OCB_OK) return rc;
    if (stream_capturing(stream))
        e->count_stale = true;
    else
        e->step_count += (uint64_t)(2 * L);
    if (values != nullptr) {
        rc = ocb_policy_value_of(pol, main_policy, obs_buf, (int)((size_t)L * PN), values, stream);
        if (rc != OCB_OK) return rc;
    }
    cudaError_t err = cudaMemsetAsync(obs_buf + (size_t)L * obs_step, 0, obs_step, st);
    if (err == cudaSuccess && values != nullptr)
        err = launch_fill_f32(values + (size_t)L * PN, PN, ocb_policy_zero_obs_value(pol, main_policy), st);
    if (err != cudaSuccess) {
        cudaGetLastError();
        return fail(OCB_ERR_CUDA, "ocb_rollout_mixed_fused: %s", cudaGetErrorString(err));
    }
    return OCB_OK;
}
