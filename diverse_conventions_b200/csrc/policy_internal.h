// policy_internal.h — entry points of policy_kernels.cu used by ocb_api.cu (not part of the C ABI)
#pragma once
#include <stdint.h>

#include "oc_kernels.h"
#include "ocb.h"

// mixed play in the fused rollout (ocb_rollout_mixed_fused): the partner's actor, the collection length L, the mask key and
// the partner's sampling key
struct FusedMixArgs {
    int L, partner_policy;
    uint64_t mix_seed, partner_seed;
};

// T-step rollout in ONE persistent launch (rollout_fused.cuh): `envp` carries the env's tables and state arrays.
// tile_policy == nullptr: self-play of weight set `policy_index` (actor + critic); else cross-play with the per-step path's
// seat-major tile table (actors only, every output buffer optional); with `population`, tile_policy is a table by 128-world
// slice and each slice is self-play of its weight set (actor + critic); with `mix`, mixed play of the actors of
// policy_index and mix->partner_policy (T = 2 L, no critic).  Returns OCB_ERR_UNSUPPORTED (with the reason in
// ocb_last_error) when the layout / handle cannot run fused.
int ocb_policy_rollout_fused_launch(ocb_policy* pol, int policy_index, const int32_t* tile_policy, bool population,
                                    const ocb::RolloutParams& envp, int env_w, int env_h, int T, int8_t* obs_slab, int32_t* actions,
                                    float* logp, float* values, int32_t* reward, int32_t* done, int deterministic, uint64_t seed,
                                    const uint64_t* d_offset, uint64_t* d_counter, void* stream, long long* d_trace = nullptr,
                                    int trace_u0 = 0, int trace_n = 0, const FusedMixArgs* mix = nullptr);

// ocb_policy_value with the critic of weight set `policy_index` and no table (hidden 64, tensor-core path only)
int ocb_policy_value_of(ocb_policy* pol, int policy_index, const int8_t* obs, int M, float* values, void* stream);

// bytes of one observation row the handle was built for (W * H * (5 P + 10)); 1 when shapes outside the tensor-core
// kernels' range run through policy_generic_kernel
int ocb_policy_obs_bytes(const ocb_policy* pol);
int ocb_policy_is_generic(const ocb_policy* pol);
// number of (actor, critic) weight sets the handle holds
int ocb_policy_num_sets(const ocb_policy* pol);
// R_Critic value of the all-zero observation under weight set `policy` (computed on the host at set_weights)
float ocb_policy_zero_obs_value(const ocb_policy* pol, int policy);
