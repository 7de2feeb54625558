/*
 * ocb.h — C ABI of the B200-native batched Overcooked / Balance-Beam simulator.
 *
 * This is the drop-in boundary under the reference's batched multi-agent env API
 * (pantheonrl_extension/vectorenv.py:26-255, VectorMultiAgentEnv.n_step / n_reset).
 * In the reference the same role is played by the nanobind class
 * `SimplecookedSimulator` (src/overcooked2_env/bindings.cpp:27-96; tensor exports
 * src/overcooked2_env/mgr.cpp:213-272) and `BalanceBeamSimulator`
 * (src/balance_beam_env/bindings.cpp, mgr.cpp:191-233).  Each entry point below cites
 * the reference interface it replaces.
 *
 * Conventions
 *   - plain C, plain pointers and sizes; no torch / C++ types cross this boundary;
 *   - return 0 on success, a negative OCB_ERR_* otherwise; never abort();
 *     ocb_last_error() returns a thread-local human readable message;
 *   - the library owns only the world state (structure-of-arrays in HBM);
 *     every input / output buffer is owned by the caller (e.g. torch tensors);
 *   - pointers are DEVICE pointers unless the function name ends in `_host`;
 *   - all launches are asynchronous on the caller supplied `stream`
 *     (a cudaStream_t passed as void*; NULL = legacy default stream); the
 *     library never synchronises except in the `_host`, get/set_state calls;
 *   - one handle is single-threaded; different handles / GPUs are independent.
 *
 * Tensor layouts (N worlds, P players, W x H grid, C = 5P + 10 channels):
 *   actions  [P, N]            int32 (or see ocb_step_ex), values 0..5
 *                              (N,S,E,W,STAY,INTERACT; envs/overcooked2_reimplement.py:35-43);
 *                              out-of-range values are treated as STAY
 *   obs      [P, N, W, H, C]   int8, lossless state encoding
 *                              (envs/overcooked2_reimplement.py:173-259, axis order
 *                              envs/overcooked2_env.py:322-325)
 *   reward   [P, N]            int32, team reward replicated per player
 *                              (envs/overcooked2_env.py:336-339; mgr.cpp:244-248)
 *   done     [N]               int32 0/1 (mgr.cpp:213-217); on a done step the world
 *                              is reset and obs is the post-reset observation
 *                              (pantheonrl_extension/vectorenv.py:369-370)
 *   K-step rollouts prepend a [K] axis to every tensor.
 */
#ifndef OCB_H_
#define OCB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OCB_ABI_VERSION 1
#define OCB_MAX_PLAYERS 4
#define OCB_MAX_CELLS 256
#define OCB_NUM_RECIPES 16 /* (MAX_NUM_INGREDIENTS+1)^2, index 4*onions+tomatoes */
#define OCB_MAX_COOK_TIME 120 /* cooking tick must fit the int8 observation */

/* error codes */
#define OCB_OK 0
#define OCB_ERR_INVALID_ARG (-1)
#define OCB_ERR_BAD_LAYOUT (-2)
#define OCB_ERR_CUDA (-3)
#define OCB_ERR_NO_DEVICE (-4)
#define OCB_ERR_BAD_STATE (-5)
#define OCB_ERR_UNSUPPORTED (-6)

/* action dtypes accepted by ocb_step_ex / ocb_rollout_actions */
#define OCB_ACT_I32 0
#define OCB_ACT_I64 1
#define OCB_ACT_F32 2
#define OCB_ACT_U8 3

/*
 * Flat POD layout description == the keyword arguments the reference passes to
 * SimplecookedSimulator / DummyMDP (envs/overcooked2_env.py:171-291,
 * envs/overcooked2_reimplement.py:121-151).
 */
typedef struct ocb_config {
    uint32_t struct_size; /* sizeof(ocb_config): versioning */
    int32_t width;
    int32_t height;
    int32_t num_players; /* 1..OCB_MAX_PLAYERS */
    int32_t horizon;     /* episode length, done = timestep >= horizon */
    int32_t placement_in_pot_rew;
    int32_t dish_pickup_rew;
    int32_t soup_pickup_rew;
    int32_t recipe_values[OCB_NUM_RECIPES];
    int32_t recipe_times[OCB_NUM_RECIPES];
    int32_t start_player_x[OCB_MAX_PLAYERS];
    int32_t start_player_y[OCB_MAX_PLAYERS];
    /* terrain codes, row-major (pos = y*width + x):
     * 0 AIR, 1 POT, 2 COUNTER, 3 ONION_SOURCE, 4 DISH_SOURCE, 5 SERVING, 6 TOMATO_SOURCE */
    uint8_t terrain[OCB_MAX_CELLS];
} ocb_config;

typedef struct ocb_env ocb_env; /* opaque Overcooked handle */
typedef struct bb_env bb_env;   /* opaque Balance-Beam handle */

/* ------------------------------------------------------------------ misc */
int ocb_abi_version(void);
/* thread-local message describing the last error on this thread */
const char* ocb_last_error(void);
/* number of visible CUDA devices, or a negative error */
int ocb_device_count(void);

/* ------------------------------------------------------- Overcooked: life-cycle */
/* replaces SimplecookedSimulator.__init__ (bindings.cpp:27-60, mgr.cpp:128-200);
 * all worlds start in the standard start state (reimplement.py:387-391). */
int ocb_create(const ocb_config* cfg, int device, uint32_t num_worlds, uint64_t seed, ocb_env** out);
int ocb_destroy(ocb_env* env);

/* shape queries */
int ocb_num_worlds(const ocb_env* env);
int ocb_num_players(const ocb_env* env);
int ocb_obs_channels(const ocb_env* env);         /* C = 5P + 10 */
int ocb_obs_bytes_per_agent(const ocb_env* env);  /* W*H*C */
int ocb_state_ints_per_world(const ocb_env* env); /* length of one packed world state */

/* kernel tuning knobs: lanes_per_world in {1,2,4,8} — lanes that serve one world in the one-warp kernel — or 16, the
 * role-split kernel (a transition warp + encoder warps per 32 worlds; two players and at most two pots, else
 * OCB_ERR_UNSUPPORTED; launches it does not serve — single steps, no observations — use the one-warp kernel);
 * 0 = default by layout and world count.  use_tma in {0,1} (default 1: TMA bulk stores of the observation tiles) */
int ocb_set_tuning(ocb_env* env, int lanes_per_world, int use_tma);
/* the launch shape currently in effect (any out pointer may be NULL) */
int ocb_get_tuning(const ocb_env* env, int* lanes_per_world, int* use_tma, int* warps_per_cta);

/* ------------------------------------------------------- Overcooked: hot path */
/* VectorMultiAgentEnv.n_reset (vectorenv.py:241-252 / SyncVectorEnv.n_reset 398-425):
 * reset every world, optionally write obs [P,N,W,H,C] (obs may be NULL). */
int ocb_reset(ocb_env* env, int8_t* obs, void* stream);

/* observation of the current state, no stepping (OvercookedMadrona.get_obs,
 * envs/overcooked2_env.py:103-114). */
int ocb_observe(ocb_env* env, int8_t* obs, void* stream);

/* VectorMultiAgentEnv.n_step (vectorenv.py:220-239; OvercookedMadrona.n_step
 * envs/overcooked2_env.py:116-125 == sim.step() + scatter glue). One fused kernel:
 * interact -> movement/collision -> cook tick -> reward -> done/auto-reset -> obs.
 * obs / reward / done may each be NULL to skip that output. */
int ocb_step(ocb_env* env, const int32_t* actions, int8_t* obs, int32_t* reward, int32_t* done, void* stream);
/* same, actions given in another dtype (trainers pass float32, envs/overcooked2_env.py:119) */
int ocb_step_ex(ocb_env* env, const void* actions, int act_dtype, int8_t* obs, int32_t* reward, int32_t* done,
                void* stream);

/* K fused steps in one launch with caller supplied actions [K,P,N]; outputs get a
 * leading [K] axis (obs_slab [K,P,N,W,H,C]); any output may be NULL. */
int ocb_rollout_actions(ocb_env* env, int K, const void* actions, int act_dtype, int8_t* obs_slab,
                        int32_t* reward, int32_t* done, void* stream);

/* K fused steps with uniform random actions drawn on the device from the
 * counter-based RNG (Philox4x32-10 keyed by seed, indexed by (world, step));
 * actions_out [K,P,N] uint8 (may be NULL) records what was played so the
 * trajectory can be replayed through the oracle. */
int ocb_rollout_random(ocb_env* env, int K, int8_t* obs_slab, int32_t* reward, int32_t* done,
                       uint8_t* actions_out, void* stream);

/* host-buffer variant of ocb_step: copies actions H2D, steps, copies outputs D2H
 * and synchronises.  Pointers are HOST pointers (pinned memory recommended);
 * h_obs / h_reward / h_done may be NULL. */
int ocb_step_host(ocb_env* env, const int32_t* h_actions, int8_t* h_obs, int32_t* h_reward, int32_t* h_done);
/* The same step as a two-deep pipeline on the env's own streams: the call enqueues H2D actions -> kernel -> D2H
 * (reward and done first, then the observation planes) and returns; at most two steps are in flight (a third call first
 * retires the oldest).  ocb_step_host_wait blocks until the OLDEST enqueued step has delivered its host buffers and
 * returns how many steps remain in flight (0 / 1) or a negative error code.  With the next actions already at hand (a
 * scripted / replayed / random partner, or a policy that acts one step late) the 13 MB observation copy of step t
 * overlaps the upload and kernel of step t + 1.  Host buffers of a step must stay untouched until its wait returns;
 * retire every step before calling any other entry point on the handle. */
int ocb_step_host_async(ocb_env* env, const int32_t* h_actions, int8_t* h_obs, int32_t* h_reward, int32_t* h_done);
int ocb_step_host_wait(ocb_env* env);

/* ------------------------------------------------------- Overcooked: state I/O */
/* Packed world state, int32 [N, L], L = ocb_state_ints_per_world():
 *   [0]            timestep
 *   per player i:  pos, orientation, held_name, held_onions, held_tomatoes, held_cooking_tick
 *   per cell c:    obj_name, obj_onions, obj_tomatoes, obj_cooking_tick   (name 0 = NONE)
 * mirrors OvercookedState / PlayerState / ObjectState (reimplement.py:46-117).
 * HOST pointers; these calls synchronise. */
int ocb_get_state(ocb_env* env, int32_t* h_state, size_t n_ints);
int ocb_set_state(ocb_env* env, const int32_t* h_state, size_t n_ints);

/* per-world episode statistics kept on the device: sum of returns of completed
 * episodes, number of completed episodes (replaces the host-side
 * running_score bookkeeping, train/MAPPO/main_player.py:256-261).
 * DEVICE pointers, each may be NULL. */
int ocb_read_episode_stats(ocb_env* env, int64_t* return_sum, int32_t* episodes, void* stream);
int ocb_clear_episode_stats(ocb_env* env, void* stream);

/* global step counter that indexes the action RNG (incremented by every step) */
uint64_t ocb_step_count(const ocb_env* env);
/* index of this handle's world 0 in the global world numbering used by the action RNG
 * (a multi-GPU shard of rank r with N worlds per rank uses r*N); default 0 */
int ocb_set_world_offset(ocb_env* env, uint32_t world0);

/* ------------------------------------------------------- policy forward (MAPPO actor / critic) */
/* Fused tensor-core forward of the reference's CNN actor / critic (R_Actor / R_Critic,
 * train/MAPPO/r_actor_critic.py:12-71,142-197; CNNLayer train/MAPPO/utils/cnn.py:22-42;
 * Categorical head train/MAPPO/utils/distributions.py:55-68), 2 players, hidden_size 64 (every
 * train script; one fused kernel) or 512 (argparse default train/config.py:199; three GEMM-sized
 * launches).  Shapes below are for hidden h: conv_w [h/2,20,3,3], fc1_w [h, (h/2)(W-2)(H-2)],
 * fc2_w [h,h], head_w [6|1, h].
 * A handle holds n_policies (actor, critic) weight sets for one layout. */
typedef struct ocb_policy ocb_policy;
int ocb_policy_create(const ocb_config* cfg, int device, int hidden, int n_policies, ocb_policy** out);
int ocb_policy_destroy(ocb_policy* pol);
/* HOST fp32 weights in the reference's state-dict layouts: conv_w [32,20,3,3] (base.cnn.cnn.0),
 * fc1_w [64, 32*(W-2)*(H-2)] (base.cnn.cnn.3), fc2_w [64,64] (base.cnn.cnn.5), head_w [6,64]
 * (act.action_out.linear, net 0) or [1,64] (v_out, net 1), and the matching biases. */
int ocb_policy_set_weights(ocb_policy* pol, int policy, int net, const float* conv_w, const float* conv_b,
                           const float* fc1_w, const float* fc1_b, const float* fc2_w, const float* fc2_b,
                           const float* head_w, const float* head_b);
/* actor: obs int8 [M, W, H, C] (DEVICE) -> sampled (or arg-max) actions int32 [M], log-probs
 * float [M], raw logits float [M,6]; any output may be NULL.  tile_policy int32 [ceil(M/128)]
 * selects the weight set per 128-row tile (NULL = set 0) — the cross-play slice multiplexing of
 * train/partner_agents.py:87-137 / train/XD/xd_player.py:177-230.  Sampling uses the counter RNG
 * keyed by (seed, row, offset). */
int ocb_policy_act(ocb_policy* pol, const int8_t* obs, int M, const int32_t* tile_policy, int32_t* actions,
                   float* logp, float* logits, int deterministic, uint64_t seed, uint64_t offset, void* stream);
/* same with a DEVICE-resident addend of `offset` (see ocb_policy_forward) */
int ocb_policy_act_ex(ocb_policy* pol, const int8_t* obs, int M, const int32_t* tile_policy, int32_t* actions,
                      float* logp, float* logits, int deterministic, uint64_t seed, uint64_t offset,
                      const uint64_t* d_offset, void* stream);
/* critic: values float [M] */
int ocb_policy_value(ocb_policy* pol, const int8_t* obs, int M, const int32_t* tile_policy, float* values,
                     void* stream);

/* both networks in ONE launch (hidden 64: one CTA runs both networks of a 128-row tile; hidden 512:
 * even CTAs run the actor, odd CTAs the critic): everything
 * ocb_policy_act and ocb_policy_value write; values is required.  d_offset (DEVICE pointer, may
 * be NULL) is added to `offset` on the device, so a CUDA graph that replays this launch samples
 * with a fresh counter (pass ocb_step_counter_device(env)). */
int ocb_policy_forward(ocb_policy* pol, const int8_t* obs, int M, const int32_t* tile_policy, int32_t* actions,
                       float* logp, float* logits, float* values, int deterministic, uint64_t seed, uint64_t offset,
                       const uint64_t* d_offset, void* stream);
/* Sampling streams that do not depend on how an env is sharded.  By default launch row r (r = seat * N + world for
 * the rollouts) draws from counter row r.  For a shard holding worlds world0 .. world0 + N - 1 of N_total, call this
 * with (N, world0, N_total - N + world0): seat-0 rows map to world0 + world, seat-1 rows to N_total + world0 + world,
 * i.e. every (seat, global world) keeps its stream on any number of GPUs — the cross-play matrix gathered from 8 ranks
 * is bit-identical to the single-GPU one.  Applies to every later sampling launch of this handle; (0, 0, 0) restores
 * the default.  Not in the reference (its sampling is torch's global generator, train/MAPPO/utils/distributions.py:14-20). */
int ocb_policy_set_sampling_rows(ocb_policy* pol, uint32_t rows_per_seat, uint32_t add_seat0, uint32_t add_seat1);
/* launch shape of the hidden-64 forward: weight-ring slots in shared memory, FC weight chunks of
 * both networks per tile (ring >= chunks means the weights stay resident), dynamic shared memory
 * per CTA; ring and shared memory are 0 for hidden 512 and for the generic kernel */
int ocb_policy_info(const ocb_policy* pol, int* ring_slots, int* chunks_per_unit, int* smem_bytes);
/* pre-size the handle's internal activation scratch (hidden 512 only) for forwards of up to M rows:
 * required before a forward of a new, larger M is captured into a CUDA graph */
int ocb_policy_reserve(ocb_policy* pol, int M);

/* diagnostic: one fused forward with the instrumented kernel build; h_prof (HOST) int64
 * [max_ctas][4 roles: epilogue, loader, MMA issuer, producer][16] = total cycles and cycles stalled
 * per hand-off; returns the number of CTAs launched (or a negative error) */
int ocb_policy_debug_profile(ocb_policy* pol, const int8_t* obs, int M, const int32_t* tile_policy, float* values,
                             int32_t* actions, int64_t* h_prof, int max_ctas);

/* ------------------------------------------------------- device-resident self-play / cross-play rollout */
/* DEVICE address of the env's step counter (uint64, += K after every K-step launch) */
const uint64_t* ocb_step_counter_device(const ocb_env* env);
/* The rollout half of MainPlayer.collect_episode / next_step (train/MAPPO/main_player.py:91-112,
 * 211-261) with the partner seat of CentralizedAgent.get_action (train/partner_agents.py:28-63)
 * or, with tile_policy, the slice-wise policy multiplexing of XDPlayer.next_step /
 * CentralizedMultiAgent (train/XD/xd_player.py:177-230, train/partner_agents.py:87-137):
 * T times { fused actor+critic forward of all P*N agent rows on obs_slab[t] -> actions[t],
 * logp[t], values[t];  one env step -> obs_slab[t+1], reward[t], done[t] } and finally the
 * bootstrap values[T] of obs_slab[T].  obs_slab[0] must hold the current observation
 * (ocb_reset / ocb_observe).  Layouts (SharedReplayBuffer, train/MAPPO/utils/shared_buffer.py:45-76,
 * kept seat-major): obs_slab [T+1,P,N,W,H,C] int8, actions [T,P,N] int32, logp [T,P,N] f32,
 * values [T+1,P,N] f32, reward [T,P,N] int32, done [T,N] int32 (masks = 1 - done).
 * logp, reward, done may be NULL; values may be NULL too, then only the actors run (evaluation
 * and cross-play scoring, train/testing.py:39-59).  2*T+1 launches on `stream`, no
 * synchronisation; the sequence is CUDA-graph capturable (sampling offsets are read from the
 * device-side step counter, so a replayed graph draws fresh actions). */
int ocb_rollout_policy(ocb_env* env, ocb_policy* pol, int T, const int32_t* tile_policy, int8_t* obs_slab,
                       int32_t* actions, float* logp, float* values, int32_t* reward, int32_t* done,
                       int deterministic, uint64_t seed, void* stream);

/* ocb_rollout_policy for self-play of ONE weight set (policy_index of the handle; hidden 64, critic
 * required: values != NULL) as a single persistent launch: each CTA owns 64 worlds (128 agent rows)
 * for all T steps, the env step and the actor+critic forward hand over through shared memory, and
 * only the rollout-buffer writes touch HBM.  Buffers are bit-identical to ocb_rollout_policy's
 * (same sampling counters); obs_slab[0] is written by the kernel (no ocb_observe needed).
 * OCB_ERR_UNSUPPORTED when the layout does not fit the kernel's shared memory — callers then use
 * ocb_rollout_policy.  Replaces the same reference loop (train/MAPPO/main_player.py:91-112,211-261). */
int ocb_rollout_policy_fused(ocb_env* env, ocb_policy* pol, int T, int policy_index, int8_t* obs_slab, int32_t* actions,
                             float* logp, float* values, int32_t* reward, int32_t* done, int deterministic,
                             uint64_t seed, void* stream);

/* Cross-play evaluation in ONE persistent launch (the slices of XDPlayer / CentralizedMultiAgent, train/XD/xd_player.py:177-230,
 * train/partner_agents.py:87-137, generalised to arbitrary pairs): the rollout of ocb_rollout_policy(values = NULL) with
 * `tile_policy` (DEVICE int32 [2 N / 128], seat-major: tile t of seat 0 rows, then of seat 1 rows) — same sampled actions, same
 * env transitions.  N must be a multiple of 128.  Every output buffer is optional (NULL): evaluation keeps no trajectory,
 * ocb_episode_stats carries the returns.  OCB_ERR_UNSUPPORTED when the layout does not fit the kernel. */
int ocb_rollout_crossplay_fused(ocb_env* env, ocb_policy* pol, int T, const int32_t* tile_policy, int8_t* obs_slab,
                                int32_t* actions, float* logp, int32_t* reward, int32_t* done, int deterministic,
                                uint64_t seed, void* stream);

/* Self-play of a population in ONE persistent launch (the per-member self-play slices of ADAP's simultaneous trainer and of
 * XD's conventions, train/ADAP/simultaneous.py, train/XD/serial.py): the worlds [128 s, 128 s + 128) are played by weight
 * set slice_policy[s] on both seats, actor + critic, hidden 64.  slice_policy: DEVICE int32 [N / 128], every entry in
 * [0, n_policies) of the handle (not checked: the table stays on the device; an entry out of range reads outside the
 * weights, as with the tile_policy tables of the other entry points).  The same buffers, bit
 * for bit, as ocb_rollout_policy(tile_policy = slice_policy ++ slice_policy, values != NULL) — same sampling counters, same
 * env transitions, same bootstrap values[T].  obs_slab, actions and values are required (OCB_ERR_INVALID_ARG otherwise, and
 * when N is not a multiple of 128); obs_slab[0] is written by the kernel.  OCB_ERR_UNSUPPORTED for hidden 512 and for
 * layouts the fused kernel does not take — callers then use ocb_rollout_policy. */
int ocb_rollout_population_fused(ocb_env* env, ocb_policy* pol, int T, const int32_t* slice_policy, int8_t* obs_slab,
                                 int32_t* actions, float* logp, float* values, int32_t* reward, int32_t* done,
                                 int deterministic, uint64_t seed, void* stream);

/* Diagnostic: ocb_rollout_policy_fused through the instrumented build of the kernel (synchronous, sampled
 * actions).  h_trace (HOST int64 [n_steps][64]) receives clock64 stamps of CTA 0 for steps u0 .. u0+n_steps-1;
 * event indices are listed at trace_ev in csrc/policy_kernels.cu (env / loader / MMA issue / epilogue hand-offs).
 * Used by tools/fused_trace.py to attribute the per-step latency of the dependent chain. */
int ocb_rollout_fused_debug_trace(ocb_env* env, ocb_policy* pol, int T, int policy_index, int8_t* obs_slab,
                                  int32_t* actions, float* logp, float* values, int32_t* reward, int32_t* done,
                                  uint64_t seed, int64_t* h_trace, int u0, int n_steps);

/* ------------------------------------------------------- mixed-play ("MP") collection */
/* XDPlayer.collect_mp_episode / next_mp_step (train/XD/xd_player.py:232-356) with the partner seat of
 * MixedAgent (train/partner_agents.py:151-244) and the buffer placement of SharedReplayBuffer.diaginsert /
 * partinsert (train/MAPPO/utils/shared_buffer.py:150-220), L = the trainer's episode_length:
 * the env holds R replicas of G = L - 1 worlds (N = R*G; the reference runs R = 1, train/XD/serial.py:29) and is
 * stepped 2L times from its current state.  At step s every agent row draws use_partner = (Philox4x32-10(counter =
 * (row, step_lo, step_hi, "MIXE"), key = mix_seed).x < 2^31), row = seat*N + world, step = the env's global
 * step count, unless world j = world mod G is FORCED to the main policy: s < L: j >= G - s (s > 0);
 * s >= L: j < s - L.  The row plays the partner_policy actor's action when use_partner, else the
 * main_policy actor's.  Exactly the forced worlds are recorded, all fields at the same slot t
 * (s < L: t = j - G + s, the diagonal of diaginsert; s >= L: t = s - L, the row prefix of partinsert):
 * obs_buf [L+1,P,N,W,H,C] int8 <- the observation acted on, actions [L,P,N] int32, logp [L,P,N] f32 and
 * values [L+1,P,N] f32 of the main policy (actor, critic = the handle's weight set main_policy; the reference
 * pairs the trained actor with mp_critic, train/XD/MCPolicy.py:21,60), reward [L,P,N] int32 and done [L,N] int32
 * of that step (the reference stores masks = 1 - done at slot t here, not t + 1).  Every (t < L, seat, world)
 * cell is written exactly once.  Slot L is what the reference leaves it: obs_buf[L] = 0 and values[L] = the
 * critic's value of the all-zero observation (MainPlayer.compute_one on the never-written share_obs[-1]).
 * logp, values, reward, done may be NULL.  `scratch` (DEVICE, 256-byte aligned, at least
 * ocb_rollout_mixed_scratch_bytes(env) bytes) holds the per-step turn data.  10L + 4 launches on `stream`, no
 * synchronisation, CUDA-graph capturable (masks and sampling offsets read the device-side step counter). */
size_t ocb_rollout_mixed_scratch_bytes(const ocb_env* env);
int ocb_rollout_mixed(ocb_env* env, ocb_policy* pol, int L, int main_policy, int partner_policy, int8_t* obs_buf,
                      int32_t* actions, float* logp, float* values, int32_t* reward, int32_t* done, int deterministic,
                      uint64_t seed, uint64_t mix_seed, void* scratch, size_t scratch_bytes, void* stream);

/* The same collection in ONE persistent launch of the fused rollout kernel (hidden 64): both actors run in the kernel's
 * pipeline, the per-row switch, the forced worlds and their record at slot t happen on the device, then main_policy's critic
 * runs once over the L * P * N rows of obs_buf[:L] (skipped when values == NULL) and slot L is written as above.  The same
 * buffers, bit for bit, and the same final env state as ocb_rollout_mixed; buffer cells of rows that are not recorded are
 * never written.  The env's step counter advances by 2L.  Needs no scratch; 5 launches with values, 3 without, on `stream`,
 * no synchronisation, CUDA-graph capturable.  OCB_ERR_INVALID_ARG as ocb_rollout_mixed and for an obs_buf that is not
 * 4-byte aligned (checked before anything is launched); OCB_ERR_UNSUPPORTED for hidden 512,
 * for layouts outside the tensor-core kernels and for layouts too large for the fused kernel — callers then use
 * ocb_rollout_mixed. */
int ocb_rollout_mixed_fused(ocb_env* env, ocb_policy* pol, int L, int main_policy, int partner_policy, int8_t* obs_buf,
                            int32_t* actions, float* logp, float* values, int32_t* reward, int32_t* done, int deterministic,
                            uint64_t seed, uint64_t mix_seed, void* stream);

/* ------------------------------------------------------- returns / GAE over the rollout buffer */
/* SharedReplayBuffer.compute_returns (train/MAPPO/utils/shared_buffer.py:248-304) with the
 * ValueNorm de-normalisation (train/MAPPO/utils/valuenorm.py:76-87) and the advantage
 * normalisation at the top of R_MAPPO.train (train/MAPPO/r_mappo.py:174-182), directly over the
 * seat-major buffers ocb_rollout_policy fills.  bad_masks are all ones for these envs
 * (main_player.py:274), so the use_proper_time_limits branches reduce to the ones below. */
typedef struct ocb_returns_cfg {
    uint32_t struct_size; /* sizeof(ocb_returns_cfg) */
    int32_t use_gae;      /* 1: GAE (default), 0: discounted sum of rewards */
    double gamma;         /* config.py:251, default 0.99; doubles because the reference forms gamma * gae_lambda in */
    double gae_lambda;    /* config.py:253, default 0.95;   Python floats before the fp32 tensor arithmetic */
    float vn_mean;        /* ValueNorm.running_mean_var(): debiased mean (0 without a value normaliser) */
    float vn_std;         /* sqrt of the debiased, clamped variance (1 without a value normaliser) */
} ocb_returns_cfg;
/* value_preds [T+1,P,N] f32 (slot T = bootstrap value), rewards [T,P,N] int32, done [T,N] int32
 * (masks[t+1] = 1 - done[t]) -> returns [T+1,P,N] f32 (slot T = value_preds[T] without GAE, shared_buffer.py:297; untouched with GAE),
 * advantages [T,P,N] f32 = returns - denormalised value_preds (un-normalised; may be NULL),
 * adv_stats double[3] = (sum, sum of squares, count) of the advantages (may be NULL).
 * All DEVICE pointers; fp32 arithmetic in the reference's operation order (bit-identical to torch
 * on the CPU), statistics in fp64. */
int ocb_compute_returns(int device, const ocb_returns_cfg* cfg, int T, int P, int N, const float* value_preds,
                        const int32_t* rewards, const int32_t* done, float* returns, float* advantages,
                        double* adv_stats, void* stream);
/* Same, with the ValueNorm statistics read on the DEVICE: vn_mean_std = float[2] (debiased mean, sqrt of the clamped
 * debiased variance), overriding cfg->vn_mean / vn_std when not NULL — no host round trip, graph-capturable. */
int ocb_compute_returns_dev(int device, const ocb_returns_cfg* cfg, int T, int P, int N, const float* value_preds,
                            const int32_t* rewards, const int32_t* done, float* returns, float* advantages,
                            double* adv_stats, const float* vn_mean_std, void* stream);
/* advantages <- (advantages - mean) / (std + 1e-5), unbiased std, from adv_stats (r_mappo.py:180-182).  Sharded runs
 * all-reduce (sum) the three doubles across ranks between the two calls so that every rank normalises with the
 * statistics of the whole batch (returns.py: compute_returns(group=...)). */
int ocb_normalize_advantages(int device, float* advantages, size_t n, const double* adv_stats, void* stream);

/* ------------------------------------------------------- PPO minibatch: gather, evaluate_actions, loss */
/* The data side of R_MAPPO.ppo_update (train/MAPPO/r_mappo.py:91-164) over the seat-major rollout
 * buffer, consuming the int8 observations in place.  A minibatch is a list of agent-row indices
 * `rows` (int32 [B], DEVICE): row = (t*P + seat)*N + world addresses obs_slab[:T], actions, logp,
 * value_preds[:T], returns[:T] and advantages alike.  (The reference flattens [T,N,P] instead,
 * shared_buffer.py:306-366; the host adapter converts its randperm indices.) */

/* evaluate_actions (R_Actor.evaluate_actions r_actor_critic.py:73-109, ACTLayer.evaluate_actions
 * utils/act.py:107-175 Discrete branch, R_Critic.forward 178-197): the tensor-core forward of
 * ocb_policy_forward over obs rows picked by `rows` (NULL = rows 0..B-1), with the log-probability
 * of the STORED action actions_src[row] and the entropy of the distribution per row instead of
 * sampling.  obs [R,W,H,C] int8, actions_src int32 [R] (both indexed by source row); outputs are
 * indexed by minibatch position: logp [B], entropy [B], logits [B,6] (may be NULL), values [B]
 * (NULL = actor only).  hidden 64 and 512. */
int ocb_policy_evaluate(ocb_policy* pol, const int8_t* obs, const int32_t* rows, int B, const int32_t* tile_policy,
                        const int32_t* actions_src, float* logp, float* entropy, float* logits, float* values,
                        void* stream);

/* feed_forward_generator's fancy-indexing (shared_buffer.py:339-361) as one launch: copies the B
 * picked rows of every non-NULL source into dense minibatch tensors (for callers that want
 * materialised batches, e.g. the reference's own ppo_update).  obs rows are obs_bytes_per_agent
 * bytes; obs_out is int8 [B,W,H,C] when obs_out_f32 == 0, else float [B,W,H,C] (the reference's
 * dtype).  f32 sources/outputs: n_f32 <= 8 pairs (src_f32[i] [R] -> out_f32[i] [B], HOST arrays of
 * DEVICE pointers); int32 likewise (n_i32 <= 4, e.g. actions).  rows == NULL copies rows 0..B-1.  HBM-bound: 2*S*C (or 5*S*C with fp32 output) + 8 bytes per scalar field per row. */
int ocb_minibatch_gather(int device, const int32_t* rows, int B, int obs_bytes_per_agent, const int8_t* obs,
                         void* obs_out, int obs_out_f32, int n_f32, const float* const* src_f32, float* const* out_f32,
                         int n_i32, const int32_t* const* src_i32, int32_t* const* out_i32, void* stream);

typedef struct ocb_ppo_cfg {
    uint32_t struct_size;            /* sizeof(ocb_ppo_cfg) */
    int32_t use_clipped_value_loss;  /* config.py use_clipped_value_loss, default 1 */
    int32_t use_huber_loss;          /* default 1 */
    int32_t use_valuenorm;           /* default 1: ValueNorm.update(return_batch) then normalize (r_mappo.py:61-64) */
    int32_t use_value_active_masks;  /* default 1 (only matters with active_src) */
    int32_t use_policy_active_masks; /* default 1 (only matters with active_src) */
    float clip_param;                /* default 0.2 */
    float huber_delta;               /* default 10.0 */
    double vn_beta;                  /* ValueNorm beta, 0.99999 (valuenorm.py:11); double: the reference forms 1 - beta in Python */
    double vn_epsilon;               /* ValueNorm epsilon, 1e-5 */
} ocb_ppo_cfg;
#define OCB_PPO_STATS 16
/* cal_value_loss + the surrogate of ppo_update (r_mappo.py:52-89, 110-127): the forward losses and
 * the analytic gradients a backward pass starts from.  Inputs by minibatch position: logp_new,
 * entropy, values_new [B] (ocb_policy_evaluate's outputs).  Inputs by source row through `rows`
 * (NULL = identity): old_logp_src, adv_src, value_preds_src, returns_src, active_src (NULL = all
 * active; the *_active_masks options then reduce to plain means).  vn_state: DEVICE float[3] =
 * ValueNorm (running_mean, running_mean_sq, debiasing_term), UPDATED in place with this batch's
 * returns before normalising, as the reference does (ignored when use_valuenorm == 0).
 * Outputs (DEVICE; the first three may be NULL): imp_weights [B]; dlogp [B] = d policy_loss /
 * d logp_new; dvalues [B] = d value_loss / d values_new (torch.autograd's tie conventions);
 * stats double[OCB_PPO_STATS]: [0] policy_loss, [1] value_loss, [2] dist_entropy, [3] mean
 * imp_weight, [4] sum of active masks, [5] batch return mean, [6] batch return sq-mean, [7] B;
 * [8..15] scratch.  Per-element arithmetic in fp32 like torch, reductions in fp64.  One memset
 * and two launches, no host synchronisation. */
int ocb_ppo_loss(int device, const ocb_ppo_cfg* cfg, int B, const int32_t* rows, const float* logp_new,
                 const float* entropy, const float* values_new, const float* old_logp_src, const float* adv_src,
                 const float* value_preds_src, const float* returns_src, const float* active_src, float* vn_state,
                 float* imp_weights, float* dlogp, float* dvalues, double* stats, void* stream);

/* ------------------------------------------------------- Balance-Beam */
/* replaces BalanceBeamSimulator (src/balance_beam_env/mgr.cpp:191-233) behind
 * MadronaEnv.n_step / n_reset (vectorenv.py:306-343).
 *   actions [2,N] int32 in 0..3 (moves -2,-1,+1,+2; envs/balance_beam_env.py:14)
 *   obs     [2,N,7] int32, reward [2,N] float32, done [N] int32. */
int bb_create(int device, uint32_t num_worlds, uint64_t seed, bb_env** out);
int bb_destroy(bb_env* env);
int bb_num_worlds(const bb_env* env);
int bb_reset(bb_env* env, int32_t* obs, void* stream);
int bb_observe(bb_env* env, int32_t* obs, void* stream);
int bb_step(bb_env* env, const int32_t* actions, int32_t* obs, float* reward, int32_t* done, void* stream);
int bb_rollout_random(bb_env* env, int K, int32_t* obs_slab, float* reward, int32_t* done, uint8_t* actions_out,
                      void* stream);
/* packed state int32 [N,8]: loc0, loc1, time, hist0[t-1], hist0[t-2], hist1[t-1], hist1[t-2], episode */
int bb_get_state(bb_env* env, int32_t* h_state, size_t n_ints);
int bb_set_state(bb_env* env, const int32_t* h_state, size_t n_ints);

#ifdef __cplusplus
}
#endif
#endif /* OCB_H_ */
