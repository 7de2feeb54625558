// rollout_fused.cuh — a whole T-step self-play or cross-play rollout in ONE persistent launch (included by
// policy_kernels.cu inside its anonymous namespace, after the pair kernel whose roles it reuses).
// Variants (FusedParams): one or two world tiles in flight per CTA (`slots`), split mode (the critic's conv stream deferred
// behind the actor's; one tile in flight, whole grid resident in TMEM), cross-play (`cross`: two actors, seat-selected rows),
// population self-play (`kPop`: the actor + critic of a weight set chosen per 128-world slice), mixed play (`kMix`: the
// actors of two weight sets, a per-row draw picks which one acts, only the forced worlds are recorded).
//
// The 2T+1-launch rollout (ocb_rollout_policy) is bound by its dependent launches: per env step a
// policy launch and an env launch, each of which fills and drains the GPU for one tile per SM.
// Here a CTA owns a tile of 64 worlds (= 128 agent rows: seat 0 rows 0-63, seat 1 rows 64-127) for
// all T steps and nothing leaves the SM between the env step and the policy forward:
//   * two env warps (one world per lane) keep the world state in registers / shared memory and the
//     2 x 64 observation planes resident in shared memory (oc_core.cuh, as in oc_rollout_kernel);
//     per step they wait for the tile's sampled actions, run the transition, rewrite the touched
//     plane bytes and stream the planes to the PPO buffer with TMA bulk stores;
//   * the loader warps of the policy pipeline read the planes straight from shared memory (no HBM
//     / L2 round trip of the observations) and feed the tcgen05 conv as in policy_pair_kernel;
//   * MMA issuer and weight producer are the pair kernel's roles, running over "virtual tiles"
//     (world tile k, step u), u = 0..T (u = T is the bootstrap value pass);
//   * the actor epilogue group samples the 128 actions, writes them (and log-probs, values) to the
//     buffer and hands them to the env warps through shared memory + an mbarrier.
// Bit-identical to the 2T+1-launch path: same MMA sequence per row tile, same sampling counters
// (row = seat * N + world, offset = device step counter + u).
#pragma once

struct FusedParams {
    PolicyParams pol;    // blobs of the selected policy, geometry, pair_ring, sampling parameters
    RolloutParams env;   // tables, template, world state arrays, N, use_tma
    int T;
    int wtiles;          // ceil(N / 64) world tiles
    int8_t* obs_slab;    // [T+1][2][N][SC] or nullptr (evaluation rollouts keep no trajectory)
    int32_t* actions;    // [T][2][N] or nullptr
    float* logp;         // [T][2][N] or nullptr
    float* values;       // [T+1][2][N] or nullptr (cross-play: no critic)
    int32_t* reward;     // [T][2][N] or nullptr
    int32_t* done;       // [T][N] or nullptr
    int vec_loader;      // loaders read the planes as 16-byte vectors (conflict-free) instead of 4-byte words
    int col_ring;        // grid columns resident in the cell region: W in split mode (whole grid), else kColRing
    // Two world tiles in flight (slots = 2): the CTA owns tiles (2c, 2c + 1), (2c + 2 gridDim, ...) and the policy pipeline
    // runs over the interleaved stream (A, u), (B, u), (A, u + 1), (B, u + 1), ... — every role works on tile B while tile A's
    // env step runs and vice versa.  One env step of one tile is a dependent chain of ~20 k cycles in which each role is busy
    // a third of the time; a second tile fills the other two thirds.  No extra tensor memory: the stream reuses every TMEM
    // region in order exactly as consecutive steps of one tile do; it costs the second tile's planes in shared memory (the FC
    // weights then stream through a smaller ring) and only pays when there are more tiles than SMs.
    int slots;
    // Cross-play (pol.tile_policy set, xd_player.py:190-207 / partner_agents.py:97-111): seat-0 rows act with the actor of
    // policy tile_policy[seat-0 tile], seat-1 rows with the actor of tile_policy[seat-1 tile]; both actors run over all 128
    // rows of the tile as the pipeline's "two networks" and each epilogue group emits the rows of its seat.  No critic.
    // Population self-play (kernel instances with kPop, pol.f_seat1_tiles = 0) is not `cross`: the two networks are the
    // actor and critic of the slice's weight set and every row is emitted, as in self-play.
    int cross;
    // Mixed play (kernel instances with kMix, T = 2 L, mixed_schedule.h): network 0 is the actor of the main weight set
    // (pol.blobs), network 1 the actor at mix_partner_blobs.  Row r = seat N + n of world j = n mod (L - 1) plays main at step
    // u if the world is forced (mix_forced_main) or the mask draw says so (!mix_draw_partner(mix_seed, r, step)), else the
    // partner; epilogue group 0 emits the main rows (and the rows past N), group 1 the partner rows, the partner sampling
    // with key mix_partner_seed.  Only forced worlds are recorded, at slot mix_record_slot of the [L, 2, N] buffers: group 0
    // writes their actions and log-probs, the env warps their observation, reward and done.  No critic, nothing at u = T.
    int mix_L;
    unsigned long long mix_seed, mix_partner_seed;
    const uint8_t* mix_partner_blobs;
};

constexpr int kFEnvWarps = 2;
constexpr int kFWarpConvC = kPWarpProd + 1;                 // warp 21: conv issuer of the critic (split mode; warps 16 / 17 issue the actor's)
constexpr int kFWarpEnv = kFWarpConvC + 1;                  // warps 22, 23
constexpr int kFThreads = 32 * (kFWarpEnv + kFEnvWarps);    // 768
constexpr int kFWorlds = 32 * kFEnvWarps;                   // worlds per CTA tile
constexpr int kFMaxColRing = 6;  // 192 cell columns / (8 columns x H = 4)
enum : int {
    FB_OBS_FULL = PB_COUNT,      // [2 slots] env warps (64 arrivals) -> loaders: planes of the slot's next virtual tile are complete
    FB_OBS_EMPTY = PB_COUNT + 2, // [2] loaders (256 arrivals) -> env warps: the slot's planes have been consumed
    FB_ACT_FULL = PB_COUNT + 4,  // [2] the epilogue threads that sample the tile's 128 actions (128 arrivals) -> env warps
    FB_COL_FULL = PB_COUNT + 6,  // [6] split mode: loader -> both conv issuers (128 arrivals)
    FB_COL_EMPTY = FB_COL_FULL + kFMaxColRing,  // [6] split mode: both conv issuers' commits (2) -> loader
    FB_COUNT = FB_COL_EMPTY + kFMaxColRing
};
static_assert((int)FB_COUNT <= (int)PB_TMEM_SLOT, "barrier block overflow");

struct FusedSmemLayout {
    int head, wring, bars, act, tables, tmpl, envw;
    int view_stride, env_warp_bytes, slot_bytes, total;
};
__host__ __device__ inline FusedSmemLayout fused_smem_layout(int npos, int ring, int S, int SC, int slots) {
    FusedSmemLayout s;
    const BlobLayout L = blob_layout(npos);
    int o = 0;
    s.head = o, o += kPRestOff + 2 * (L.head_bytes - L.bias1);
    s.wring = o, o += ring * kChunk;
    s.bars = o, o += 1024;
    s.act = o, o += 2 * 128;  // the sampled actions of a slot's tile, one byte per agent row
    s.tables = o, o += (int)align16(sizeof(Tables));
    s.tmpl = o, o += (int)align16((size_t)SC);
    s.envw = o;
    s.view_stride = (int)align16((size_t)32 * SC);
    s.env_warp_bytes = 2 * s.view_stride + (int)align16((size_t)S * 32 * 2);
    s.slot_bytes = kFEnvWarps * s.env_warp_bytes;
    o += slots * s.slot_bytes;
    s.total = o + 128;
    return s;
}

// The CTA's stream of virtual tiles: rounds of `slots` world tiles, T + 1 steps each, the tiles of a round interleaved step by
// step.  Every role walks the same cursor (a slot without a tile — only possible in the last round — is skipped).
struct FusedCursor {
    int kt0, u, s, T, wtiles, stride, slots;
    bool two;
    __device__ __forceinline__ FusedCursor(const FusedParams& fp)
        : kt0((int)blockIdx.x * fp.slots), u(0), s(0), T(fp.T), wtiles(fp.wtiles), stride((int)gridDim.x * fp.slots), slots(fp.slots) {
        two = slots == 2 && kt0 + 1 < wtiles;
    }
    __device__ __forceinline__ int kt() const { return kt0 + s; }
    __device__ __forceinline__ void next() {
        if (two && s == 0) {
            s = 1;
            return;
        }
        s = 0;
        if (++u > T) u = 0, kt0 += stride, two = slots == 2 && kt0 + 1 < wtiles;
    }
};
__host__ __device__ inline int fused_virtual_tiles(int wtiles, int slots, int grid, int cta, int T) {
    int n = 0;
    for (int kt0 = cta * slots; kt0 < wtiles; kt0 += grid * slots) n += ((slots == 2 && kt0 + 1 < wtiles) ? 2 : 1) * (T + 1);
    return n;
}

// loaders: shared-memory planes -> bf16 cell blocks in TMEM.  Thread (lw, lane) owns row 32 lw + lane
// = seat lw / 2, env warp lw % 2, world `lane`; the two groups take alternate columns of the stream.
template <bool kProf, bool kSplit>
__device__ __forceinline__ void fused_loader_role(const FusedParams& fp, uint32_t nvt, uint32_t tmem, const uint8_t* s_env,
                                                  const FusedSmemLayout& sl, uint32_t bars) {
    const int lwarp = (threadIdx.x >> 5) - kEpiWarps, lg = lwarp >> 2, lw = lwarp & 3, lane = threadIdx.x & 31;
    const int W = fp.pol.W, H = fp.pol.H, seg = 5 * H;
    const uint32_t* myrow0 = reinterpret_cast<const uint32_t*>(s_env + (lw & 1) * sl.env_warp_bytes + (lw >> 1) * sl.view_stride +
                                                               lane * fp.pol.SC);
    const uint32_t* myrow = myrow0;
    const uint32_t tcells = tmem + ((uint32_t)(lw * 32) << 16) + kColCells;
    const uint32_t ncols = nvt * (uint32_t)W;
    uint32_t lt = 0;  // virtual tile of the column
    int lx = lg;      // grid column inside it
    bool fresh = true;  // first column of this group in tile lt
    FusedCursor cur(fp);
    uint32_t seen[2] = {0, 0};  // virtual tiles of each slot consumed so far (phase of the slot's barriers)
    for (uint32_t gc = lg; gc < ncols; gc += 2) {
        if (fresh) {
            myrow = myrow0 + cur.s * (sl.slot_bytes >> 2);
            mbar_wait(bars + 8 * (FB_OBS_FULL + cur.s), (cur.s ? seen[1] : seen[0]) & 1);
            if (kProf && lwarp == 0) trace_ev<kProf>(fp.pol, (int)lt, 8);
        }
        const bool first_col = fresh;
        fresh = false;
        const uint32_t ring = kSplit ? (uint32_t)fp.col_ring : (uint32_t)kColRing;
        const int slot = gc % ring;
        if (gc >= ring) {
            mbar_wait(bars + 8 * ((kSplit ? FB_COL_EMPTY : PB_COL_EMPTY) + slot), ((gc / ring) - 1) & 1);
            tc_fence_after();
        }
        if (fp.vec_loader) {
            // The 20 H bytes of this row's grid column, read as 16-byte vectors from the enclosing aligned range: rows are SC
            // bytes apart (100 / 125 / 225 words), so 4-byte loads of a warp hit 4-way bank conflicts while 16-byte loads are
            // conflict-free; eight loader warps on 4-byte loads alone kept the shared-memory pipe busy for ~650 cycles per
            // column pair (tools/fused_trace.py).  `r` = words the column starts after the aligned address.
            const uint32_t* colp = myrow + lx * seg;
            const int r = (int)((reinterpret_cast<uintptr_t>(colp) >> 2) & 3);  // per lane when SC is not a multiple of 16
            const uint4* src4 = reinterpret_cast<const uint4*>(colp - r);
            constexpr int kMaxVec = (5 * kMaxH + 3 + 3) / 4;  // 9
            const int nvec = (seg + r + 3) >> 2;
            uint32_t c[4 * kMaxVec];
    #pragma unroll
            for (int i = 0; i < kMaxVec; ++i) {
                if (i < nvec) {
                    const uint4 q = src4[i];
                    c[4 * i] = q.x, c[4 * i + 1] = q.y, c[4 * i + 2] = q.z, c[4 * i + 3] = q.w;
                } else {
                    c[4 * i] = c[4 * i + 1] = c[4 * i + 2] = c[4 * i + 3] = 0u;
                }
            }
            auto word = [&](int k) -> uint32_t {  // word k of the column = c[k + r], r in 0..3 (static register indices)
                const uint32_t a = (r & 1) ? c[k + 1] : c[k], b = (r & 1) ? c[k + 3] : c[k + 2];
                return (r & 2) ? b : a;
            };
    #pragma unroll
            for (int y = 0; y < kMaxH; ++y) {
                if (y < H) {
                    uint32_t w[5];
    #pragma unroll
                    for (int q = 0; q < 5; ++q) w[q] = word(y * 5 + q);
                    const uint4 c0 = make_uint4(bytes_bf16x2(w[0], pair_sel(0, 1)), bytes_bf16x2(w[0], pair_sel(2, 3)),
                                                bytes_bf16x2(w[1], pair_sel(0, 1)), bytes_bf16x2(w[1], pair_sel(2, 3)));
                    const uint4 c1 = make_uint4(bytes_bf16x2(w[2], pair_sel(0, 1)), bytes_bf16x2(w[4], pair_sel(0, 1)),
                                                bytes_bf16x2(w[4], pair_sel(2, 3)), bytes_bf16x2(w[3], pair_sel(3, 4)));
                    tmem_st8(tcells + (slot * H + y) * kCellCols, c0, c1);
                }
            }
        } else {
            const uint32_t* mine = myrow + lx * seg;
            for (int y = 0; y < H; ++y) {
                uint32_t w[5];
#pragma unroll
                for (int q = 0; q < 5; ++q) w[q] = mine[y * 5 + q];
                const uint4 c0 = make_uint4(bytes_bf16x2(w[0], pair_sel(0, 1)), bytes_bf16x2(w[0], pair_sel(2, 3)),
                                            bytes_bf16x2(w[1], pair_sel(0, 1)), bytes_bf16x2(w[1], pair_sel(2, 3)));
                const uint4 c1 = make_uint4(bytes_bf16x2(w[2], pair_sel(0, 1)), bytes_bf16x2(w[4], pair_sel(0, 1)),
                                            bytes_bf16x2(w[4], pair_sel(2, 3)), bytes_bf16x2(w[3], pair_sel(3, 4)));
                tmem_st8(tcells + (slot * H + y) * kCellCols, c0, c1);
            }
        }
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(bars + 8 * ((kSplit ? FB_COL_FULL : PB_COL_FULL) + slot));
        if (kProf && lwarp == 0 && first_col) trace_ev<kProf>(fp.pol, (int)lt, 9);
        if (kProf && lw == 0 && lx >= 1 && lx <= 4) trace_ev<kProf>(fp.pol, (int)lt, 3 + lx);  // grid columns 1..4 in tensor memory
        lx += 2;
        if (lx >= W) {  // this group's last column of the tile: its plane reads are done
            mbar_arrive(bars + 8 * (FB_OBS_EMPTY + cur.s));
            if (kProf && lwarp == 0) trace_ev<kProf>(fp.pol, (int)lt, 10);
            if (cur.s) ++seen[1]; else ++seen[0];
            cur.next();
            lx -= W, ++lt, fresh = true;
        }
    }
}

// env warps: one world per lane and slot, state in registers / shared memory across the T steps.  With two tiles in flight the
// same two warps serve both slots in stream order (A, u), (B, u), (A, u + 1), ...: a slot's env step takes a sixth of its
// policy pass, so the warps are idle most of the time either way.
__device__ __forceinline__ void bulk_wait_read_1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }

template <int P>
struct FusedSlot {
    World<P> w;
    int cur_return, ep_add;
    long long ret_add;
    int n, nbytes;
    int j;  // kMix: world index inside its replica (n mod (L - 1))
    bool valid, tma_ok, tma_pending;
    int8_t* obs_ptr;
    int32_t *rew_ptr, *done_ptr;
    uint32_t vts, acts;  // virtual tiles / action hand-offs of this slot so far (barrier phases); never reset
};

template <bool kProf, int kSlots, bool kMix = false>
__device__ __forceinline__ void fused_env_role(const FusedParams& fp, uint8_t* s_env, const FusedSmemLayout& sl, const Tables& tb,
                                               const uint8_t* tmpl, const uint8_t* s_act, uint32_t bars) {
    constexpr int P = 2;
    const int ew = (threadIdx.x >> 5) - kFWarpEnv, lane = threadIdx.x & 31;
    const Consts c = load_consts(tb);
    const int SC = tb.SC, N = fp.env.N, T = fp.T;
    const int view_stride = sl.view_stride;
    const size_t PN = (size_t)P * N, obs_view_stride = (size_t)N * SC, obs_step_stride = PN * SC;
    const bool store_obs = fp.obs_slab != nullptr;

    FusedSlot<P> sa, sb;  // slot 0 / slot 1 (two named objects: an array of them ends up in local memory)
    // One tile in flight: the step time IS the chain env -> loaders -> conv -> FC -> head -> sampling, so the env warps compute
    // everything of the next transition that depends on the state only (step_pre, oc_core.cuh) while the policy forward
    // runs, and only pick among those outcomes once the actions arrive (step_post).  With two tiles in flight the other
    // tile's policy pass hides the transition, and the outcomes of two slots would have to stay in registers.
    StepPre2 pre;
    sa.vts = sa.acts = sb.vts = sb.acts = 0;
    sa.tma_pending = sb.tma_pending = false;

    // `slot` is a literal at both call sites
    auto planes_of = [&](int slot) { return s_env + slot * sl.slot_bytes + ew * sl.env_warp_bytes; };  // [P][32][SC]
    auto objs_of = [&](int slot) { return reinterpret_cast<uint16_t*>(planes_of(slot) + (size_t)P * view_stride) + lane; };  // [S][32]

    auto begin_tile = [&](FusedSlot<P>& q, int slot, int kt) {
        const int n0 = kt * kFWorlds + ew * 32;
        q.n = n0 + lane;
        q.valid = q.n < N;
        const int nl = q.valid ? q.n : N - 1;
        q.nbytes = max(0, min(32, N - n0)) * SC;
        q.obs_ptr = store_obs ? fp.obs_slab + (size_t)n0 * SC : nullptr;
        q.tma_ok = store_obs && fp.env.use_tma && q.nbytes > 0 && ((q.nbytes & 15) == 0) &&
                   ((reinterpret_cast<uintptr_t>(q.obs_ptr) & 15u) == 0) && ((obs_view_stride & 15u) == 0);
        q.rew_ptr = fp.reward ? fp.reward + q.n : nullptr;
        q.done_ptr = fp.done ? fp.done + q.n : nullptr;
        if constexpr (kMix) {  // per-world stores of SC bytes: 16-byte aligned exactly when SC is
            q.j = q.n % (fp.mix_L - 1);
            q.tma_ok = store_obs && fp.env.use_tma && (SC & 15) == 0 && (reinterpret_cast<uintptr_t>(fp.obs_slab) & 15u) == 0;
        }
        load_world<P, 1, 8>(tb, c, fp.env, nl, 0, objs_of(slot), q.w);
        q.cur_return = fp.env.cur_return[nl];
        q.ret_add = 0, q.ep_add = 0;
    };

    // `other_pending`: the other slot has a bulk store in flight that was committed AFTER this slot's last one
    auto step_tile = [&](FusedSlot<P>& q, int slot, int u, bool other_pending) {
        uint8_t* planes = planes_of(slot);
        uint16_t* myobjs = objs_of(slot);
        uint8_t* myplanes = planes + lane * SC;
        bool full = true;
        int oldslot[P] = {0, 0};
        uint32_t dirty[P] = {0xFFFFFFFFu, 0xFFFFFFFFu};
        uint32_t ticked = 0;
        // the planes still hold the slot's previous virtual tile: its loaders and its bulk store must be done with them (both
        // finish long before the actions arrive, so these waits sit before the action wait, off the critical path)
        if (q.vts > 0) mbar_wait(bars + 8 * (FB_OBS_EMPTY + slot), (q.vts - 1) & 1);
        if (q.tma_pending) {
            if (kMix) {
                bulk_wait_read_all();  // every lane stores its own world's planes
            } else if (lane == 0) {
                if (other_pending)
                    bulk_wait_read_1();  // all but the newest group: the other slot's store may go on reading ITS planes
                else
                    bulk_wait_read_all();
            }
            q.tma_pending = false;
        }
        if (u > 0) {
            // the cells the players stand on are cleared now, while the actions are still being computed (one lane owns all
            // views of its world, so nothing has to be ordered against other lanes); an episode end overwrites them anyway
            __syncwarp();  // lane 0's wait for the bulk store above covers the warp
#pragma unroll
            for (int i = 0; i < P; ++i) oldslot[i] = q.w.slot[i];
            obs_phase1<P, 1>(tb, myplanes, view_stride, tmpl, false, 0, oldslot);
            mbar_wait(bars + 8 * (FB_ACT_FULL + slot), q.acts & 1);
            if (kProf && ew == 0) trace_ev<kProf>(fp.pol, (int)q.vts, 0);
            ++q.acts;
            int act[P];
            act[0] = s_act[slot * 128 + ew * 32 + lane], act[1] = s_act[slot * 128 + kFWorlds + ew * 32 + lane];
            int r;
            if constexpr (kSlots == 1)
                r = step_post(tb, c, q.w, myobjs, 32, act, pre, dirty, ticked);
            else
                r = step_world<P>(tb, c, q.w, myobjs, 32, act, dirty, ticked);
            const bool done = q.w.timestep >= c.horizon;
            q.cur_return += r;
            if (done) {
                q.ret_add += q.cur_return;
                q.ep_add += 1;
                q.cur_return = 0;
                reset_world<P>(tb, q.w);
                for (int idx = 0; idx < c.n_objcells; ++idx) myobjs[(int)tb.objcells[idx] * 32] = 0;
            }
            if constexpr (kMix) {  // the transition of step u - 1: recorded at the forced world's slot of that step
                if (q.valid && mix_forced_main(fp.mix_L, u - 1, q.j)) {
                    const size_t t = (size_t)mix_record_slot(fp.mix_L, u - 1, q.j);
                    if (fp.reward != nullptr) fp.reward[t * PN + q.n] = r, fp.reward[t * PN + N + q.n] = r;
                    if (fp.done != nullptr) fp.done[t * N + q.n] = done ? 1 : 0;
                }
            } else {
                if (q.rew_ptr != nullptr) {
                    if (q.valid) q.rew_ptr[0] = r, q.rew_ptr[N] = r;
                    q.rew_ptr += PN;
                }
                if (q.done_ptr != nullptr) {
                    if (q.valid) *q.done_ptr = done ? 1 : 0;
                    q.done_ptr += N;
                }
            }
            full = done;
            if (kProf && ew == 0) trace_ev<kProf>(fp.pol, (int)q.vts, 1);
        }
        __syncwarp();
        if (kProf && ew == 0) trace_ev<kProf>(fp.pol, (int)q.vts, 2);
        if (full) obs_phase1<P, 1>(tb, myplanes, view_stride, tmpl, true, 0, oldslot);  // (else: cleared before the action wait)
        obs_phase2<P, 1>(tb, c, myplanes, view_stride, myobjs, 32, full, 0, q.w, dirty, ticked);
        mbar_arrive(bars + 8 * (FB_OBS_FULL + slot));  // release: the loaders may read this lane's planes
        if (kProf && ew == 0) trace_ev<kProf>(fp.pol, (int)q.vts, 3);
        ++q.vts;
        if (kMix && store_obs) {
            // the observation a forced world acts on, at its slot of this step (u = T: no step, no record)
            const bool rec = q.valid && u < T && mix_forced_main(fp.mix_L, u, q.j);
            int8_t* dst = rec ? fp.obs_slab + ((size_t)mix_record_slot(fp.mix_L, u, q.j) * PN + q.n) * SC : nullptr;
            if (q.tma_ok) {
                if (rec) {
                    fence_proxy_async_smem();
#pragma unroll
                    for (int v = 0; v < P; ++v)
                        bulk_store_s2g(dst + v * obs_view_stride, smem_addr(myplanes) + v * view_stride, (uint32_t)SC);
                    bulk_commit();
                }
                q.tma_pending = true;
            } else {
                // word copies, the warp on one world at a time (SC is a multiple of 4; rows are 4-byte aligned only)
                __syncwarp();
                for (uint32_t todo = __ballot_sync(0xFFFFFFFFu, rec); todo != 0u; todo &= todo - 1u) {
                    const int b = __ffs(todo) - 1;
                    int8_t* d = reinterpret_cast<int8_t*>(__shfl_sync(0xFFFFFFFFu, reinterpret_cast<unsigned long long>(dst), b));
#pragma unroll
                    for (int v = 0; v < P; ++v) {
                        const uint32_t* s4 = reinterpret_cast<const uint32_t*>(planes + v * view_stride + b * SC);
                        uint32_t* d4 = reinterpret_cast<uint32_t*>(d + v * obs_view_stride);
                        for (int w4 = lane; w4 < (SC >> 2); w4 += 32) __stcs(d4 + w4, s4[w4]);
                    }
                }
            }
        } else if (store_obs) {
            int8_t* dst = q.obs_ptr + (size_t)u * obs_step_stride;
            if (q.tma_ok) {
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) {
#pragma unroll
                    for (int v = 0; v < P; ++v)
                        bulk_store_s2g(dst + v * obs_view_stride, smem_addr(planes) + v * view_stride, (uint32_t)q.nbytes);
                    bulk_commit();
                }
                q.tma_pending = true;
            } else if (q.nbytes > 0) {
                __syncwarp();
#pragma unroll
                for (int v = 0; v < P; ++v) warp_copy_out(dst + v * obs_view_stride, planes + v * view_stride, q.nbytes, lane);
            }
        }
        if constexpr (kSlots == 1) step_pre(tb, c, q.w, myobjs, 32, pre);  // for the next step, off the critical path
    };

    // world state back to HBM (the next launch, or ocb_get_state, continues from it)
    auto end_tile = [&](FusedSlot<P>& q, int slot) {
        if (q.valid) {
            fp.env.players[q.n] = player_pack(q.w.pos[0], q.w.orient[0], q.w.held[0]);
            fp.env.players[(size_t)N + q.n] = player_pack(q.w.pos[1], q.w.orient[1], q.w.held[1]);
            store_world_objs<1>(tb, c, fp.env, q.n, 0, objs_of(slot));
            fp.env.timestep[q.n] = q.w.timestep;
            fp.env.cur_return[q.n] = q.cur_return;
            if (q.ep_add) {
                fp.env.ret_sum[q.n] += q.ret_add;
                fp.env.episodes[q.n] += q.ep_add;
            }
        }
        __syncwarp();
    };

    for (int kt0 = (int)blockIdx.x * kSlots; kt0 < fp.wtiles; kt0 += (int)gridDim.x * kSlots) {
        const bool two = kSlots == 2 && kt0 + 1 < fp.wtiles;
        begin_tile(sa, 0, kt0);
        if (kSlots == 2 && two) begin_tile(sb, 1, kt0 + 1);
        for (int u = 0; u <= T; ++u) {
            step_tile(sa, 0, u, kSlots == 2 && two && sb.tma_pending);
            if (kSlots == 2 && two) step_tile(sb, 1, u, sa.tma_pending);
        }
        end_tile(sa, 0);
        if (kSlots == 2 && two) end_tile(sb, 1);
    }
    if ((sa.tma_pending || (kSlots == 2 && sb.tma_pending)) && (kMix || lane == 0)) bulk_wait_read_all();
}

// output stage of the epilogue in the fused rollout.  `net` = 0: six logits of the tile's rows, 1: head[0] = value.
// Cross-play: both pipeline networks are actors; group 0 (net 0) owns the rows of seat 0, group 1 those of seat 1.
// Mixed play (kMix): both are actors too; group 1 owns the rows the partner plays at this step, group 0 all others.
template <bool kMix = false>
struct FusedOut {
    const FusedParams& fp;
    uint8_t* s_act;
    uint32_t bars;
    unsigned long long base;
    FusedCursor cur;
    int g;
    bool partner_row;  // kMix: the partner plays this thread's row of the current virtual tile (set by draw)
    __device__ __forceinline__ FusedOut(const FusedParams& f, uint8_t* sa, uint32_t b) : fp(f), s_act(sa), bars(b), cur(f) {
        base = f.pol.offset;
        if (f.pol.d_offset != nullptr) base += *f.pol.d_offset;
        g = (int)(threadIdx.x >> 7);  // epilogue group of this thread
        partner_row = false;
    }
    __device__ __forceinline__ bool mine(int trow_id) const {
        if constexpr (kMix)
            return partner_row == (g == 1);
        else
            return !fp.cross || (trow_id >> 6) == g;
    }
    // mixed_schedule.h, with the per-step path's counters (mask step = sampling offset = step counter + u); every row of the
    // tile is claimed by exactly one group, or FB_ACT_FULL never completes: rows past N and the pass u = T go to group 0
    __device__ __forceinline__ bool mix_partner_plays(int trow_id) const {
        const int n = cur.kt() * kFWorlds + (trow_id & (kFWorlds - 1)), seat = trow_id >> 6;
        if (n >= fp.env.N || cur.u >= fp.T || mix_forced_main(fp.mix_L, cur.u, n % (fp.mix_L - 1))) return false;
        return mix_draw_partner(fp.mix_seed, (uint32_t)(seat * fp.env.N + n), base + (unsigned long long)cur.u);
    }
    __device__ __forceinline__ uint32_t draw(int, int trow_id) {
        if constexpr (kMix) partner_row = mix_partner_plays(trow_id);
        if (fp.pol.deterministic || cur.u >= fp.T || !mine(trow_id)) return 0u;
        const int wl = trow_id & (kFWorlds - 1), seat = trow_id >> 6;
        const long long row = (long long)seat * fp.env.N + (cur.kt() * kFWorlds + wl);
        if constexpr (kMix) {
            if (g == 1) {  // the partner samples from its own stream: same counters, another key
                PolicyParams kp = fp.pol;
                kp.seed = fp.mix_partner_seed;
                return policy_draw(kp, (uint32_t)row, base + (unsigned long long)cur.u);
            }
        }
        return policy_draw(fp.pol, (uint32_t)row, base + (unsigned long long)cur.u);
    }
    __device__ __forceinline__ void operator()(int, int trow_id, int net, const float (&head)[6], uint32_t drawn) {
        const int N = fp.env.N, wl = trow_id & (kFWorlds - 1), seat = trow_id >> 6, u = cur.u;
        const int n = cur.kt() * kFWorlds + wl;
        const long long row = (long long)seat * N + n;               // row of one step's [2][N] block
        const long long store = (long long)u * 2 * N + row;
        if (net == 1) {
            if (n < N && fp.values != nullptr) fp.values[store] = head[0];
        } else if (u < fp.T && mine(trow_id)) {
            PolicyParams op = fp.pol;  // output pointers of this step; rows past N sample but store nothing
            const bool valid = n < N;
            bool rec = valid;
            long long at = store;
            if constexpr (kMix) {  // a forced world's row (main's) lands at its slot; every other row stores nothing
                const int j = valid ? n % (fp.mix_L - 1) : 0;
                rec = valid && g == 0 && mix_forced_main(fp.mix_L, u, j);
                at = ((long long)mix_record_slot(fp.mix_L, u, j) * 2 + seat) * N + n;
            }
            op.actions = rec ? fp.actions : nullptr, op.logp = rec ? fp.logp : nullptr, op.logits = nullptr;
            emit_actor_row(op, at, (uint32_t)row, head, base + (unsigned long long)u, true, &drawn, s_act + cur.s * 128 + trow_id,
                           bars + 8 * (FB_ACT_FULL + cur.s));
        }
        cur.next();
    }
};

template <bool kProf, bool kSplit, int kSlots, bool kPop = false, bool kMix = false>
__global__ void __launch_bounds__(kFThreads, 1) rollout_fused_kernel(const FusedParams fp) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((128u - (smem_addr(smem_raw) & 127u)) & 127u);
    const int tid = threadIdx.x, warp = tid >> 5;
    const PolicyParams& prm = fp.pol;
    const BlobLayout L = blob_layout(prm.npos);
    const FusedSmemLayout sl = fused_smem_layout(prm.npos, prm.pair_ring, prm.S, prm.SC, fp.slots);
    uint8_t* s_head = smem + sl.head;
    uint8_t* s_wring = smem + sl.wring;
    uint64_t* s_bars = reinterpret_cast<uint64_t*>(smem + sl.bars);
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bars + PB_TMEM_SLOT);
    uint8_t* s_act = smem + sl.act;
    Tables* s_tables = reinterpret_cast<Tables*>(smem + sl.tables);
    uint8_t* s_tmpl = smem + sl.tmpl;
    uint8_t* s_env = smem + sl.envw;
    const uint32_t bars = smem_addr(s_bars);

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_addr(s_tmem)),
                     "r"((uint32_t)kTmemCols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 32) {
        for (int i = 0; i < FB_COUNT; ++i) {
            uint32_t count = 1;
            if ((i >= PB_COL_FULL && i < PB_COL_FULL + 4) || (i >= PB_A2_FULL && i < PB_A2_FULL + 2) ||
                (i >= PB_D3_EMPTY && i < PB_D3_EMPTY + 2))
                count = 128;
            if (i >= PB_COL_EMPTY && i < PB_COL_EMPTY + 4) count = 2;  // plain mode: two conv issuers
            if (i >= PB_HEAD_EMPTY && i < PB_HEAD_EMPTY + 2) count = 32 * kEpiWarps + (kSplit ? 3 : 2);
            if (i >= PB_D1_EMPTY && i < PB_D1_EMPTY + 2) count = 32 * kEpiWarps;
            if (i >= PBS_D1_EMPTY && i < PBS_D1_EMPTY + 4) count = 128;
            if (i >= FB_COL_FULL && i < FB_COL_FULL + kFMaxColRing) count = 128;
            if (i >= FB_COL_EMPTY && i < FB_COL_EMPTY + kFMaxColRing) count = 3;  // the actor's two issuers and the critic's one
            if (i >= FB_OBS_FULL && i < FB_OBS_FULL + 2) count = 32 * kFEnvWarps;
            if (i >= FB_OBS_EMPTY && i < FB_OBS_EMPTY + 2) count = 32 * kLoadWarps;
            if (i >= FB_ACT_FULL && i < FB_ACT_FULL + 2) count = 128;
            mbar_init(bars + 8 * i, count);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    {  // static layout tables and the observation template
        const uint32_t* src = reinterpret_cast<const uint32_t*>(fp.env.tables);
        uint32_t* dst = reinterpret_cast<uint32_t*>(s_tables);
        for (int i = tid; i < (int)(sizeof(Tables) / 4); i += kFThreads) dst[i] = src[i];
        for (int i = tid; i < prm.SC; i += kFThreads) s_tmpl[i] = fp.env.tmpl[i];
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *s_tmem;
    // virtual tiles of this CTA: (world tile, step u), u = 0..T, the tiles of a round interleaved (FusedCursor)
    const int nvt = fused_virtual_tiles(fp.wtiles, fp.slots, (int)gridDim.x, (int)blockIdx.x, fp.T);

    long long pw[kProf ? PW_COUNT : 1] = {};
    if (warp < kEpiWarps) {
        pair_epilogue_role<kProf, kSplit, kPop, kMix>(pw, prm, 0, nvt, L, tmem, s_head, bars, FusedOut<kMix>(fp, s_act, bars));
    } else if (warp < kWarpMma) {
        fused_loader_role<kProf, kSplit>(fp, (uint32_t)nvt, tmem, s_env, sl, bars);
    } else if (warp == kWarpMma || warp == kWarpConv2) {
        const int half = warp == kWarpMma ? 0 : 1;
        if (kSplit)
            pair_conv_role<kProf, 0>(pw, prm, 0, nvt, L, tmem, smem_addr(s_head), bars, half, 2, (uint32_t)fp.col_ring, FB_COL_FULL,
                                     FB_COL_EMPTY);
        else
            pair_conv_role<kProf, -1>(pw, prm, 0, nvt, L, tmem, smem_addr(s_head), bars, half, 2);
    } else if (warp == kPWarpProd) {
        pair_producer_role<kProf, kPop, kMix>(pw, prm, 0, nvt, L, smem_addr(s_head), smem_addr(s_wring), bars,
                                              kMix ? fp.mix_partner_blobs : nullptr);
    } else if (warp < kPWarpProd) {
        pair_fc_role<kProf, kSplit>(pw, prm, warp - kWarpFc, 0, nvt, L, tmem, smem_addr(s_wring), bars);
    } else if (warp == kFWarpConvC) {
        if (kSplit)
            pair_conv_role<kProf, 1>(pw, prm, 0, nvt, L, tmem, smem_addr(s_head), bars, 0, 1, (uint32_t)fp.col_ring, FB_COL_FULL,
                                     FB_COL_EMPTY);
    } else {
        fused_env_role<kProf, kSlots, kMix>(fp, s_env, sl, *s_tables, s_tmpl, s_act, bars);
    }
    __syncwarp();
    tc_fence_before();
    __syncthreads();
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)kTmemCols) : "memory");
}

// device step counter += k, after the rollout kernel (every CTA reads the counter at its start)
__global__ void counter_add_kernel(unsigned long long* ctr, unsigned long long k) { *ctr += k; }
