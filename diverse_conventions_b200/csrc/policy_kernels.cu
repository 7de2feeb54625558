// policy_kernels.cu — fused MAPPO actor / critic forward on the 5th-gen tensor cores.
//
// Network (reference: R_Actor / R_Critic with CNNBase, train/MAPPO/r_actor_critic.py:12-71,
// 142-197; train/MAPPO/utils/cnn.py:22-42; hidden 64 as in every train/*.sh):
//   obs int8 [M, W, H, C=20] -> Conv3x3(20->32) -> ReLU -> FC((W-2)(H-2)*32 -> 64) -> ReLU
//   -> FC(64->64) -> ReLU -> head (6 logits, orthogonal gain 0.01 | 1 value).
//
// One persistent, warp-specialised kernel (policy_pair_kernel, one CTA per SM) runs BOTH networks of
// every tile of 128 observation rows in the same CTA:
//   * loader warps (2 groups of 4, alternating grid columns): coalesced loads of one grid column
//     of the tile ([128 rows] x H cells x 20 B, software-prefetched in registers), transposed
//     through a small staging buffer into per-cell [128 x 16] bf16 K-major operand blocks held in
//     a ring of 4 grid columns (int8 -> bf16 is one PRMT + one HADD2.BF16 per channel pair).  The
//     convolution needs NO im2col: for output position (ox, oy) the k-slice of window cell
//     (dx, dy) is the block of cell (ox+dx, oy+dy), so the conv is 9 x (hi, lo) tcgen05.mma
//     per position pointing at different blocks; the 5 static terrain channels are folded into a
//     per-position bias on the host;
//   * two conv issuers (even / odd positions = the two accumulator stages) run one N = 64 conv
//     for both networks, one FC issuer per network issues its FC1 partial products and FC2;
//     accumulators live in TMEM (see the pair kernel's section below);
//   * epilogue warps (2 groups of 4, group g = network g): tcgen05.ld a conv position, bias + ReLU,
//     split into bf16 hi + lo and store it as the A operand of the FC1 partial product of that
//     position; FC2 flows through the same A stage as two more K=32 items fed from the FC1
//     accumulator; the tiny head (64 -> 6 | 1), softmax sampling and log-prob run in fp32 on CUDA cores;
//   * one producer thread streams the FC weights of both networks as 8 KB chunks with cp.async.bulk
//     (global -> shared, mbarrier complete_tx) into a ring; when the whole set fits the ring
//     the chunks stay resident and are only re-fetched when a tile selects another policy;
//   * single mode (ocb_policy_act / ocb_policy_value): one network per tile as one stream, both
//     epilogue groups on it, bit-identical to the two-network forward;
//   * precision: operands are bf16 hi+lo splits (x = hi + lo, 3 products, fp32 accumulate),
//     observations are exact in bf16, so logits agree with the fp32 reference to ~1e-5
//     relative (the 1e-3 bar of the north star is not reachable with plain bf16 operands);
//   * activations never touch HBM; per tile the kernel reads the tile's observations once.
// All inter-role hand-offs are mbarriers; waits are bounded spins that trap instead of hanging.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <new>
#include <vector>

#include "api_common.h"
#include "oc_core.cuh"
#include "oc_device.cuh"
#include "mixed_schedule.h"
#include "ocb.h"
#include "policy_internal.h"

using namespace ocb;

namespace {

constexpr int kRows = 128;     // rows (agents) per tile == UMMA M
constexpr int kHid = 64;       // hidden size
constexpr int kCo = 32;        // conv output channels (hidden / 2)
constexpr int kSlots = 16;     // bf16 slots per cell: channels 0-9, 16-19, 15, one zero pad
constexpr int kK1 = 9 * kSlots;  // conv K
constexpr int kCellCols = kSlots / 2;  // TMEM columns of one cell block
constexpr int kColRing = 4;    // grid columns resident per CTA (3 in use by the conv + 1 being loaded)
constexpr int kChunk = 8192;   // one FC weight chunk: [64 x 32] bf16 hi | lo
constexpr int kA2Cols = 32;    // TMEM columns of one FC A-operand stage: [128 x 32] bf16 hi (16) | lo (16)
constexpr int kMaxH = 6;       // a grid column must fit one warp-wide load (5*H words <= 32)
constexpr int kEpiWarps = 8;   // warps 0-7: two epilogue groups (group = warp / 4; TMEM lanes 32 (warp % 4) ..)
constexpr int kLoadWarps = 8;  // warps 8-15: two loader groups
constexpr int kWarpMma = kEpiWarps + kLoadWarps, kWarpProd = kWarpMma + 1;
constexpr int kThreads = 32 * (kWarpProd + 1);  // 576
constexpr int kTmemCols = 512;
// TMEM (32-bit columns x 128 lanes = rows of the tile): the cell blocks of the loaders start at column 0, two bf16 per column
constexpr int kColCells = 0;    // ring of 4 grid columns x H cells x 8 columns ([128 x 16] bf16 each), <= 192
constexpr int kSmemBudget = 227 * 1024 - 256;

// packed weight blob of one network: a resident "head" followed by 8 KB FC chunks
struct BlobLayout {
    int wc_hi, wc_lo;    // [32 x 144] bf16 canonical, 9216 B each
    int bias1;           // [npos][32] fp32 (conv bias + static terrain contribution)
    int b1, b2;          // [64] fp32
    int wh, bh;          // head weights fp32, 2 KB: actor [64][8] (hidden-major: unit i -> 6 logit weights + 2 zeros, two
                         // 16-byte loads per unit), critic [64] contiguous; bh [8] fp32
    int head_bytes;      // everything above (multiple of 128)
    int chunks;          // npos FC1 chunks + 2 FC2 chunks (K halves)
    int total;
};
__host__ __device__ inline int al128(int x) { return (x + 127) & ~127; }
__host__ __device__ inline BlobLayout blob_layout(int npos) {
    BlobLayout L;
    int o = 0;
    L.wc_hi = o, o += 9216;
    L.wc_lo = o, o += 9216;
    L.bias1 = o, o += al128(npos * kCo * 4);
    L.b1 = o, o += 256;
    L.b2 = o, o += 256;
    L.wh = o, o += 8 * kHid * 4;
    L.bh = o, o += 128;
    L.head_bytes = o;
    L.chunks = npos + 2;
    L.total = o + L.chunks * kChunk;
    return L;
}

struct PolicyParams {
    const uint8_t* blobs;     // [n_policies][2 nets][blob]
    size_t blob_stride;       // bytes between nets
    int W, H, S, SC, npos;
    const int8_t* obs;        // [M][SC]
    int M, tiles;             // critic pass over a rollout slab (policy_pair_kernel<kProf, true>): tiles = seat tiles per step
    const int32_t* tile_policy;  // [tiles] or nullptr
    const int32_t* row_index;    // [M] source row of each forward row (obs / given_actions are indexed by it) or nullptr
    const int32_t* given_actions;  // evaluate_actions: log-prob of the stored action of the source row instead of sampling
    float* entropy;              // [M] entropy of the action distribution, or nullptr
    float* logits;            // [M][6] or nullptr
    int32_t* actions;         // [M] or nullptr
    float* logp;              // [M] or nullptr
    float* values;            // [M] or nullptr
    int deterministic;
    unsigned long long seed, offset;
    const unsigned long long* d_offset;  // optional device-resident addend of `offset`
    // sampling rows of a sharded env (ocb_policy_set_sampling_rows): launch row r draws from counter row
    // r + (r < rng_rows_per_seat ? rng_add0 : rng_add1); all zero = the launch row itself
    unsigned int rng_rows_per_seat, rng_add0, rng_add1;
    int net_mask;             // 1 actor, 2 critic, 3 both (hidden 512: even CTAs actor, odd critic)
    int pair_ring;            // weight-ring slots in shared memory (chunks of both networks)
    int stage_stride;         // words per row of the loader staging buffer (odd)
    long long* prof;          // diagnostic build: [ctas][4 roles][PW_COUNT] stall cycles
    long long* trace;         // diagnostic build of the fused rollout: [trace_n steps][kTraceEvents] clock64 stamps of CTA 0
    int trace_u0, trace_n;    // first traced virtual tile (step) and number of traced steps
    int single;               // policy_pair_kernel: 0 = both networks of a tile, 1 = the actor only, 2 = the critic only (one stream)
    // fused rollout (rollout_fused.cuh): a CTA's virtual tiles come in rounds of f_vt_round = slots * (T + 1); with
    // tile_policy set (cross-play) the round's world tiles 2 c, 2 c + 1 play seat 0 / seat 1 with the actors of
    // tile_policy[kt / 2] / tile_policy[f_seat1_tiles + kt / 2] (the per-step path's seat-major 128-row tile table).
    // Population self-play (the kernel instances with kPop) sets f_seat1_tiles = 0 and a table by 128-world slice: fused_pair
    // gives p | p << 16 and the two networks are the actor and the critic of weight set p
    // The critic pass over a rollout slab (policy_pair_kernel<kProf, true>) sets f_slots = the slab's steps (SlabWalk).
    int f_vt_round, f_slots, f_seat1_tiles;
};

// barrier indices (8 bytes each) of loader_role's grid-column ring, the same in every kernel that runs it
enum : int {
    B_COL_FULL = 0,                      // [4]  loader -> MMA (128 arrivals)
    B_COL_EMPTY = 4,                     // [4]  MMA commit -> loader
};

// ---------------------------------------------------------------- PTX helpers
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// K-major, no-swizzle ("interleave") shared-memory matrix descriptor: 8-row x 16-byte core
// matrices; LBO = byte distance between the two K-chunks of one MMA, SBO = byte distance between
// 8-row groups (cute/arch/mma_sm100_desc.hpp: SmemDescriptor, version 1 on sm_100).
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) |
           (1ull << 46);
}
// instruction descriptor: D=f32, A=B=bf16, K-major both, dense (InstrDescriptor bit layout)
__device__ __forceinline__ uint32_t make_idesc(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// A operand from tensor memory ([128 lanes] x K/2 columns, two bf16 per column), B from shared memory
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, {%5, %6, %7, %8}, p;\n\t}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(db), "r"(idesc), "r"(accumulate), "r"(0u), "r"(0u), "r"(0u), "r"(0u)
        : "memory");
}
// registers -> TMEM: thread l of warp w writes lane 32(w%4)+l, 8 / 16 consecutive columns
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint4& a, const uint4& b) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(a.x),
                 "r"(a.y), "r"(a.z), "r"(a.w), "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w)
                 : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::
            "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint32_t mbar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(mbar) : "memory");
}
__device__ __forceinline__ void mbar_init(uint32_t mbar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t mbar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(mbar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t mbar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t parity) {
    // bounded spin: a pipeline that never signals traps instead of hanging the GPU
    for (uint32_t spins = 0;; ++spins) {
        uint32_t ok;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}\n"
            : "=r"(ok)
            : "r"(mbar), "r"(parity)
            : "memory");
        if (ok) return;
        if (spins > (1u << 24)) __trap();
    }
}
// wait that optionally accounts the stall cycles (diagnostic build of the kernel only)
template <bool kProf>
__device__ __forceinline__ void mbar_wait_p(uint32_t mbar, uint32_t parity, long long& acc) {
    if (kProf) {
        const long long t0 = clock64();
        mbar_wait(mbar, parity);
        acc += clock64() - t0;
    } else {
        mbar_wait(mbar, parity);
    }
}
// stall accounts written by ocb_policy_debug_profile: per CTA, per role, [0] = total cycles of the role
enum : int { PW_TOTAL = 0, PW_COL_EMPTY, PW_HEAD_FULL, PW_COL_FULL, PW_A2_FULL, PW_W_FULL, PW_D1_FULL, PW_D2_FULL,
             PW_A2_EMPTY, PW_D3_FULL, PW_HEAD_EMPTY, PW_W_EMPTY, PW_ISSUE_CONV, PW_ISSUE_FC, PW_LDG, PW_CVT, PW_COUNT = 16 };

// event trace of the fused rollout (ocb_rollout_fused_debug_trace): one clock64 stamp per (step, event) of CTA 0.
// Events: 0 env got actions | 1 env stepped | 2 env planes free | 3 env planes published | 8 loader sees planes |
// 9 loader first column done | 10 loader last column done | 16+p conv p issued | 24+j FC item j of the actor issued |
// 32+p epilogue (actor group) sees conv p | 40+j epilogue published item j | 48 D2 seen | 49 D3 seen | 50 head done |
// 51 actions handed to the env | 52 critic group sees D3 | 53 critic head done
constexpr int kTraceEvents = 64;
template <bool kProf>
__device__ __forceinline__ void trace_ev(const PolicyParams& prm, int vt, int ev) {
    if (kProf && prm.trace != nullptr && blockIdx.x == 0 && (threadIdx.x & 31) == 0) {
        const int s = vt - prm.trace_u0;
        if (s >= 0 && s < prm.trace_n && ev < kTraceEvents) prm.trace[s * kTraceEvents + ev] = clock64();
    }
}

// global -> shared bulk copy that completes `bytes` of transaction count on `mbar`
__device__ __forceinline__ void bulk_g2s(uint32_t sdst, const void* gsrc, uint32_t bytes, uint32_t mbar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(sdst),
                 "l"(gsrc), "r"(bytes), "r"(mbar)
                 : "memory");
}
// one lane of the (converged) warp; the tcgen05 / bulk-copy instructions below are issued under it so
// that the compiler keeps their operands in uniform registers instead of a per-lane waterfall loop
__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile(
        "{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\t"
        "elect.sync rx|px, 0xFFFFFFFF;\n\t"
        "selp.u32 %0, 1, 0, px;\n\t}\n"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// 32 lanes x 32 columns of fp32: thread l of warp w receives row 32w+l, columns col..col+31
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// (x0, x1) -> packed bf16 pair of the high parts and of the residuals: x = hi + lo
__device__ __forceinline__ void split2(float x0, float x1, uint32_t& hi, uint32_t& lo) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(x0, x1);  // .x = x0 (low half)
    hi = *reinterpret_cast<const uint32_t*>(&h);
    const float h0 = __uint_as_float(hi << 16), h1 = __uint_as_float(hi & 0xFFFF0000u);
    const __nv_bfloat162 l = __floats2bfloat162_rn(x0 - h0, x1 - h1);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}
// two observation bytes (each < 128) of `w` -> packed bf16 pair, exact: 0x43bb is bf16(128 + bb), so
// one byte permute builds (128 + b_i, 128 + b_j) and one packed subtract removes the 128s.
// `sel` picks byte i (0-3 of w; 4 = a zero byte) for the low half and byte j for the high half.
__device__ __forceinline__ uint32_t bytes_bf16x2(uint32_t w, uint32_t sel) {
    const uint32_t biased = __byte_perm(w, 0x00004300u, sel);
    const __nv_bfloat162 v = __hsub2(*reinterpret_cast<const __nv_bfloat162*>(&biased), __float2bfloat162_rn(128.0f));
    return *reinterpret_cast<const uint32_t*>(&v);
}
__host__ __device__ constexpr uint32_t pair_sel(int i, int j) { return (uint32_t)i | (5u << 4) | ((uint32_t)j << 8) | (5u << 12); }

// ---------------------------------------------------------------- unit iteration shared by all roles
struct UnitRange {
    int net, t0, t1;
};
__device__ __forceinline__ UnitRange my_units(const PolicyParams& prm) {
    UnitRange u;
    int c, g;
    if (prm.net_mask == 3) {
        u.net = blockIdx.x & 1, c = blockIdx.x >> 1, g = gridDim.x >> 1;
    } else {
        u.net = prm.net_mask == 1 ? 0 : 1, c = blockIdx.x, g = gridDim.x;
    }
    u.t0 = (int)(((long long)c * prm.tiles) / g);
    u.t1 = (int)(((long long)(c + 1) * prm.tiles) / g);
    return u;
}
// fused cross-play rollout: (seat-0 policy | seat-1 policy << 16) of the round virtual tile t belongs to
__device__ __forceinline__ uint32_t fused_pair(const PolicyParams& prm, int t) {
    const int kt0 = prm.f_slots * ((int)blockIdx.x + (t / prm.f_vt_round) * (int)gridDim.x);
    return (uint32_t)prm.tile_policy[kt0 >> 1] | ((uint32_t)prm.tile_policy[prm.f_seat1_tiles + (kt0 >> 1)] << 16);
}
__device__ __forceinline__ int tile_pol(const PolicyParams& prm, int t) {
    if (prm.tile_policy == nullptr) return 0;
    return prm.f_vt_round ? (int)fused_pair(prm, t) : prm.tile_policy[t];
}
// does tile t need another weight set than the previous tile of this CTA
__device__ __forceinline__ bool blob_changed(const PolicyParams& prm, int t, int t0) {
    if (t == t0) return true;
    if (prm.tile_policy == nullptr) return false;
    if (prm.f_vt_round) return (t % prm.f_vt_round) == 0 && fused_pair(prm, t) != fused_pair(prm, t - 1);
    return prm.tile_policy[t] != prm.tile_policy[t - 1];
}

// critic pass over a rollout slab (policy_pair_kernel<kProf, true>, ocb_policy_value_slab): a unit is (seat tile k, step s)
// for every seat tile whose table entry is >= 0, tile-major (all steps of tile k, then the next such tile), so a CTA's run of
// units changes weights only where it crosses into a tile with another entry.  Each role walks the run with its own copy of
// this cursor; unit (k, s) is the 128-row tile s * n + k of the slab (n = prm.tiles seat tiles per step, table
// prm.tile_policy, prm.f_slots steps).
struct SlabWalk {
    int k, s, pol;  // the current unit and its weight set
    __device__ __forceinline__ int tile(const PolicyParams& prm) const { return s * prm.tiles + k; }
    // advance one unit; true when the new unit needs other weights than the previous one
    __device__ __forceinline__ bool next(const PolicyParams& prm) {
        if (++s < prm.f_slots) return false;
        s = 0;
        do ++k; while (k < prm.tiles && __ldg(prm.tile_policy + k) < 0);
        const int np = k < prm.tiles ? __ldg(prm.tile_policy + k) : pol;  // the loader's look-ahead may step past the last unit
        const bool chg = np != pol;
        pol = np;
        return chg;
    }
};
// blob_changed of unit t of the run [t0, ...); the slab walk advances to unit t here
template <bool kSlab>
__device__ __forceinline__ bool unit_changed(const PolicyParams& prm, int t, int t0, SlabWalk& sw) {
    if (!kSlab) return blob_changed(prm, t, t0);
    return t == t0 || sw.next(prm);
}

// ---------------------------------------------------------------- roles
// loader: global observations -> bf16 cell blocks, one grid column at a time; the two loader
// groups take alternate columns of the CTA's column stream
template <bool kProf, bool kSlab = false>
__device__ __forceinline__ void loader_role(long long* pw, const PolicyParams& prm, const UnitRange ur, uint32_t tmem, uint32_t* s_stage,
                                            uint32_t bars, SlabWalk sw = {}) {
    const int lwarp = (threadIdx.x >> 5) - kEpiWarps, lg = lwarp >> 2, lw = lwarp & 3, lane = threadIdx.x & 31;
    const int W = prm.W, H = prm.H, SC4 = prm.SC >> 2, seg = 5 * H, stride = prm.stage_stride;
    uint32_t* stg = s_stage + lwarp * 32 * stride;
    const uint32_t* obs32 = reinterpret_cast<const uint32_t*>(prm.obs);
    const uint32_t tcells = tmem + ((uint32_t)(lw * 32) << 16) + kColCells;  // this warp's 32 TMEM lanes (rows)
    uint32_t pre[32];
    const bool active = lane < seg;

    // column c of the stream = grid column c % W of tile t0 + c / W; (lt, lx) track the column being
    // prefetched incrementally (no runtime divisions in this latency-bound role)
    const uint32_t ncols = (uint32_t)(ur.t1 - ur.t0) * (uint32_t)W;
    int lt = ur.t0, lx = lg;
    while (lx >= W) lx -= W, ++lt;
    auto issue_loads = [&]() {
        const long long r0 = (long long)(kSlab ? sw.tile(prm) : lt) * kRows + lw * 32;
        if (!kSlab && prm.row_index != nullptr) {  // minibatch rows picked out of the rollout buffer (ocb_policy_evaluate)
            long long mine = r0 + lane;
            mine = mine < prm.M ? mine : prm.M - 1;
            const int src = __ldg(prm.row_index + mine);
#pragma unroll
            for (int r = 0; r < 32; ++r) {
                const long long row = __shfl_sync(0xffffffffu, src, r);
                pre[r] = active ? __ldg(obs32 + row * SC4 + lx * seg + lane) : 0u;
            }
        } else if (kSlab || r0 + 32 <= prm.M) {  // full 32-row slab: constant-stride addresses (a rollout slab has only full tiles)
            const uint32_t* p = obs32 + r0 * SC4 + lx * seg + (active ? lane : 0);
#pragma unroll
            for (int r = 0; r < 32; ++r) pre[r] = active ? __ldg(p + r * SC4) : 0u;
        } else {  // ragged tail: rows past M re-read the last row (their results are never stored)
#pragma unroll
            for (int r = 0; r < 32; ++r) {
                long long row = r0 + r;
                row = row < prm.M ? row : prm.M - 1;
                pre[r] = active ? __ldg(obs32 + row * SC4 + lx * seg + lane) : 0u;
            }
        }
        lx += 2;
        while (lx >= W) {
            lx -= W, ++lt;
            if (kSlab) sw.next(prm);
        }
    };
    if ((uint32_t)lg < ncols) issue_loads();
    for (uint32_t gc = lg; gc < ncols; gc += 2) {
        const long long tl0 = kProf ? clock64() : 0;
        if (active) {
#pragma unroll
            for (int r = 0; r < 32; ++r) stg[r * stride + lane] = pre[r];
        }
        __syncwarp();
        if (kProf) pw[PW_LDG] += clock64() - tl0;
        if (gc + 2 < ncols) issue_loads();
        const int slot = gc % kColRing;
        if (gc >= kColRing) {
            mbar_wait_p<kProf>(bars + 8 * (B_COL_EMPTY + slot), ((gc / kColRing) - 1) & 1, pw[PW_COL_EMPTY]);
            tc_fence_after();
        }
        const uint32_t* mine = stg + lane * stride;
        const long long tc0 = kProf ? clock64() : 0;
        for (int y = 0; y < H; ++y) {
            uint32_t w[5];
#pragma unroll
            for (int q = 0; q < 5; ++q) w[q] = mine[y * 5 + q];
            // chunk 0: channels 0..7 ; chunk 1: channels 8, 9, 16, 17, 18, 19, 15, pad (slot_channel())
            const uint4 c0 = make_uint4(bytes_bf16x2(w[0], pair_sel(0, 1)), bytes_bf16x2(w[0], pair_sel(2, 3)),
                                        bytes_bf16x2(w[1], pair_sel(0, 1)), bytes_bf16x2(w[1], pair_sel(2, 3)));
            const uint4 c1 = make_uint4(bytes_bf16x2(w[2], pair_sel(0, 1)), bytes_bf16x2(w[4], pair_sel(0, 1)),
                                        bytes_bf16x2(w[4], pair_sel(2, 3)), bytes_bf16x2(w[3], pair_sel(3, 4)));
            tmem_st8(tcells + (slot * H + y) * kCellCols, c0, c1);
        }
        tmem_st_wait();
        if (kProf) pw[PW_CVT] += clock64() - tc0;
        tc_fence_before();
        mbar_arrive(bars + 8 * (B_COL_FULL + slot));
        __syncwarp();  // the staging rows are rewritten by the next column
    }
}

// actor outputs of one row: raw logits, sampled (or arg-max) action and its log-prob
// FixedCategorical(logits): sample / mode and log-prob (train/MAPPO/utils/distributions.py:14-28)
// `store` indexes the output arrays, `rng_row` keys the sampling counter (they differ in the fused
// rollout, where a step's outputs land at step * rows + row); returns the action
// the 32 random bits that sample the action of (row, step): Philox4x32-10, counter (row, offset lo, offset hi, tag)
__device__ __forceinline__ uint32_t policy_draw(const PolicyParams& prm, uint32_t rng_row, unsigned long long offset) {
    const uint32_t grow = rng_row + (rng_row < prm.rng_rows_per_seat ? prm.rng_add0 : prm.rng_add1);
    uint32_t r[4] = {grow, (uint32_t)offset, (uint32_t)(offset >> 32), 0x5A17u};
    philox4x32_10(r, (uint32_t)prm.seed, (uint32_t)(prm.seed >> 32));
    return r[0];
}
// `drawn` (optional): policy_draw of this row, computed by the caller while it was waiting for the accumulator.
// `early_slot` / `early_bar` (fused rollout): the action byte is published there and the mbarrier arrived on as soon as
// the action is known — the env warps start the transition while this thread still computes the log-prob and stores.
__device__ __forceinline__ int emit_actor_row(const PolicyParams& prm, long long store, uint32_t rng_row, const float (&head)[6],
                                              unsigned long long offset, bool force_sample = false, const uint32_t* drawn = nullptr,
                                              uint8_t* early_slot = nullptr, uint32_t early_bar = 0) {
    if (prm.logits) {
#pragma unroll
        for (int a = 0; a < 6; ++a) prm.logits[store * 6 + a] = head[a];
    }
    int act = 0;
    if (prm.actions || prm.logp || prm.entropy || force_sample) {
        float mx = head[0];
#pragma unroll
        for (int a = 1; a < 6; ++a) mx = fmaxf(mx, head[a]);
        float e[6], sum = 0.0f;
#pragma unroll
        for (int a = 0; a < 6; ++a) e[a] = expf(head[a] - mx), sum += e[a];
        if (prm.entropy) {  // -sum p log p with log p = (x - max) - log(sum) (torch Categorical.entropy on normalised logits)
            const float ls = logf(sum);
            float ent = 0.0f;
#pragma unroll
            for (int a = 0; a < 6; ++a) ent -= (e[a] / sum) * (head[a] - mx - ls);
            prm.entropy[store] = ent;
        }
        if (prm.given_actions) {
            const long long src = prm.row_index ? (long long)prm.row_index[store] : store;
            act = prm.given_actions[src];
            act = act < 0 ? 0 : (act > 5 ? 5 : act);
        } else if (prm.deterministic) {
#pragma unroll
            for (int a = 1; a < 6; ++a) act = (head[a] > head[act]) ? a : act;
        } else {
            const uint32_t r0 = drawn != nullptr ? *drawn : policy_draw(prm, rng_row, offset);
            const float uu = (float)(r0 >> 8) * (1.0f / 16777216.0f) * sum;
            float cum = 0.0f;
            act = 5;  // inverse CDF; falls through to the last action on round-off
            bool found = false;
#pragma unroll
            for (int a = 0; a < 6; ++a) {
                cum += e[a];
                if (!found && uu < cum) act = a, found = true;
            }
        }
        if (early_slot != nullptr) {
            *early_slot = (uint8_t)act;
            mbar_arrive(early_bar);
        }
        if (prm.actions) prm.actions[store] = act;
        if (prm.logp) {
            float la = head[0];
#pragma unroll
            for (int a = 1; a < 6; ++a) la = (act == a) ? head[a] : la;
            prm.logp[store] = la - mx - logf(sum);
        }
    }
    return act;
}

// head (64 -> 6 logits | 1 value) over 32 hidden units [i0, i0 + 32): h = relu(acc + b2), head += h * W.  The weights
// are read as 16-byte broadcast loads (actor: [64][8] hidden-major, critic: [64]); fp32 FMAs on CUDA cores.
__device__ __forceinline__ void head_accumulate(int net, const float (&v)[32], const float* b2, const float* s_wh, int i0,
                                                float (&head)[6]) {
    const float4* b4 = reinterpret_cast<const float4*>(b2);
    if (net == 0) {
        const float4* w4 = reinterpret_cast<const float4*>(s_wh) + 2 * i0;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const float4 b = b4[q];
            const float bb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int i = 4 * q + k;
                const float h = fmaxf(v[i] + bb[k], 0.0f);
                const float4 wa = w4[2 * i], wb = w4[2 * i + 1];
                head[0] = fmaf(h, wa.x, head[0]), head[1] = fmaf(h, wa.y, head[1]), head[2] = fmaf(h, wa.z, head[2]);
                head[3] = fmaf(h, wa.w, head[3]), head[4] = fmaf(h, wb.x, head[4]), head[5] = fmaf(h, wb.y, head[5]);
            }
        }
    } else {
        const float4* w4 = reinterpret_cast<const float4*>(s_wh + i0);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const float4 b = b4[q], w = w4[q];
            head[0] = fmaf(fmaxf(v[4 * q + 0] + b.x, 0.0f), w.x, head[0]);
            head[0] = fmaf(fmaxf(v[4 * q + 1] + b.y, 0.0f), w.y, head[0]);
            head[0] = fmaf(fmaxf(v[4 * q + 2] + b.z, 0.0f), w.z, head[0]);
            head[0] = fmaf(fmaxf(v[4 * q + 3] + b.w, 0.0f), w.w, head[0]);
        }
    }
}

// ================================================================ pair kernel: both networks of a tile in ONE CTA
// Every hidden-64 forward runs this kernel (the single-network calls in its single mode, below).  A work
// unit is a tile of 128 rows; the CTA computes the actor AND the critic for it:
//   * the observation columns are loaded and converted once for both networks (loader_role above);
//   * the conv is ONE accumulate of N = 64 (actor channels 0-31 | critic channels 32-63): the two
//     networks' conv weights sit back to back in shared memory and form one canonical K-major operand;
//   * epilogue group g (warps 4g .. 4g+3) owns network g end to end: conv position -> bias/ReLU/split ->
//     A operand stage g -> FC1 partial sums into D2[g]; FC2's two K halves go through the same stage and
//     accumulate into the (by then drained) conv accumulator stage g; the whole head of network g is
//     evaluated by group g (no cross-group reduction);
//   * TMEM: cells 0-191 | conv accumulators 2 x 64 (later D3 of net 0 / net 1) | A stage 2 x 32 | D2 2 x 64.
// Compared with one network per CTA this doubles the work in flight per SM
// (the pipeline is latency-bound: every hand-off is an mbarrier round trip), halves the loader work
// and the number of conv MMA instructions, and lets 128 tiles (config 4: 8,192 worlds) run as ONE wave.
constexpr int kPColD1 = 192;   // conv accumulators: stage s at + 64 s (actor 32 | critic 32); D3 of net g = stage g
constexpr int kPColA2 = 320;   // A operand of net g at + 32 g (hi 16 | lo 16)
constexpr int kPColD2 = 384;   // FC1 accumulator of net g at + 64 g
constexpr int kPMaxRing = 24;  // weight-ring slots (chunks of both networks)
// The four MMA issuers sit on four different SM sub-partitions (warp % 4): each UTCHMMA needs its operands moved into
// uniform registers, and two issuers on one sub-partition share that datapath (measured: no gain from the second one).
constexpr int kWarpConv2 = kWarpMma + 1;        // warp 17: second conv issuer (odd positions; warp kWarpMma = 16 issues the even ones)
constexpr int kWarpFc = kWarpConv2 + 1;         // warps 18, 19: FC issuers of the actor / the critic
constexpr int kPWarpProd = kWarpFc + 2;         // warp 20: weight producer of the pair / fused kernels
constexpr int kPThreads = 32 * (kPWarpProd + 1);  // 672: 8 epilogue + 8 loader + 2 conv issuers + 2 FC issuers + producer
constexpr int kPConvBytes = 9216;  // one network's conv weights, hi or lo
constexpr int kPRestOff = 4 * kPConvBytes;  // per-network remainder of the head (bias1 .. bh) starts here
enum : int {
    PB_COL_FULL = B_COL_FULL,   // [4] shared with loader_role
    PB_COL_EMPTY = B_COL_EMPTY, // [4]
    PB_D1_FULL = 8,             // [2] MMA commit -> both epilogue groups
    PB_A2_FULL = 10,            // [2] epilogue group g -> MMA (128 arrivals)
    PB_A2_EMPTY = 12,           // [2] MMA commit -> epilogue group g
    PB_D2_FULL = 14,            // [2] MMA commit -> epilogue group g
    PB_D3_FULL = 16,            // [2] MMA commit -> epilogue group g
    PB_D3_EMPTY = 18,           // [2] epilogue group g (128 arrivals) -> MMA: conv stage g may be overwritten
    PB_HEAD_FULL = 20,          //     bulk copies -> MMA, epilogue
    PB_HEAD_EMPTY = 21,         // [2] by tile parity: MMA commit + 256 epilogue arrivals -> producer
    PB_W_FULL = 24,             // [24] bulk copy complete_tx -> MMA
    PB_W_EMPTY = 48,            // [24] MMA commit -> producer
    PB_D1_EMPTY = 72,           // [2] both epilogue groups (256 arrivals) -> conv issuer: stage has been read
    // split mode (fused rollout): one conv stream per network, accumulator stages [net][2] of 32 columns
    PBS_D1_FULL = 74,           // [2][2] conv issuer of net g -> epilogue group g
    PBS_D1_EMPTY = 78,          // [2][2] epilogue group g (128 arrivals) -> conv issuer of net g
    PB_COUNT = 82,
    PB_TMEM_SLOT = 120          // 8-byte slot index that holds the TMEM base address
};

struct PairSmemLayout {
    int stage, head, wring, bars, total;
};
__host__ __device__ inline PairSmemLayout pair_smem_layout(int npos, int ring, int stage_stride) {
    PairSmemLayout s;
    const BlobLayout L = blob_layout(npos);
    int o = 0;
    s.stage = o, o += al128(kLoadWarps * 32 * stage_stride * 4);
    s.head = o, o += kPRestOff + 2 * (L.head_bytes - L.bias1);
    s.wring = o, o += ring * kChunk;
    s.bars = o, o += 1024;
    s.total = o + 128;
    return s;
}

// kPop (population self-play in the fused rollout): the two streams are the actor and critic of the slice's weight set
// kMix (mixed play in the fused rollout): stream 0 is the actor at prm.blobs, stream 1 the actor at `mix_partner`
template <bool kProf, bool kPop = false, bool kMix = false, bool kSlab = false>
__device__ __forceinline__ void pair_producer_role(long long* pw, const PolicyParams& prm, int t0, int t1, const BlobLayout L,
                                                   uint32_t s_head, uint32_t s_wring, uint32_t bars,
                                                   const uint8_t* mix_partner = nullptr, SlabWalk sw = {}) {
    const int nets = prm.single ? 1 : 2;  // single mode: the one network takes the actor's places (stream 0, ring slots 0, 1, ...)
    const int R = prm.pair_ring, nch = nets * L.chunks;
    const bool resident = R >= nch;
    const bool static_w = resident && prm.tile_policy == nullptr;  // nothing to do after the first tile (pair_fc_role)
    const int Reff = resident ? nch : R;
    const uint32_t rest = (uint32_t)(L.head_bytes - L.bias1);
    uint32_t u = 0, round = 0;
    int slot = 0;
    for (int t = t0; t < t1; ++t, ++u) {
        if (static_w && u > 0) break;
        const bool chg = unit_changed<kSlab>(prm, t, t0, sw);
        const int tp = kSlab ? sw.pol : tile_pol(prm, t);
        const bool cross = prm.f_vt_round != 0 && prm.tile_policy != nullptr;  // both streams are actors (of two policies)
        const uint8_t* blob_a = prm.blobs + ((size_t)(cross ? (tp & 0xFFFF) : tp) * 2 + (prm.single == 2 ? 1 : 0)) * prm.blob_stride;
        const uint8_t* blob_c = kMix ? mix_partner
                                     : cross && !kPop ? prm.blobs + (size_t)(tp >> 16) * 2 * prm.blob_stride : blob_a + prm.blob_stride;
        if (chg) {
            if (u > 0) mbar_wait_p<kProf>(bars + 8 * (PB_HEAD_EMPTY + ((u - 1) & 1)), ((u - 1) >> 1) & 1, pw[PW_HEAD_EMPTY]);
            if (elect_one()) {
                const uint32_t hb = bars + 8 * PB_HEAD_FULL;
                mbar_arrive_expect_tx(hb, (uint32_t)nets * (2u * kPConvBytes + rest));
                bulk_g2s(s_head, blob_a + L.wc_hi, kPConvBytes, hb);
                bulk_g2s(s_head + 2 * kPConvBytes, blob_a + L.wc_lo, kPConvBytes, hb);
                bulk_g2s(s_head + kPRestOff, blob_a + L.bias1, rest, hb);
                if (nets == 2) {
                    bulk_g2s(s_head + kPConvBytes, blob_c + L.wc_hi, kPConvBytes, hb);
                    bulk_g2s(s_head + 3 * kPConvBytes, blob_c + L.wc_lo, kPConvBytes, hb);
                    bulk_g2s(s_head + kPRestOff + rest, blob_c + L.bias1, rest, hb);
                }
            }
            __syncwarp();
        }
        const bool load = !resident || chg;
        for (int j = 0; j < L.chunks; ++j) {
#pragma unroll
            for (int g = 0; g < 2; ++g) {  // ring order: (actor, j), (critic, j) -> pair_fc_role g takes every other chunk
                if (g >= nets) break;
                if (round > 0) mbar_wait_p<kProf>(bars + 8 * (PB_W_EMPTY + slot), (round - 1) & 1, pw[PW_W_EMPTY]);
                if (load) {
                    if (elect_one()) {
                        mbar_arrive_expect_tx(bars + 8 * (PB_W_FULL + slot), kChunk);
                        bulk_g2s(s_wring + slot * kChunk, (g ? blob_c : blob_a) + L.head_bytes + (size_t)j * kChunk, kChunk,
                                 bars + 8 * (PB_W_FULL + slot));
                    }
                    __syncwarp();
                }
                if (++slot == Reff) slot = 0, ++round;
            }
        }
    }
}

// MMA issue is split over THREE single-lane issuers (round 2; tools/fused_trace.py showed the one-warp issuer of round 1
// spending ~2/3 of a conv position in its own serial code — waits, fences, commits — with the tensor pipe idle):
//   * the conv warp streams the 18 MMAs of every conv position, gated only by the grid columns (loaders) and by the
//     accumulator stage having been read by both epilogue groups (PB_D1_EMPTY), so it runs up to two positions ahead;
//   * FC warp g issues the FC1 partial products and the two FC2 halves of network g as soon as epilogue group g has
//     published their A operand; the two networks no longer wait for each other.
// tcgen05.mma from different warps of a CTA execute in issue order; the three streams touch disjoint accumulators and
// every cross-stream dependency is an mbarrier.
// kNet = -1: one stream for both networks (N = 64, pair kernel).  kNet = 0 / 1 (fused rollout): the stream of ONE network
// (N = 32, its own two 32-column accumulator stages inside the same 128 columns).  The critic's stream of a tile starts
// only when the actor's FC2 of that tile has been issued: the tensor pipe then carries nothing but the actor — the only
// network the next env step waits for — until the actions are out, and the critic's forward fills the pipe's idle time
// under the head / sampling / env step / plane loading of the next step.  Same products per output element, same order.
// `ring` grid columns are resident in the cell region (barriers col_full + slot / col_empty + slot): 4 in the pair kernel;
// the split mode needs the WHOLE grid resident (ring >= W), because the critic's stream starts after the actor's finished.
// An issuer handles the conv positions cp0, cp0 + cpstep, ... of every tile: with cpstep = 2 two warps share a stream
// (position parity == accumulator stage), because ONE thread issuing 18 MMAs + commits + its waits per position
// (~1.15 k cycles, tools/fused_trace.py) is slower than the epilogue that consumes them.  Every issuer releases a grid
// column (col_empty) once none of ITS later positions reads it; the barrier counts the issuers.
template <bool kProf, int kNet, bool kSlab = false>
__device__ __forceinline__ void pair_conv_role(long long* pw, const PolicyParams& prm, int t0, int t1, const BlobLayout L, uint32_t tmem,
                                               uint32_t a_head, uint32_t bars, const int cp0 = 0, const int cpstep = 1,
                                               const uint32_t ring = kColRing, const int col_full = PB_COL_FULL,
                                               const int col_empty = PB_COL_EMPTY, SlabWalk sw = {}) {
    const int W = prm.W, H = prm.H, PH = H - 2, npos = prm.npos;
    constexpr int kN = kNet < 0 ? kHid : kCo;
    const uint32_t idesc = make_idesc(kRows, kN);  // N = 64: actor channels 0-31 | critic channels 32-63
    const uint32_t a_wchi = a_head + (kNet == 1 ? kPConvBytes : 0), a_wclo = a_wchi + 2 * kPConvBytes;
    const int b_full = kNet < 0 ? PB_D1_FULL : PBS_D1_FULL + 2 * kNet, b_empty = kNet < 0 ? PB_D1_EMPTY : PBS_D1_EMPTY + 2 * kNet;
    uint32_t head_gen = 0, u = 0;
    uint32_t uses[2] = {0, 0};   // conv positions THIS issuer put into each accumulator stage so far
    const bool tracer = kNet <= 0;
    // Ring bookkeeping without divisions (ring is a runtime value in the fused kernel; a `% ring` costs ~40 uniform-datapath
    // instructions in front of every issue block): (slot, round) of grid column 0 of the tile, of the next column to wait
    // for and of the next column to release advance by one column at a time.
    uint32_t t_slot = 0, t_round = 0;  // grid column 0 of the current tile
    auto advance = [&](uint32_t& slot, uint32_t& round, int n) {
        for (int i = 0; i < n; ++i)
            if (++slot == ring) slot = 0, ++round;
    };

    for (int t = t0; t < t1; ++t, ++u) {
        if (unit_changed<kSlab>(prm, t, t0, sw)) {
            mbar_wait_p<kProf>(bars + 8 * PB_HEAD_FULL, head_gen & 1, pw[PW_HEAD_FULL]);
            ++head_gen;
        }
        if (kNet == 1) {
            // the critic's stream starts when the actor's LAST conv position of this tile has completed: the pipe carried only
            // the actor during its conv phase, and the critic's conv (one issuer, ~1.1 k cycles per position) still ends
            // before the loaders of the next step want the cell columns back
            const int s_last = (npos - 1) & 1;
            const uint32_t cum = (u + 1) * (uint32_t)((npos + 1 - s_last) / 2);
            mbar_wait_p<kProf>(bars + 8 * (PBS_D1_FULL + s_last), (cum - 1) & 1, pw[PW_D3_FULL]);
        }
        uint32_t w_slot = t_slot, w_round = t_round;  // next column to wait for
        uint32_t r_slot = t_slot;                     // next column to release
        uint32_t c_slot = t_slot;                     // slot of grid column ox (the window's first column)
        int cols_seen = 0, released = 0, ox = 0, oy = cp0;
        while (oy >= PH) oy -= PH, ++ox, c_slot = (c_slot + 1 == ring) ? 0 : c_slot + 1;
        for (int cp = cp0; cp < npos; cp += cpstep) {
            const int st = cp & 1;
            for (; cols_seen < ox + 3; ++cols_seen) {  // new window column(s)
                mbar_wait_p<kProf>(bars + 8 * (col_full + w_slot), w_round & 1, pw[PW_COL_FULL]);
                if (++w_slot == ring) w_slot = 0, ++w_round;
            }
            // the stage's previous conv position has been loaded by its reader(s): with cpstep = 2 the stage belongs to this
            // issuer alone; with cpstep = 1 the issuer alternates stages and counts per stage
            if (uses[st] > 0) mbar_wait_p<kProf>(bars + 8 * (b_empty + st), (uses[st] - 1) & 1, pw[PW_D1_FULL]);
            // ... and stage cp (< 2) was (part of) D3 of a network of the previous tile until its head epilogue read it
            // (single mode keeps D3 in the idle FC1 accumulator of "network 1": the next tile's conv does not wait for the head)
            if (u > 0 && cp < 2 && !prm.single)
                mbar_wait_p<kProf>(bars + 8 * (PB_D3_EMPTY + (kNet < 0 ? cp : kNet)), (u - 1) & 1, pw[PW_D3_FULL]);
            tc_fence_after();
            const uint32_t d1 = tmem + kPColD1 + (kNet < 0 ? st * kHid : kNet * kHid + st * kCo);
            // position of the next conv of this issuer -> first grid column it still reads
            int nox = ox, noy = oy + cpstep;
            uint32_t n_slot = c_slot;
            while (noy >= PH) noy -= PH, ++nox, n_slot = (n_slot + 1 == ring) ? 0 : n_slot + 1;
            const int keep = cp + cpstep < npos ? nox : W;
            const uint32_t s1 = (c_slot + 1 >= ring) ? c_slot + 1 - ring : c_slot + 1;
            const uint32_t s2 = (c_slot + 2 >= ring) ? c_slot + 2 - ring : c_slot + 2;
            const uint32_t cellb = tmem + kColCells + (uint32_t)oy * kCellCols, colw = (uint32_t)H * kCellCols;
            const uint32_t cb0 = cellb + c_slot * colw, cb1 = cellb + s1 * colw, cb2 = cellb + s2 * colw;
            const long long ti0 = kProf ? clock64() : 0;
            if (cp == 3 && tracer) trace_ev<kProf>(prm, t - t0, 54);  // waits of conv 3 done, issue starts
            if (cp < 2 && tracer) trace_ev<kProf>(prm, t - t0, 11 + cp);  // waits of conv 0 / 1 done
            if (elect_one()) {
#pragma unroll
                for (int j = 0; j < 9; ++j) {
                    const int dx = j / 3, dy = j - dx * 3;
                    const uint32_t ta = (dx == 0 ? cb0 : dx == 1 ? cb1 : cb2) + dy * kCellCols;
                    umma_bf16_ts(d1, ta, make_desc(a_wchi + j * 256, 128, 2304), idesc, j > 0);
                    umma_bf16_ts(d1, ta, make_desc(a_wclo + j * 256, 128, 2304), idesc, 1);
                }
                umma_commit(bars + 8 * (b_full + st));
                uint32_t rs = r_slot;
                for (int c = released; c < keep; ++c) {
                    umma_commit(bars + 8 * (col_empty + rs));
                    rs = (rs + 1 == ring) ? 0 : rs + 1;
                }
                // last conv of this issuer in the tile: its reads of the conv weights are done once these MMAs complete
                if (cp + cpstep >= npos) umma_commit(bars + 8 * (PB_HEAD_EMPTY + (u & 1)));
            }
            __syncwarp();
            for (; released < keep; ++released) r_slot = (r_slot + 1 == ring) ? 0 : r_slot + 1;
            if (kProf) pw[PW_ISSUE_CONV] += clock64() - ti0;
            if (cp < 8 && tracer) trace_ev<kProf>(prm, t - t0, 16 + cp);
            ++uses[st];
            ox = nox, oy = noy, c_slot = n_slot;
        }
        advance(t_slot, t_round, W);
    }
}

// FC issuer of network g: D2[g] (+)= A[g] x W1_j (j < npos), then D3[g] (+)= A[g] x W2_half (j = npos, npos + 1)
template <bool kProf, bool kSplit>
__device__ __forceinline__ void pair_fc_role(long long* pw, const PolicyParams& prm, const int g, int t0, int t1, const BlobLayout L,
                                             uint32_t tmem, uint32_t a_wring, uint32_t bars) {
    const int npos = prm.npos;
    const int nets = prm.single ? 1 : 2;
    const int R = prm.pair_ring, nch = nets * L.chunks;
    const bool resident = R >= nch;
    const bool static_w = resident && prm.tile_policy == nullptr;  // one weight set for the whole launch: loaded once
    const int Reff = resident ? nch : R;
    const uint32_t idesc = make_idesc(kRows, kHid);
    const uint32_t a_hi = tmem + kPColA2 + g * kA2Cols, a_lo = a_hi + 16;
    uint32_t item = 0, u = 0, w_gen = 0, wround = 0;
    int slot = g;              // ring slot of this network's next chunk (the producer interleaves actor / critic chunks)
    while (slot >= Reff) slot -= Reff, ++wround;
    uint32_t d1_uses = 0;      // conv positions that went through accumulator stage g so far (PB_D1_EMPTY phase)

    for (int t = t0; t < t1; ++t, ++u) {
        const bool chg = blob_changed(prm, t, t0);
        const bool w_loaded = !resident || chg;
        if (resident && w_loaded) ++w_gen;
        d1_uses += (uint32_t)(npos + 1 - g) / 2;
        for (int j = 0; j < npos + 2; ++j, ++item) {
            mbar_wait_p<kProf>(bars + 8 * (PB_A2_FULL + g), item & 1, pw[PW_A2_FULL]);
            if (g == 0 && j == npos) trace_ev<kProf>(prm, t - t0, 62);  // FC2 first half: A operand seen
            // the first FC2 product overwrites accumulator stage g: its last conv position must have been read by BOTH groups
            // (split mode: D3[g] covers the two stages of network g alone, which group g drained before it published this item)
            if (!kSplit && j == npos) mbar_wait_p<kProf>(bars + 8 * (PB_D1_EMPTY + g), (d1_uses - 1) & 1, pw[PW_D1_FULL]);
            if (w_loaded) mbar_wait_p<kProf>(bars + 8 * (PB_W_FULL + slot), resident ? ((w_gen - 1) & 1) : (wround & 1), pw[PW_W_FULL]);
            tc_fence_after();
            const uint32_t dst = tmem + (j < npos ? kPColD2 : kPColD1) + g * kHid;
            const bool first = (j == 0 || j == npos);
            const uint32_t b_hi = a_wring + slot * kChunk, b_lo = b_hi + 4096;
            const long long tf0 = kProf ? clock64() : 0;
            if (j == npos) trace_ev<kProf>(prm, t - t0, g == 0 ? 55 : 57);  // waits of the first FC2 item done, issue starts
            if (elect_one()) {
#pragma unroll
                for (int ks = 0; ks < 2; ++ks) {
                    const uint64_t bhi = make_desc(b_hi + ks * 256, 128, 512), blo = make_desc(b_lo + ks * 256, 128, 512);
                    umma_bf16_ts(dst, a_hi + ks * 8, bhi, idesc, (!first || ks != 0) ? 1u : 0u);
                    umma_bf16_ts(dst, a_hi + ks * 8, blo, idesc, 1);
                    umma_bf16_ts(dst, a_lo + ks * 8, bhi, idesc, 1);
                }
                umma_commit(bars + 8 * (PB_A2_EMPTY + g));
                if (!static_w) umma_commit(bars + 8 * (PB_W_EMPTY + slot));
                if (j == npos - 1) umma_commit(bars + 8 * (PB_D2_FULL + g));
                if (j == npos + 1) umma_commit(bars + 8 * (PB_D3_FULL + g));
            }
            __syncwarp();
            if (kProf) pw[PW_ISSUE_FC] += clock64() - tf0;
            if (g == 0 && j < 8) trace_ev<kProf>(prm, t - t0, 24 + j);
            if (g == 1 && j == npos) trace_ev<kProf>(prm, t - t0, 58);
            slot += nets;
            if (slot >= Reff) slot -= Reff, ++wround;
        }
    }
}

// `out(t, trow_id, g, head)` consumes the head outputs of row trow_id of tile t (g = 0: six logits, g = 1: head[0] = value)
template <bool kProf, bool kSplit, bool kPop = false, bool kMix = false, class Out>
__device__ __forceinline__ void pair_epilogue_role(long long* pw, const PolicyParams& prm, int t0, int t1, const BlobLayout L, uint32_t tmem,
                                                   const uint8_t* s_head, uint32_t bars, Out&& out) {
    const int warp = threadIdx.x >> 5, g = warp >> 2, trow_id = (warp & 3) * 32 + (threadIdx.x & 31);
    const int npos = prm.npos;
    const uint32_t trow = tmem + ((uint32_t)((warp & 3) * 32) << 16);  // this warp's 32 TMEM lanes
    const uint8_t* rest = s_head + kPRestOff + g * (L.head_bytes - L.bias1) - L.bias1;  // network g's bias1 .. bh, blob offsets
    const float* s_bias1 = reinterpret_cast<const float*>(rest + L.bias1);
    const float* s_b1 = reinterpret_cast<const float*>(rest + L.b1);
    const float* s_b2 = reinterpret_cast<const float*>(rest + L.b2);
    const float* s_wh = reinterpret_cast<const float*>(rest + L.wh);
    const float* s_bh = reinterpret_cast<const float*>(rest + L.bh);
    const uint32_t a2 = trow + kPColA2 + g * kA2Cols;
    // head layout / outputs: 0 = actor (6 logits), 1 = critic (value); fused cross-play and mixed play: two actors
    const int net = (kMix || (!kPop && prm.f_vt_round != 0 && prm.tile_policy != nullptr)) ? 0 : (prm.single == 2 ? 1 : g);

    uint32_t u = 0, head_gen = 0, item = 0, d1_par = 0;  // d1_par: phase parity bit per conv accumulator stage
    int trace_vt = 0, trace_item = 0;
    // bias + ReLU + hi/lo split of 32 activations -> A operand stage of this network
    auto publish = [&](float (&v)[32], const float* bias) {
        const float4* b4 = reinterpret_cast<const float4*>(bias);
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int q = 0; q < 8; ++q) {  // the conversion runs before the wait: the stage is usually still being read
            const float4 b = b4[q];
            split2(fmaxf(v[4 * q] + b.x, 0.0f), fmaxf(v[4 * q + 1] + b.y, 0.0f), hi[2 * q], lo[2 * q]);
            split2(fmaxf(v[4 * q + 2] + b.z, 0.0f), fmaxf(v[4 * q + 3] + b.w, 0.0f), hi[2 * q + 1], lo[2 * q + 1]);
        }
        if (item >= 1) {
            mbar_wait_p<kProf>(bars + 8 * (PB_A2_EMPTY + g), (item - 1) & 1, pw[PW_A2_EMPTY]);
            tc_fence_after();
        }
        if (kProf && warp == 0 && trace_item == 2) trace_ev<kProf>(prm, trace_vt, 60);  // A2 stage free and split done
        tmem_st16(a2, hi);
        tmem_st16(a2 + 16, lo);
        tmem_st_wait();
        if (kProf && warp == 0 && trace_item == 2) trace_ev<kProf>(prm, trace_vt, 61);  // stores landed
        tc_fence_before();
        mbar_arrive(bars + 8 * (PB_A2_FULL + g));
        if (kProf && warp == 0 && trace_item < 8) trace_ev<kProf>(prm, trace_vt, 40 + trace_item);
        ++trace_item;
        ++item;
    };

    for (int t = t0; t < t1; ++t, ++u) {
        if (blob_changed(prm, t, t0)) {
            mbar_wait_p<kProf>(bars + 8 * PB_HEAD_FULL, head_gen & 1, pw[PW_HEAD_FULL]);
            ++head_gen;
        }
        trace_vt = t - t0, trace_item = 0;
        for (int j = 0; j < npos; ++j) {
            const int st = j & 1;
            mbar_wait_p<kProf>(bars + 8 * ((kSplit ? PBS_D1_FULL + 2 * g : PB_D1_FULL) + st), (d1_par >> st) & 1, pw[PW_D1_FULL]);
            if (kProf && warp == 0 && j < 8) trace_ev<kProf>(prm, trace_vt, 32 + j);
            d1_par ^= 1u << st;
            tc_fence_after();
            float v[32];
            tmem_ld32(trow + kPColD1 + (kSplit ? g * kHid + st * kCo : st * kHid + g * kCo), v);
            tc_fence_before();
            // the conv issuer may overwrite this stage (pair kernel: once the other group has read its half too)
            mbar_arrive(bars + 8 * ((kSplit ? PBS_D1_EMPTY + 2 * g : PB_D1_EMPTY) + st));
            if (kProf && warp == 0 && j == 2) trace_ev<kProf>(prm, trace_vt, 59);  // accumulator in registers
            publish(v, s_bias1 + j * kCo);
        }
        mbar_wait_p<kProf>(bars + 8 * (PB_D2_FULL + g), u & 1, pw[PW_D2_FULL]);
        if (kProf && warp == 0) trace_ev<kProf>(prm, trace_vt, 48);
        tc_fence_after();
#pragma unroll 1
        for (int half = 0; half < 2; ++half) {
            float v[32];
            tmem_ld32(trow + kPColD2 + g * kHid + half * 32, v);
            publish(v, s_b1 + half * 32);
        }

        // ---- FC2 epilogue + head (fp32 on CUDA cores), all 64 hidden units of this network
        const uint32_t drawn = net == 0 ? out.draw(t, trow_id) : 0u;  // off the critical path: while FC2 runs
        mbar_wait_p<kProf>(bars + 8 * (PB_D3_FULL + g), u & 1, pw[PW_D3_FULL]);
        if (kProf && (warp & 3) == 0) trace_ev<kProf>(prm, trace_vt, g == 0 ? 49 : 52);
        tc_fence_after();
        float head[6];
#pragma unroll
        for (int a = 0; a < 6; ++a) head[a] = s_bh[a];
#pragma unroll 1
        for (int half = 0; half < 2; ++half) {
            float v[32];
            tmem_ld32(trow + kPColD1 + g * kHid + half * 32, v);
            if (half == 1) {  // both halves are in registers: the accumulator stage may be overwritten by the next tile
                tc_fence_before();
                mbar_arrive(bars + 8 * (PB_D3_EMPTY + g));
            }
            head_accumulate(net, v, s_b2 + half * 32, s_wh, half * 32, head);
        }
        mbar_arrive(bars + 8 * (PB_HEAD_EMPTY + (u & 1)));  // done with the head block of this tile
        if (kProf && (warp & 3) == 0) trace_ev<kProf>(prm, trace_vt, g == 0 ? 50 : 53);
        out(t, trow_id, net, head, drawn);
        if (kProf && warp == 0) trace_ev<kProf>(prm, trace_vt, 51);
    }
}
// ---------------------------------------------------------------- single mode: ONE network per tile
// ocb_policy_act / ocb_policy_value / cross-play evaluation.  The conv is the split-mode stream of "network 0" (N = 32, two
// issuers by position parity = accumulator stage).  BOTH epilogue groups work on the tile: group g takes the conv positions of
// parity g (it reads accumulator stage g and owns A-operand stage g) and K half g of FC2's input; ONE FC issuer consumes the
// items in position order, so every output element sums the same products in the same order as in the pair kernel; group 1
// evaluates the head while group 0 is already at the next tile's positions.  D3 sits in the FC1 accumulator columns of the
// absent second network, so the next tile's conv never waits for the head.  (Round 2a ran this mode on group 0 alone: the
// epilogue group was the bottleneck, 14 k cycles per coordination_ring tile.)
constexpr int kSColD3 = kPColD2 + kHid;
constexpr int kSHeadGroup = 1;
// Measured and dropped (524,288 rows of coordination_ring, 206 us): a second A-operand stage per group in the conv
// accumulator columns of the absent second network (218 us), a nanosleep back-off in the loaders' ring-slot wait (209 us:
// try_wait polls are a third of the issued instructions, but not what the working warps wait for), suspend-time hints on
// every wait of this mode (211 us).  ncu: 47.7 k warp instructions per tile; the roles wait on each other in turn (role
// profile, tools/policy_roles.py with OCB_PROFILE_MASK=1): loaders 60 % busy, conv issuers 60 %, epilogue groups 40 %.

template <bool kProf, bool kSlab = false>
__device__ __forceinline__ void single_fc_role(long long* pw, const PolicyParams& prm, int t0, int t1, const BlobLayout L, uint32_t tmem,
                                               uint32_t a_wring, uint32_t bars, SlabWalk sw = {}) {
    const int npos = prm.npos;
    const int R = prm.pair_ring, nch = L.chunks;
    const bool resident = R >= nch;
    const bool static_w = resident && prm.tile_policy == nullptr;
    const int Reff = resident ? nch : R;
    const uint32_t idesc = make_idesc(kRows, kHid);
    uint32_t u = 0, w_gen = 0, wround = 0;
    uint32_t cnt0 = 0, cnt1 = 0;  // items consumed from group 0 / group 1
    int slot = 0;
    for (int t = t0; t < t1; ++t, ++u) {
        const bool chg = unit_changed<kSlab>(prm, t, t0, sw);
        const bool w_loaded = !resident || chg;
        if (resident && w_loaded) ++w_gen;
        for (int j = 0; j < npos + 2; ++j) {
            const int sg = j < npos ? (j & 1) : (j - npos);  // the group that published this item
            const uint32_t k = sg ? cnt1 : cnt0;
            mbar_wait_p<kProf>(bars + 8 * (PB_A2_FULL + sg), k & 1, pw[PW_A2_FULL]);
            if (sg) ++cnt1; else ++cnt0;
            // D3 of the previous tile must have been loaded by the head group before FC2 overwrites it
            if (j == npos && u > 0) mbar_wait_p<kProf>(bars + 8 * PB_D3_EMPTY, (u - 1) & 1, pw[PW_D3_FULL]);
            if (w_loaded) mbar_wait_p<kProf>(bars + 8 * (PB_W_FULL + slot), resident ? ((w_gen - 1) & 1) : (wround & 1), pw[PW_W_FULL]);
            tc_fence_after();
            const uint32_t dst = tmem + (j < npos ? kPColD2 : kSColD3);
            const bool first = (j == 0 || j == npos);
            const uint32_t a_hi = tmem + kPColA2 + sg * kA2Cols, a_lo = a_hi + 16;
            const uint32_t b_hi = a_wring + slot * kChunk, b_lo = b_hi + 4096;
            const long long tf0 = kProf ? clock64() : 0;
            if (elect_one()) {
#pragma unroll
                for (int ks = 0; ks < 2; ++ks) {
                    const uint64_t bhi = make_desc(b_hi + ks * 256, 128, 512), blo = make_desc(b_lo + ks * 256, 128, 512);
                    umma_bf16_ts(dst, a_hi + ks * 8, bhi, idesc, (!first || ks != 0) ? 1u : 0u);
                    umma_bf16_ts(dst, a_hi + ks * 8, blo, idesc, 1);
                    umma_bf16_ts(dst, a_lo + ks * 8, bhi, idesc, 1);
                }
                umma_commit(bars + 8 * (PB_A2_EMPTY + sg));
                if (!static_w) umma_commit(bars + 8 * (PB_W_EMPTY + slot));
                if (j == npos - 1) umma_commit(bars + 8 * PB_D2_FULL);
                if (j == npos + 1) umma_commit(bars + 8 * PB_D3_FULL);
            }
            __syncwarp();
            if (kProf) pw[PW_ISSUE_FC] += clock64() - tf0;
            if (++slot >= Reff) slot = 0, ++wround;
        }
    }
}

template <bool kProf, bool kSlab = false, class Out>
__device__ __forceinline__ void single_epilogue_role(long long* pw, const PolicyParams& prm, int t0, int t1, const BlobLayout L,
                                                     uint32_t tmem, const uint8_t* s_head, uint32_t bars, Out&& out,
                                                     SlabWalk sw = {}) {
    const int warp = threadIdx.x >> 5, g = warp >> 2, trow_id = (warp & 3) * 32 + (threadIdx.x & 31);
    const int npos = prm.npos;
    const int net = (kSlab || prm.single == 2) ? 1 : 0;  // head layout / outputs: 0 = actor (6 logits), 1 = critic (value)
    const uint32_t trow = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const uint8_t* rest = s_head + kPRestOff - L.bias1;  // the network's bias1 .. bh at their blob offsets
    const float* s_bias1 = reinterpret_cast<const float*>(rest + L.bias1);
    const float* s_b1 = reinterpret_cast<const float*>(rest + L.b1);
    const float* s_b2 = reinterpret_cast<const float*>(rest + L.b2);
    const float* s_wh = reinterpret_cast<const float*>(rest + L.wh);
    const float* s_bh = reinterpret_cast<const float*>(rest + L.bh);
    uint32_t u = 0, head_gen = 0, pubs = 0, d1_uses = 0;
    auto publish = [&](float (&v)[32], const float* bias) {
        const uint32_t a2 = trow + kPColA2 + g * kA2Cols;
        const float4* b4 = reinterpret_cast<const float4*>(bias);
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const float4 b = b4[q];
            split2(fmaxf(v[4 * q] + b.x, 0.0f), fmaxf(v[4 * q + 1] + b.y, 0.0f), hi[2 * q], lo[2 * q]);
            split2(fmaxf(v[4 * q + 2] + b.z, 0.0f), fmaxf(v[4 * q + 3] + b.w, 0.0f), hi[2 * q + 1], lo[2 * q + 1]);
        }
        if (pubs >= 1) {  // the group's previous item has been consumed
            mbar_wait_p<kProf>(bars + 8 * (PB_A2_EMPTY + g), (pubs - 1) & 1, pw[PW_A2_EMPTY]);
            tc_fence_after();
        }
        tmem_st16(a2, hi);
        tmem_st16(a2 + 16, lo);
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(bars + 8 * (PB_A2_FULL + g));
        ++pubs;
    };
    for (int t = t0; t < t1; ++t, ++u) {
        if (unit_changed<kSlab>(prm, t, t0, sw)) {
            mbar_wait_p<kProf>(bars + 8 * PB_HEAD_FULL, head_gen & 1, pw[PW_HEAD_FULL]);
            ++head_gen;
        }
        for (int j = g; j < npos; j += 2, ++d1_uses) {  // positions of parity g sit in accumulator stage g
            mbar_wait_p<kProf>(bars + 8 * (PBS_D1_FULL + g), d1_uses & 1, pw[PW_D1_FULL]);
            tc_fence_after();
            float v[32];
            tmem_ld32(trow + kPColD1 + g * kCo, v);
            tc_fence_before();
            mbar_arrive(bars + 8 * (PBS_D1_EMPTY + g));
            publish(v, s_bias1 + j * kCo);
        }
        mbar_wait_p<kProf>(bars + 8 * PB_D2_FULL, u & 1, pw[PW_D2_FULL]);
        tc_fence_after();
        {
            float v[32];
            tmem_ld32(trow + kPColD2 + g * 32, v);
            publish(v, s_b1 + g * 32);
        }
        if (g != kSHeadGroup) {
            mbar_arrive(bars + 8 * (PB_HEAD_EMPTY + (u & 1)));  // this group is done with the tile's biases
            continue;
        }
        const uint32_t drawn = net == 0 ? out.draw(t, trow_id) : 0u;
        mbar_wait_p<kProf>(bars + 8 * PB_D3_FULL, u & 1, pw[PW_D3_FULL]);
        tc_fence_after();
        float head[6];
#pragma unroll
        for (int a = 0; a < 6; ++a) head[a] = s_bh[a];
#pragma unroll 1
        for (int half = 0; half < 2; ++half) {
            float v[32];
            tmem_ld32(trow + kSColD3 + half * 32, v);
            if (half == 1) {
                tc_fence_before();
                mbar_arrive(bars + 8 * PB_D3_EMPTY);
            }
            head_accumulate(net, v, s_b2 + half * 32, s_wh, half * 32, head);
        }
        mbar_arrive(bars + 8 * (PB_HEAD_EMPTY + (u & 1)));
        out(kSlab ? sw.tile(prm) : t, trow_id, net, head, drawn);
    }
}

// output stage of the plain forward: rows are tile-major
struct PairForwardOut {
    const PolicyParams& prm;
    unsigned long long offset;
    __device__ __forceinline__ PairForwardOut(const PolicyParams& p) : prm(p), offset(p.offset) {
        if (p.d_offset != nullptr) offset += *p.d_offset;
    }
    __device__ __forceinline__ uint32_t draw(int t, int trow_id) const {
        if (prm.deterministic || prm.given_actions != nullptr || !(prm.actions || prm.logp)) return 0u;
        return policy_draw(prm, (uint32_t)((long long)t * kRows + trow_id), offset);
    }
    __device__ __forceinline__ void operator()(int t, int trow_id, int net, const float (&head)[6], uint32_t drawn) const {
        const long long row = (long long)t * kRows + trow_id;
        if (row < prm.M) {
            if (net == 1) {
                if (prm.values) prm.values[row] = head[0];
            } else {
                emit_actor_row(prm, row, (uint32_t)row, head, offset, false, &drawn);
            }
        }
    }
};

// kSlab: the critic over a rollout slab (single == 2): prm.tile_policy is the table of prm.tiles seat tiles per step,
// prm.f_slots the number of steps and prm.M = steps * 128 * prm.tiles rows.  The CTA counts the tiles with an entry >= 0 (A) in the device table itself, takes its
// even share [u0, u1) of the A * steps units and starts the walk at unit u0 (every thread scans a contiguous share of the
// table; one block-wide prefix sum finds the tile of rank u0 / steps).
__device__ __forceinline__ void slab_run(const PolicyParams& prm, uint32_t* s_scan, int* s_k0, SlabWalk& sw, int& u0, int& u1) {
    const int n = prm.tiles, steps = prm.f_slots, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int per = (n + kPThreads - 1) / kPThreads, lo = tid * per < n ? tid * per : n, hi = lo + per < n ? lo + per : n;
    int cnt = 0;
    for (int i = lo; i < hi; ++i) cnt += __ldg(prm.tile_policy + i) >= 0;
    int incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += v;
    }
    if (lane == 31) s_scan[warp] = (uint32_t)incl;
    __syncthreads();
    int A = 0, excl = incl - cnt;
    for (int w = 0; w < kPThreads / 32; ++w) {
        A += (int)s_scan[w];
        if (w < warp) excl += (int)s_scan[w];
    }
    const long long U = (long long)A * steps;
    u0 = (int)(((long long)blockIdx.x * U) / gridDim.x);
    u1 = (int)(((long long)(blockIdx.x + 1) * U) / gridDim.x);
    const int r0 = u0 / steps;
    if (u0 < u1 && r0 >= excl && r0 < excl + cnt) {  // this thread's share holds the run's first tile
        int r = excl;
        for (int i = lo; i < hi; ++i) {
            if (__ldg(prm.tile_policy + i) < 0) continue;
            if (r++ == r0) {
                *s_k0 = i;
                break;
            }
        }
    }
    sw.s = u0 - r0 * steps;
}

template <bool kProf, bool kSlab = false>
__global__ void __launch_bounds__(kPThreads, 1) policy_pair_kernel(const PolicyParams prm) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((128u - (smem_addr(smem_raw) & 127u)) & 127u);
    const int tid = threadIdx.x, warp = tid >> 5;
    const BlobLayout L = blob_layout(prm.npos);
    const PairSmemLayout sl = pair_smem_layout(prm.npos, prm.pair_ring, prm.stage_stride);
    uint32_t* s_stage = reinterpret_cast<uint32_t*>(smem + sl.stage);
    uint8_t* s_head = smem + sl.head;
    uint8_t* s_wring = smem + sl.wring;
    uint64_t* s_bars = reinterpret_cast<uint64_t*>(smem + sl.bars);
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bars + PB_TMEM_SLOT);
    const uint32_t bars = smem_addr(s_bars);

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_addr(s_tmem)),
                     "r"((uint32_t)kTmemCols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 32) {
        for (int i = 0; i < PB_COUNT; ++i) {
            uint32_t count = 1;
            if ((i >= PB_COL_FULL && i < PB_COL_FULL + 4) || (i >= PB_A2_FULL && i < PB_A2_FULL + 2) ||
                (i >= PB_D3_EMPTY && i < PB_D3_EMPTY + 2))
                count = 128;
            if (i >= PB_COL_EMPTY && i < PB_COL_EMPTY + 4) count = 2;  // both conv issuers are done with the column
            if (i >= PB_HEAD_EMPTY && i < PB_HEAD_EMPTY + 2) count = 32 * kEpiWarps + 2;
            if (i >= PB_D1_EMPTY && i < PB_D1_EMPTY + 2) count = 32 * kEpiWarps;
            if (i >= PBS_D1_EMPTY && i < PBS_D1_EMPTY + 4) count = 128;  // single mode runs the split-mode stream of "network 0"
            mbar_init(bars + 8 * i, count);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // the loaders' staging buffer is free until the roles start; the first tile of the slab run goes next to the TMEM slot
    SlabWalk sw = {};
    int* s_k0 = reinterpret_cast<int*>(s_bars + PB_TMEM_SLOT + 1);
    int su0 = 0, su1 = 0;
    if (kSlab) slab_run(prm, s_stage, s_k0, sw, su0, su1);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *s_tmem;
    // tiles of this CTA
    UnitRange ur;
    ur.net = 0;
    ur.t0 = kSlab ? su0 : (int)(((long long)blockIdx.x * prm.tiles) / gridDim.x);
    ur.t1 = kSlab ? su1 : (int)(((long long)(blockIdx.x + 1) * prm.tiles) / gridDim.x);
    if (kSlab && su0 < su1) sw.k = *s_k0, sw.pol = __ldg(prm.tile_policy + sw.k);

    long long pw[kProf ? PW_COUNT : 1] = {};
    const long long t_begin = kProf ? clock64() : 0;
    if (kSlab || prm.single) {  // ONE network per tile (see single_epilogue_role)
        if (warp < kEpiWarps) {
            single_epilogue_role<kProf, kSlab>(pw, prm, ur.t0, ur.t1, L, tmem, s_head, bars, PairForwardOut(prm), sw);
        } else if (warp < kWarpMma) {
            loader_role<kProf, kSlab>(pw, prm, ur, tmem, s_stage, bars, sw);
        } else if (warp == kWarpMma || warp == kWarpConv2) {
            pair_conv_role<kProf, 0, kSlab>(pw, prm, ur.t0, ur.t1, L, tmem, smem_addr(s_head), bars, warp == kWarpMma ? 0 : 1, 2,
                                            kColRing, PB_COL_FULL, PB_COL_EMPTY, sw);
        } else if (warp == kPWarpProd) {
            pair_producer_role<kProf, false, false, kSlab>(pw, prm, ur.t0, ur.t1, L, smem_addr(s_head), smem_addr(s_wring), bars,
                                                           nullptr, sw);
        } else if (warp == kWarpFc) {
            single_fc_role<kProf, kSlab>(pw, prm, ur.t0, ur.t1, L, tmem, smem_addr(s_wring), bars, sw);
        }
    } else if (warp < kEpiWarps) {
        pair_epilogue_role<kProf, false>(pw, prm, ur.t0, ur.t1, L, tmem, s_head, bars, PairForwardOut(prm));
    } else if (warp < kWarpMma) {
        loader_role<kProf>(pw, prm, ur, tmem, s_stage, bars);
    } else if (warp == kWarpMma || warp == kWarpConv2) {
        pair_conv_role<kProf, -1>(pw, prm, ur.t0, ur.t1, L, tmem, smem_addr(s_head), bars, warp == kWarpMma ? 0 : 1, 2);
    } else if (warp == kPWarpProd) {
        pair_producer_role<kProf>(pw, prm, ur.t0, ur.t1, L, smem_addr(s_head), smem_addr(s_wring), bars);
    } else {
        pair_fc_role<kProf, false>(pw, prm, warp - kWarpFc, ur.t0, ur.t1, L, tmem, smem_addr(s_wring), bars);
    }
    // single mode reports its FC issuer in the producer's slot (the producer idles once the weights are resident)
    const int tid_r3 = prm.single ? 32 * kWarpFc : 32 * kPWarpProd;
    if (kProf && prm.prof != nullptr && (tid == 0 || tid == 32 * kEpiWarps || tid == 32 * kWarpMma || tid == tid_r3)) {
        pw[PW_TOTAL] = clock64() - t_begin;
        const int role = tid == 0 ? 0 : tid == 32 * kEpiWarps ? 1 : tid == 32 * kWarpMma ? 2 : 3;
        for (int i = 0; i < PW_COUNT; ++i) prm.prof[((size_t)blockIdx.x * 4 + role) * PW_COUNT + i] = pw[i];
    }
    __syncwarp();
    tc_fence_before();
    __syncthreads();
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)kTmemCols) : "memory");
}

#include "policy512.cuh"
#include "rollout_fused.cuh"
#include "policy_generic.cuh"

// ---------------------------------------------------------------- packing rules
// One definition for both writers of a blob: ocb_policy_set_weights (host loops over HOST weights) and policy_pack_kernel
// (ocb_policy_set_weights_device, DEVICE weights).  Both must produce the same bytes, so every rounding here is explicit.
__host__ __device__ inline uint16_t bf16_bits(float x) {
    uint32_t u;
    memcpy(&u, &x, 4);
    const uint32_t r = u + 0x7FFFu + ((u >> 16) & 1u);  // round to nearest even
    return (uint16_t)(r >> 16);
}
__host__ __device__ inline float bf16_val(uint16_t b) {
    uint32_t u = (uint32_t)b << 16;
    float f;
    memcpy(&f, &u, 4);
    return f;
}
// element (n, k) of an [N x K] K-major operand in the canonical no-swizzle layout
__host__ __device__ inline size_t canon_off(int n, int k, int K) {
    return (size_t)(n / 8) * (K / 8) * 128 + (size_t)(k / 8) * 128 + (n % 8) * 16 + (k % 8) * 2;
}
__host__ __device__ inline void put_split(uint8_t* hi, uint8_t* lo, size_t off, float w) {
    const uint16_t h = bf16_bits(w);
    const uint16_t l = bf16_bits(w - bf16_val(h));
    memcpy(hi + off, &h, 2);
    memcpy(lo + off, &l, 2);
}
// observation channel of bf16 slot s of a cell block (== loader_role): channels 0-9, 16-19, 15, one zero pad (-1)
__host__ __device__ inline int slot_channel(int s) { return s < 10 ? s : s < 14 ? s + 6 : s == 14 ? 15 : -1; }
// element (co, k = window cell j * kSlots + slot) of the conv operand [co x 144]; conv_w is [CO, 20, 3, 3]
__host__ __device__ inline float conv_slot_weight(const float* conv_w, int co, int k) {
    const int j = k / kSlots, ch = slot_channel(k % kSlots);
    return ch < 0 ? 0.0f : conv_w[((co * 20 + ch) * 3 + j / 3) * 3 + j % 3];
}
// conv bias of output position pos plus the static terrain channels (shift+0..4 == channels 10..14, one-hot of terrain-1;
// setup_base_observation, envs/overcooked2_reimplement.py:165-171), summed in double in this order and rounded once
__host__ __device__ inline float terrain_bias(const uint8_t* terrain, int W, int H, const float* conv_w, const float* conv_b,
                                              int pos, int co) {
    const int PH = H - 2, ox = pos / PH, oy = pos % PH;
    double acc = conv_b[co];
    for (int dx = 0; dx < 3; ++dx)
        for (int dy = 0; dy < 3; ++dy) {
            const int t = terrain[(oy + dy) * W + ox + dx];
            if (t >= 1 && t <= 5) acc += conv_w[((co * 20 + 10 + (t - 1)) * 3 + dx) * 3 + dy];
        }
    return (float)acc;
}

// R_Critic.forward on an all-zero observation: the conv output is its bias at every position (flatten index co*npos + pos,
// cnn.py:41), then FC -> ReLU -> FC -> ReLU -> v_out.  Each unit is a sequential sum in k with every product and every sum
// rounded on its own: the device spells that out (nvcc would contract them into FMAs), the host build (-O3 for plain x86-64)
// has no FMA instruction to contract into.
__host__ __device__ inline float mul_rn(float a, float b) {
#ifdef __CUDA_ARCH__
    return __fmul_rn(a, b);
#else
    return a * b;
#endif
}
__host__ __device__ inline float add_rn(float a, float b) {
#ifdef __CUDA_ARCH__
    return __fadd_rn(a, b);
#else
    return a + b;
#endif
}
// unit o of the first hidden layer, after the ReLU
__host__ __device__ inline float zero_obs_fc1(int o, int hidden, int npos, const float* conv_b, const float* fc1_w,
                                              const float* fc1_b) {
    const int co_n = hidden / 2;
    const float* w = fc1_w + (size_t)o * co_n * npos;
    float acc = fc1_b[o];
    for (int co = 0; co < co_n; ++co) {
        const float x = fmaxf(conv_b[co], 0.0f);
        for (int pos = 0; pos < npos; ++pos) acc = add_rn(acc, mul_rn(w[co * npos + pos], x));
    }
    return fmaxf(acc, 0.0f);
}
// b + w . x over n inputs (FC2 units and the value head)
__host__ __device__ inline float zero_obs_dot(float b, const float* w, const float* x, int n) {
    float acc = b;
    for (int k = 0; k < n; ++k) acc = add_rn(acc, mul_rn(w[k], x[k]));
    return acc;
}

// ---------------------------------------------------------------- device-side packing (ocb_policy_set_weights_device)
// One launch packs up to kPackMax networks: blockIdx.y = network, the last block of every row computes the zero-observation
// value of a critic, the others walk the blob in 16-byte units.  A unit inside a bf16 hi operand packs one canonical core-matrix
// row (8 K-consecutive elements) into hi AND lo; units inside lo operands are skipped; every other unit is fp32 (padding as
// zeros), so every byte of the blob is written and the result does not depend on what was there.
constexpr int kPackMax = 40;       // descriptors per launch (a 4 KB kernel-parameter block)
constexpr int kPackThreads = 256;
constexpr int kPackMaxBlocks = 1024;
enum : int { PACK_H64 = 0, PACK_H512 = 1, PACK_GENERIC = 2 };

struct PackDesc {
    uint8_t* dst;  // the blob
    const float *conv_w, *conv_b, *fc1_w, *fc1_b, *fc2_w, *fc2_b, *head_w, *head_b;
    int policy, net;
};
struct PackArgs {
    int fmt, W, H, C, npos, hidden, n;
    size_t blob_bytes;
    const uint8_t* terrain;  // [W * H] terrain codes of the layout
    float* zero_value;       // [n_policies]
    PackDesc d[kPackMax];
};

// row `row` of an [N x K] operand (rows enumerated in canonical order, so consecutive threads store consecutive 16 bytes);
// wf(n, k) gives the fp32 weight
template <class WF>
__device__ __forceinline__ void pack_split_row(uint8_t* hi, uint8_t* lo, int row, int K, WF wf) {
    const int n = (row / K) * 8 + row % 8, k0 = (row / 8) % (K / 8) * 8;
    uint4 h, l;
#pragma unroll
    for (int kk = 0; kk < 8; ++kk) put_split(reinterpret_cast<uint8_t*>(&h), reinterpret_cast<uint8_t*>(&l), kk * 2, wf(n, k0 + kk));
    const size_t o = canon_off(n, k0, K);
    *reinterpret_cast<uint4*>(hi + o) = h;
    *reinterpret_cast<uint4*>(lo + o) = l;
}

// the fp32 word at byte offset o of a hidden-64 blob's head (bias1 .. bh)
__device__ float pack_f32_h64(const PackArgs& a, const PackDesc& d, const BlobLayout& L, int o) {
    if (o < L.b1) {
        const int i = (o - L.bias1) / 4;
        return i < a.npos * kCo ? terrain_bias(a.terrain, a.W, a.H, d.conv_w, d.conv_b, i / kCo, i % kCo) : 0.0f;
    }
    if (o < L.b2) return d.fc1_b[(o - L.b1) / 4];
    if (o < L.wh) return d.fc2_b[(o - L.b2) / 4];
    if (o < L.bh) {
        const int i = (o - L.wh) / 4;
        if (d.net == 0) return i % 8 < 6 ? d.head_w[(i % 8) * kHid + i / 8] : 0.0f;  // hidden-major [64][8]
        return i < kHid ? d.head_w[i] : 0.0f;
    }
    const int i = (o - L.bh) / 4;
    return i < (d.net == 0 ? 6 : 1) ? d.head_b[i] : 0.0f;
}

// the fp32 word at byte offset o of a Blob5 outside its bf16 operands
__device__ float pack_f32_h512(const PackArgs& a, const PackDesc& d, const Blob5& L, size_t o) {
    const int head_out = d.net == 0 ? 6 : 1;
    if (o < L.w1) {
        const int i = (int)((o - L.bias1) / 4);
        return terrain_bias(a.terrain, a.W, a.H, d.conv_w, d.conv_b, i / kCo5, i % kCo5);
    }
    if (o < L.w2) return d.fc1_b[(o - L.b1) / 4];
    if (o < L.wh) return d.fc2_b[(o - L.b2) / 4];
    if (o < L.bh) {
        const size_t i = (o - L.wh) / 4;
        return i < (size_t)head_out * kH5 ? d.head_w[i] : 0.0f;
    }
    const size_t i = (o - L.bh) / 4;
    return i < (size_t)head_out ? d.head_b[i] : 0.0f;
}

// float i of a GBlob (the transposes of ocb_policy_set_weights' generic branch)
__device__ float pack_f32_generic(const PackArgs& a, const PackDesc& d, const GBlob& G, size_t i) {
    const int C = a.C, h = a.hidden, CO = h / 2, np = a.npos, head_out = d.net == 0 ? 6 : 1;
    if (i < G.conv_b) {
        const size_t x = i - G.conv_w;
        const int co = (int)(x % CO), c = (int)(x / CO % C), ij = (int)(x / CO / C);
        return d.conv_w[((size_t)(co * C + c) * 3 + ij / 3) * 3 + ij % 3];
    }
    if (i < G.w1) return d.conv_b[i - G.conv_b];
    if (i < G.b1) {
        const size_t x = i - G.w1;
        const int n = (int)(x % h), co = (int)(x / h % CO), pos = (int)(x / h / CO);
        return d.fc1_w[(size_t)n * (CO * np) + (size_t)co * np + pos];
    }
    if (i < G.w2) return d.fc1_b[i - G.b1];
    if (i < G.b2) {
        const size_t x = i - G.w2;
        return d.fc2_w[(x % h) * h + x / h];
    }
    if (i < G.wh) return d.fc2_b[i - G.b2];
    if (i < G.bh) {
        const size_t x = i - G.wh;
        return x / h < (size_t)head_out ? d.head_w[x] : 0.0f;
    }
    return i - G.bh < (size_t)head_out ? d.head_b[i - G.bh] : 0.0f;
}

// the zero-observation value of critic d (one block): zero_obs_fc1 / zero_obs_dot with the units spread over the threads
__device__ void pack_zero_value(const PackArgs& a, const PackDesc& d) {
    __shared__ float x1[kH5], x2[kH5];
    const int h = a.hidden;
    for (int o = threadIdx.x; o < h; o += blockDim.x) x1[o] = zero_obs_fc1(o, h, a.npos, d.conv_b, d.fc1_w, d.fc1_b);
    __syncthreads();
    for (int o = threadIdx.x; o < h; o += blockDim.x) x2[o] = fmaxf(zero_obs_dot(d.fc2_b[o], d.fc2_w + (size_t)o * h, x1, h), 0.0f);
    __syncthreads();
    if (threadIdx.x == 0) a.zero_value[d.policy] = zero_obs_dot(d.head_b[0], d.head_w, x2, h);
}

__global__ void __launch_bounds__(kPackThreads) policy_pack_kernel(const __grid_constant__ PackArgs a) {
    const PackDesc& d = a.d[blockIdx.y];
    if (blockIdx.x == gridDim.x - 1) {
        if (d.net == 1) pack_zero_value(a, d);
        return;
    }
    uint8_t* const b = d.dst;
    const int npos = a.npos;
    const size_t units = a.blob_bytes / 16, stride = (size_t)(gridDim.x - 1) * blockDim.x;
    for (size_t u = (size_t)blockIdx.x * blockDim.x + threadIdx.x; u < units; u += stride) {
        const size_t o = u * 16;
        float f[4];
        if (a.fmt == PACK_H64) {
            const BlobLayout L = blob_layout(npos);
            const int oi = (int)o;
            if (oi < L.wc_lo) {
                pack_split_row(b + L.wc_hi, b + L.wc_lo, oi / 16, kK1, [&](int n, int k) { return conv_slot_weight(d.conv_w, n, k); });
                continue;
            }
            if (oi < L.bias1) continue;
            if (oi >= L.head_bytes) {  // FC chunk c: [64 x 32] hi | lo; chunks npos, npos + 1 = the K halves of W2
                const int c = (oi - L.head_bytes) / kChunk, r = (oi - L.head_bytes) % kChunk;
                if (r >= kChunk / 2) continue;
                uint8_t* hi = b + L.head_bytes + (size_t)c * kChunk;
                if (c < npos)
                    pack_split_row(hi, hi + kChunk / 2, r / 16, kCo,
                                   [&](int n, int k) { return d.fc1_w[(size_t)n * (kCo * npos) + k * npos + c]; });
                else
                    pack_split_row(hi, hi + kChunk / 2, r / 16, 32,
                                   [&](int n, int k) { return d.fc2_w[n * kHid + (c - npos) * 32 + k]; });
                continue;
            }
            for (int j = 0; j < 4; ++j) f[j] = pack_f32_h64(a, d, L, oi + 4 * j);
        } else if (a.fmt == PACK_H512) {
            const Blob5 L = blob5_layout(npos);
            if (o < L.wc_lo) {
                pack_split_row(b + L.wc_hi, b + L.wc_lo, (int)(o / 16), kK1, [&](int n, int k) { return conv_slot_weight(d.conv_w, n, k); });
                continue;
            }
            if (o < L.bias1) continue;
            const bool in_w1 = o >= L.w1 && o < L.b1, in_w2 = o >= L.w2 && o < L.b2;
            if (in_w1 || in_w2) {  // K block kc: [512 x 16] hi | lo
                const size_t base = in_w1 ? L.w1 : L.w2;
                const int kc = (int)((o - base) / kWBlk), r = (int)((o - base) % kWBlk);
                if (r >= kWBlk / 2) continue;
                uint8_t* hi = b + base + (size_t)kc * kWBlk;
                if (in_w1)  // packed K index k = pos * 256 + co
                    pack_split_row(hi, hi + kWBlk / 2, r / 16, kKc, [&](int n, int k) {
                        const int kg = kc * kKc + k;
                        return d.fc1_w[(size_t)n * (kCo5 * npos) + (size_t)(kg % kCo5) * npos + kg / kCo5];
                    });
                else
                    pack_split_row(hi, hi + kWBlk / 2, r / 16, kKc, [&](int n, int k) { return d.fc2_w[(size_t)n * kH5 + kc * kKc + k]; });
                continue;
            }
            for (int j = 0; j < 4; ++j) f[j] = pack_f32_h512(a, d, L, o + 4 * j);
        } else {
            const GBlob G = gblob_layout(a.C, a.hidden, npos);
            for (int j = 0; j < 4; ++j) f[j] = pack_f32_generic(a, d, G, u * 4 + j);
        }
        *reinterpret_cast<float4*>(b + o) = make_float4(f[0], f[1], f[2], f[3]);
    }
}

}  // namespace

struct ocb_policy {
    int device;
    int W, H, S, SC, C, npos, n_policies;
    int sm_count, stage_stride;
    int pair_ring;            // weight-ring slots of policy_pair_kernel (0 for hidden 512 and the generic kernel)
    size_t pair_smem_bytes;
    std::vector<uint8_t> terrain;
    BlobLayout L;
    uint8_t* d_blobs;
    uint64_t calls;
    // hidden_size 512 (policy512.cuh): packed blobs in d_blobs, activation scratch sized for the largest M seen
    int hidden;
    Blob5 L5;
    uint8_t* d_scratch;
    size_t scratch_tiles;
    // critic value of the all-zero observation per weight set, on the device (a constant of the weights, written by
    // whichever path packs the critic; the mixed-play buffer bootstraps from the never-written slot L, which holds zeros in
    // the reference, and reads it when the launch runs, so a replayed graph sees the current critic)
    float* d_zero_value = nullptr;
    uint8_t* d_terrain = nullptr;  // [S] terrain codes, for the device-side fold of the static planes
    uint32_t rng_rows_per_seat = 0, rng_add0 = 0, rng_add1 = 0;  // ocb_policy_set_sampling_rows
    // generic mode (policy_generic.cuh): shapes outside the tensor-core kernels' range (P != 2, H > 6, one conv position)
    int generic = 0;
    GBlob LG;
    float* d_gblobs = nullptr;
};

extern "C" int ocb_policy_destroy(ocb_policy* p) {
    if (p == nullptr) return OCB_OK;
    DeviceGuard guard(p->device);
    CaptureRelaxed relaxed;  // safe while another stream is being captured
    cudaFree(p->d_scratch);
    cudaFree(p->d_blobs);
    cudaFree(p->d_gblobs);
    cudaFree(p->d_zero_value);
    cudaFree(p->d_terrain);
    delete p;
    return OCB_OK;
}

int ocb_policy_num_sets(const ocb_policy* p) { return p ? p->n_policies : 0; }
int ocb_policy_obs_bytes(const ocb_policy* p) { return p ? p->SC : 0; }
int ocb_policy_is_generic(const ocb_policy* p) { return p ? p->generic : 0; }
const float* ocb_policy_zero_value_device(const ocb_policy* p, int policy) {
    return (p && policy >= 0 && policy < p->n_policies) ? p->d_zero_value + policy : nullptr;
}

// the zero-observation critic value on the host (the rules of pack_zero_value, one unit after the other)
static float zero_obs_value(int hidden, int npos, const float* conv_b, const float* fc1_w, const float* fc1_b,
                            const float* fc2_w, const float* fc2_b, const float* head_w, const float* head_b) {
    std::vector<float> x1((size_t)hidden), x2((size_t)hidden);
    for (int o = 0; o < hidden; ++o) x1[o] = zero_obs_fc1(o, hidden, npos, conv_b, fc1_w, fc1_b);
    for (int o = 0; o < hidden; ++o) x2[o] = fmaxf(zero_obs_dot(fc2_b[o], fc2_w + (size_t)o * hidden, x1.data(), hidden), 0.0f);
    return zero_obs_dot(head_b[0], head_w, x2.data(), hidden);
}

extern "C" int ocb_policy_create(const ocb_config* cfg, int device, int hidden, int n_policies, ocb_policy** out) {
    if (out == nullptr || cfg == nullptr) return fail(OCB_ERR_INVALID_ARG, "NULL argument");
    *out = nullptr;
    if (cfg->struct_size != sizeof(ocb_config)) return fail(OCB_ERR_INVALID_ARG, "ocb_config ABI mismatch");
    if (hidden != kHid && hidden != kH5)
        return fail(OCB_ERR_UNSUPPORTED, "the policy kernels support hidden_size 64 and 512 (got %d)", hidden);
    if (cfg->num_players < 1 || cfg->num_players > OCB_MAX_PLAYERS) return fail(OCB_ERR_BAD_LAYOUT, "1..%d players", OCB_MAX_PLAYERS);
    if (cfg->width < 3 || cfg->height < 3) return fail(OCB_ERR_BAD_LAYOUT, "grid smaller than the 3x3 convolution");
    if (cfg->width * cfg->height > OCB_MAX_CELLS) return fail(OCB_ERR_BAD_LAYOUT, "grid larger than OCB_MAX_CELLS");
    if (n_policies < 1 || n_policies > 4096) return fail(OCB_ERR_INVALID_ARG, "n_policies out of range");
    // Shapes the tensor-core kernels do not take (they pack 2-player observations and need a grid column per warp-wide
    // load) run the same networks through policy_generic_kernel (fp32 CUDA cores): schelling, corridor,
    // multiplayer_schelling, simple_single ...  OCB_POLICY_GENERIC=1 forces that path (tests compare the two).
    bool generic = cfg->num_players != 2 || cfg->height > kMaxH || (cfg->width - 2) * (cfg->height - 2) < 2;
    if (const char* e = getenv("OCB_POLICY_GENERIC")) generic = generic || e[0] == '1';
    const int ndev = ocb_device_count();
    if (ndev <= 0) return fail(OCB_ERR_NO_DEVICE, "no CUDA device available (this library has no CPU path)");
    if (device < 0 || device >= ndev) return fail(OCB_ERR_INVALID_ARG, "device %d not in 0..%d", device, ndev - 1);
    ocb_policy* p = new (std::nothrow) ocb_policy();
    if (p == nullptr) return fail(OCB_ERR_INVALID_ARG, "out of host memory");
    p->device = device, p->W = cfg->width, p->H = cfg->height, p->S = p->W * p->H, p->C = 5 * cfg->num_players + 10;
    p->SC = p->S * p->C;
    p->generic = generic ? 1 : 0;
    p->npos = (p->W - 2) * (p->H - 2), p->n_policies = n_policies, p->calls = 0, p->d_blobs = nullptr;
    p->hidden = hidden, p->d_scratch = nullptr, p->scratch_tiles = 0, p->L5 = blob5_layout(p->npos);
    p->pair_ring = 0, p->pair_smem_bytes = 0;
    p->terrain.assign(cfg->terrain, cfg->terrain + p->S);
    p->L = blob_layout(p->npos);
    p->stage_stride = (5 * p->H) | 1;
    if (generic) {
        p->LG = gblob_layout(p->C, hidden, p->npos);
        if (generic_smem_bytes(p->SC, hidden) > (size_t)kSmemBudget) {
            delete p;
            return fail(OCB_ERR_UNSUPPORTED, "layout too large for the generic policy kernel (%d x %d)", cfg->width, cfg->height);
        }
    } else if (hidden == kHid) {
        // weight ring over the FC chunks of both networks: as many 8 KB slots as fit; all of them (resident weights) when
        // possible.  Every layout with H <= kMaxH and at most OCB_MAX_CELLS cells leaves room for 8 or more.
        int ring = (kSmemBudget - pair_smem_layout(p->npos, 0, p->stage_stride).total) / kChunk;
        if (ring > kPMaxRing) ring = kPMaxRing;
        if (ring > 2 * p->L.chunks) ring = 2 * p->L.chunks;
        if (ring < 4) {
            delete p;
            return fail(OCB_ERR_UNSUPPORTED, "layout too large for the fused policy kernel (%d x %d)", cfg->width, cfg->height);
        }
        p->pair_ring = ring;
        p->pair_smem_bytes = (size_t)pair_smem_layout(p->npos, ring, p->stage_stride).total;
    } else if (c5_smem_layout(p->npos, p->stage_stride).total > kSmemBudget + 128) {
        delete p;
        return fail(OCB_ERR_UNSUPPORTED, "layout too large for the hidden-512 conv kernel (%d x %d)", cfg->width, cfg->height);
    }
    DeviceGuard guard(device);
    const size_t bytes = generic ? 256 : (size_t)n_policies * 2 * (hidden == kHid ? (size_t)p->L.total : p->L5.total);
    cudaError_t err = cudaDeviceGetAttribute(&p->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (err == cudaSuccess) err = cudaMalloc(&p->d_blobs, bytes);
    if (err == cudaSuccess) err = cudaMemset(p->d_blobs, 0, bytes);
    if (err == cudaSuccess) err = cudaMalloc(&p->d_zero_value, (size_t)n_policies * sizeof(float));
    if (err == cudaSuccess) err = cudaMemset(p->d_zero_value, 0, (size_t)n_policies * sizeof(float));
    if (err == cudaSuccess) err = cudaMalloc(&p->d_terrain, (size_t)p->S);
    if (err == cudaSuccess) err = cudaMemcpy(p->d_terrain, p->terrain.data(), (size_t)p->S, cudaMemcpyHostToDevice);
    if (generic) {
        const size_t gbytes = (size_t)n_policies * 2 * p->LG.total * sizeof(float);
        if (err == cudaSuccess) err = cudaMalloc(&p->d_gblobs, gbytes);
        if (err == cudaSuccess) err = cudaMemset(p->d_gblobs, 0, gbytes);
        if (err == cudaSuccess) err = cudaFuncSetAttribute(policy_generic_kernel<kHid>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget + 128);
        if (err == cudaSuccess) err = cudaFuncSetAttribute(policy_generic_kernel<kH5>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget + 128);
    }
    // the opt-in limit is per function, not per handle: always raise it to the full budget
    const int smem_max = kSmemBudget + 128;
    if (err == cudaSuccess) err = cudaFuncSetAttribute(policy_pair_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(policy_pair_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(policy_pair_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(rollout_fused_kernel<false, false, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(rollout_fused_kernel<true, false, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(rollout_fused_kernel<false, true, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(rollout_fused_kernel<true, true, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(rollout_fused_kernel<false, false, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(rollout_fused_kernel<true, false, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(rollout_fused_kernel<false, false, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(rollout_fused_kernel<false, true, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(rollout_fused_kernel<false, false, 2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(rollout_fused_kernel<false, false, 1, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(rollout_fused_kernel<false, false, 2, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(conv512_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(gemm512_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(gemm512_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
    if (err != cudaSuccess) {
        cudaGetLastError();
        ocb_policy_destroy(p);
        return fail(OCB_ERR_CUDA, "ocb_policy_create: %s", cudaGetErrorString(err));
    }
    *out = p;
    return OCB_OK;
}

// hidden 512: weights in the reference's layouts (conv_w [256,20,3,3], fc1_w [512, 256*npos] with column
// co*npos + pos, fc2_w [512,512], head_w [head_out,512]) -> Blob5 (policy512.cuh)
static int set_weights512(ocb_policy* p, int policy, int net, const float* conv_w, const float* conv_b, const float* fc1_w,
                          const float* fc1_b, const float* fc2_w, const float* fc2_b, const float* head_w, const float* head_b) {
    const Blob5& L = p->L5;
    std::vector<uint8_t> blob(L.total, 0);
    const int npos = p->npos;
    for (int co = 0; co < kCo5; ++co)
        for (int k = 0; k < kK1; ++k)
            put_split(blob.data() + L.wc_hi, blob.data() + L.wc_lo, canon_off(co, k, kK1), conv_slot_weight(conv_w, co, k));
    float* bias1 = reinterpret_cast<float*>(blob.data() + L.bias1);
    for (int pos = 0; pos < npos; ++pos)
        for (int co = 0; co < kCo5; ++co)
            bias1[pos * kCo5 + co] = terrain_bias(p->terrain.data(), p->W, p->H, conv_w, conv_b, pos, co);
    // FC1: packed K index k = pos * 256 + co; block kc holds k in [32 kc, 32 kc + 32)
    const int K1 = kCo5 * npos;
    for (int n = 0; n < kH5; ++n) {
        for (int k = 0; k < K1; ++k) {
            const int pos = k / kCo5, co = k % kCo5;
            uint8_t* blk = blob.data() + L.w1 + (size_t)(k / kKc) * kWBlk;
            put_split(blk, blk + kWBlk / 2, canon_off(n, k % kKc, kKc), fc1_w[(size_t)n * K1 + (size_t)co * npos + pos]);
        }
        for (int k = 0; k < kH5; ++k) {
            uint8_t* blk = blob.data() + L.w2 + (size_t)(k / kKc) * kWBlk;
            put_split(blk, blk + kWBlk / 2, canon_off(n, k % kKc, kKc), fc2_w[(size_t)n * kH5 + k]);
        }
    }
    memcpy(blob.data() + L.b1, fc1_b, kH5 * 4);
    memcpy(blob.data() + L.b2, fc2_b, kH5 * 4);
    const int head_out = net == 0 ? 6 : 1;
    memcpy(blob.data() + L.wh, head_w, (size_t)head_out * kH5 * 4);
    memcpy(blob.data() + L.wh + 8 * kH5 * 4, head_b, (size_t)head_out * 4);  // bh follows wh
    DeviceGuard guard(p->device);
    cudaError_t err = cudaMemcpy(p->d_blobs + ((size_t)policy * 2 + net) * L.total, blob.data(), L.total, cudaMemcpyHostToDevice);
    if (err != cudaSuccess) {
        cudaGetLastError();
        return fail(OCB_ERR_CUDA, "ocb_policy_set_weights: %s", cudaGetErrorString(err));
    }
    return OCB_OK;
}

// activation scratch of the hidden-512 forward for `tiles` row tiles (grow only)
static int reserve512(ocb_policy* p, size_t tiles, cudaStream_t stream) {
    if (tiles <= p->scratch_tiles) return OCB_OK;
    // growing is not possible while the stream is being captured
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(stream, &cs);
    if (cs != cudaStreamCaptureStatusNone)
        return fail(OCB_ERR_INVALID_ARG, "hidden-512 scratch must grow: call ocb_policy_reserve before capturing a graph");
    cudaError_t e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaFree(p->d_scratch);
    p->d_scratch = nullptr, p->scratch_tiles = 0;
    const size_t bytes = 2 * tiles * ((size_t)p->L5.kc1 + kKc2) * kABlk;
    if (e == cudaSuccess) e = cudaMalloc(&p->d_scratch, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(OCB_ERR_CUDA, "hidden-512 scratch (%zu bytes): %s", bytes, cudaGetErrorString(e));
    }
    p->scratch_tiles = tiles;
    return OCB_OK;
}

// the three launches of the hidden-512 forward
static int policy_launch512(ocb_policy* p, PolicyParams& prm, cudaStream_t stream) {
    const size_t tiles = (size_t)prm.tiles;
    const int rrc = reserve512(p, tiles, stream);
    if (rrc != OCB_OK) return rrc;
    P5Params q;
    prm.blobs = p->d_blobs, prm.blob_stride = p->L5.total;
    q.base = prm;
    q.kc1 = p->L5.kc1;
    q.a1 = p->d_scratch;
    q.a2 = p->d_scratch + 2 * tiles * (size_t)p->L5.kc1 * kABlk;
    int ctas;
    if (prm.net_mask == 3) {
        const int per_net = prm.tiles < p->sm_count / 2 ? prm.tiles : p->sm_count / 2;
        ctas = 2 * per_net;
    } else {
        ctas = prm.tiles < p->sm_count ? prm.tiles : p->sm_count;
    }
    conv512_kernel<<<ctas, kThreads, c5_smem_layout(p->npos, p->stage_stride).total, stream>>>(q);
    // FC1 in one pass over K (two passes measured 2-4 % slower there: it streams 3 x the weights of FC2 and sits near the L2
    // bound), FC2 + head in two (policy512.cuh)
    gemm512_kernel<false, false><<<ctas, kGThreads, g5_smem_layout().total, stream>>>(q);
    gemm512_kernel<true, true><<<ctas, kGThreads, g5_smem_layout().total, stream>>>(q);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return fail(OCB_ERR_CUDA, "hidden-512 policy launch failed: %s", cudaGetErrorString(err));
    p->calls += 1;
    return OCB_OK;
}

// pre-size internal scratch for forwards of up to M rows (no-op for hidden 64, which has none)
extern "C" int ocb_policy_reserve(ocb_policy* p, int M) {
    if (p == nullptr || M < 1) return fail(OCB_ERR_INVALID_ARG, "bad handle / M");
    if (p->hidden != kH5 || p->generic) return OCB_OK;
    DeviceGuard guard(p->device);
    return reserve512(p, (size_t)((M + kRows - 1) / kRows), nullptr);
}

// weights in the reference's layouts (HOST fp32): conv_w [32,20,3,3], conv_b [32], fc1_w [64, 32*npos]
// (column = co*npos + pos), fc1_b [64], fc2_w [64,64], fc2_b [64], head_w [head_out,64], head_b [head_out];
// net 0 = actor (head_out 6), 1 = critic (head_out 1)
extern "C" int ocb_policy_set_weights(ocb_policy* p, int policy, int net, const float* conv_w, const float* conv_b,
                                      const float* fc1_w, const float* fc1_b, const float* fc2_w, const float* fc2_b,
                                      const float* head_w, const float* head_b) {
    if (p == nullptr || !conv_w || !conv_b || !fc1_w || !fc1_b || !fc2_w || !fc2_b || !head_w || !head_b)
        return fail(OCB_ERR_INVALID_ARG, "NULL argument");
    if (policy < 0 || policy >= p->n_policies || net < 0 || net > 1) return fail(OCB_ERR_INVALID_ARG, "bad policy / net index");
    if (net == 1) {
        const float v = zero_obs_value(p->hidden, p->npos, conv_b, fc1_w, fc1_b, fc2_w, fc2_b, head_w, head_b);
        DeviceGuard guard(p->device);
        const cudaError_t err = cudaMemcpy(p->d_zero_value + policy, &v, sizeof(float), cudaMemcpyHostToDevice);
        if (err != cudaSuccess) {
            cudaGetLastError();
            return fail(OCB_ERR_CUDA, "ocb_policy_set_weights: %s", cudaGetErrorString(err));
        }
    }
    if (p->generic) {  // fp32, transposed so that consecutive output units are consecutive words (policy_generic.cuh)
        const GBlob& G = p->LG;
        const int C = p->C, h = p->hidden, CO = h / 2, np = p->npos, head_out = net == 0 ? 6 : 1;
        std::vector<float> blob(G.total, 0.0f);
        for (int co = 0; co < CO; ++co) {
            blob[G.conv_b + co] = conv_b[co];
            for (int c = 0; c < C; ++c)
                for (int i = 0; i < 3; ++i)
                    for (int j = 0; j < 3; ++j)
                        blob[G.conv_w + (size_t)((i * 3 + j) * C + c) * CO + co] = conv_w[((size_t)(co * C + c) * 3 + i) * 3 + j];
        }
        for (int n = 0; n < h; ++n) {
            blob[G.b1 + n] = fc1_b[n], blob[G.b2 + n] = fc2_b[n];
            for (int pos = 0; pos < np; ++pos)
                for (int co = 0; co < CO; ++co)
                    blob[G.w1 + ((size_t)pos * CO + co) * h + n] = fc1_w[(size_t)n * (CO * np) + (size_t)co * np + pos];
            for (int k = 0; k < h; ++k) blob[G.w2 + (size_t)k * h + n] = fc2_w[(size_t)n * h + k];
        }
        for (int a = 0; a < head_out; ++a) {
            blob[G.bh + a] = head_b[a];
            for (int k = 0; k < h; ++k) blob[G.wh + (size_t)a * h + k] = head_w[(size_t)a * h + k];
        }
        DeviceGuard guard(p->device);
        cudaError_t err = cudaMemcpy(p->d_gblobs + ((size_t)policy * 2 + net) * G.total, blob.data(), G.total * sizeof(float),
                                     cudaMemcpyHostToDevice);
        if (err != cudaSuccess) {
            cudaGetLastError();
            return fail(OCB_ERR_CUDA, "ocb_policy_set_weights: %s", cudaGetErrorString(err));
        }
        return OCB_OK;
    }
    if (p->hidden == kH5) return set_weights512(p, policy, net, conv_w, conv_b, fc1_w, fc1_b, fc2_w, fc2_b, head_w, head_b);
    const BlobLayout& L = p->L;
    std::vector<uint8_t> blob((size_t)L.total, 0);
    const int npos = p->npos;
    for (int co = 0; co < kCo; ++co)
        for (int k = 0; k < kK1; ++k)
            put_split(blob.data() + L.wc_hi, blob.data() + L.wc_lo, canon_off(co, k, kK1), conv_slot_weight(conv_w, co, k));
    // the static terrain planes folded into a per-position bias
    float* bias1 = reinterpret_cast<float*>(blob.data() + L.bias1);
    for (int pos = 0; pos < npos; ++pos)
        for (int co = 0; co < kCo; ++co) bias1[pos * kCo + co] = terrain_bias(p->terrain.data(), p->W, p->H, conv_w, conv_b, pos, co);
    // FC chunks: chunk pos = W1 of that position [64 x 32]; chunks npos, npos+1 = the K halves of W2 [64 x 32]
    uint8_t* chunks = blob.data() + L.head_bytes;
    for (int n = 0; n < kHid; ++n) {
        for (int pos = 0; pos < npos; ++pos)
            for (int co = 0; co < kCo; ++co)
                put_split(chunks + (size_t)pos * kChunk, chunks + (size_t)pos * kChunk + 4096, canon_off(n, co, kCo),
                          fc1_w[(size_t)n * (kCo * npos) + co * npos + pos]);
        for (int k = 0; k < kHid; ++k) {
            uint8_t* c = chunks + (size_t)(npos + k / 32) * kChunk;
            put_split(c, c + 4096, canon_off(n, k % 32, 32), fc2_w[n * kHid + k]);
        }
    }
    memcpy(blob.data() + L.b1, fc1_b, kHid * 4);
    memcpy(blob.data() + L.b2, fc2_b, kHid * 4);
    const int head_out = net == 0 ? 6 : 1;
    float* whp = reinterpret_cast<float*>(blob.data() + L.wh);
    if (net == 0) {  // actor: hidden-major [64][8] (head_accumulate)
        for (int i = 0; i < kHid; ++i)
            for (int a = 0; a < head_out; ++a) whp[i * 8 + a] = head_w[(size_t)a * kHid + i];
    } else {
        memcpy(whp, head_w, (size_t)kHid * 4);
    }
    memcpy(blob.data() + L.bh, head_b, (size_t)head_out * 4);
    DeviceGuard guard(p->device);
    cudaError_t err = cudaMemcpy(p->d_blobs + ((size_t)policy * 2 + net) * L.total, blob.data(), (size_t)L.total,
                                 cudaMemcpyHostToDevice);
    if (err != cudaSuccess) {
        cudaGetLastError();
        return fail(OCB_ERR_CUDA, "ocb_policy_set_weights: %s", cudaGetErrorString(err));
    }
    return OCB_OK;
}

// blob of (policy, net) and its size in bytes, in whichever of the three formats the handle uses
static uint8_t* blob_of(const ocb_policy* p, int policy, int net, size_t* bytes) {
    const size_t unit = (size_t)policy * 2 + net;
    if (p->generic) {
        *bytes = p->LG.total * sizeof(float);
        return reinterpret_cast<uint8_t*>(p->d_gblobs + unit * p->LG.total);
    }
    *bytes = p->hidden == kH5 ? p->L5.total : (size_t)p->L.total;
    return p->d_blobs + unit * *bytes;
}

// a weight pointer of ocb_policy_set_weights_device: 4-byte aligned device (or managed) memory of the handle's device
static int check_weight_ptr(const ocb_policy* p, int i, const char* name, const float* ptr) {
    if (ptr == nullptr) return fail(OCB_ERR_INVALID_ARG, "ocb_policy_set_weights_device: src[%d].%s is NULL", i, name);
    if ((reinterpret_cast<uintptr_t>(ptr) & 3u) != 0)
        return fail(OCB_ERR_INVALID_ARG, "ocb_policy_set_weights_device: src[%d].%s is not 4-byte aligned", i, name);
    cudaPointerAttributes at;
    const cudaError_t err = cudaPointerGetAttributes(&at, ptr);
    if (err != cudaSuccess) {
        cudaGetLastError();
        return fail(OCB_ERR_INVALID_ARG, "ocb_policy_set_weights_device: src[%d].%s: %s", i, name, cudaGetErrorString(err));
    }
    if ((at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged) || at.device != p->device)
        return fail(OCB_ERR_INVALID_ARG, "ocb_policy_set_weights_device: src[%d].%s is not device memory of device %d", i, name,
                    p->device);
    return OCB_OK;
}

// DEVICE fp32 weights -> the same blobs (and zero-observation values) as ocb_policy_set_weights, on `stream`
extern "C" int ocb_policy_set_weights_device(ocb_policy* p, int n, const ocb_weight_src* src, void* stream) {
    if (p == nullptr || src == nullptr) return fail(OCB_ERR_INVALID_ARG, "ocb_policy_set_weights_device: NULL argument");
    if (n < 1) return fail(OCB_ERR_INVALID_ARG, "ocb_policy_set_weights_device: n must be >= 1 (got %d)", n);
    DeviceGuard guard(p->device);
    CaptureRelaxed relaxed;  // the pointer queries below while `stream` may be capturing a graph
    std::vector<uint8_t> seen((size_t)p->n_policies * 2, 0);
    for (int i = 0; i < n; ++i) {
        const ocb_weight_src& w = src[i];
        if (w.policy < 0 || w.policy >= p->n_policies || w.net < 0 || w.net > 1)
            return fail(OCB_ERR_INVALID_ARG, "ocb_policy_set_weights_device: src[%d] has policy %d / net %d (the handle holds %d sets, "
                        "nets 0 and 1)", i, w.policy, w.net, p->n_policies);
        if (seen[(size_t)w.policy * 2 + w.net]++)
            return fail(OCB_ERR_INVALID_ARG, "ocb_policy_set_weights_device: policy %d net %d appears twice", w.policy, w.net);
        const char* names[8] = {"conv_w", "conv_b", "fc1_w", "fc1_b", "fc2_w", "fc2_b", "head_w", "head_b"};
        const float* ptrs[8] = {w.conv_w, w.conv_b, w.fc1_w, w.fc1_b, w.fc2_w, w.fc2_b, w.head_w, w.head_b};
        for (int k = 0; k < 8; ++k) {
            const int rc = check_weight_ptr(p, i, names[k], ptrs[k]);
            if (rc != OCB_OK) return rc;
        }
    }
    PackArgs a;
    a.fmt = p->generic ? PACK_GENERIC : p->hidden == kH5 ? PACK_H512 : PACK_H64;
    a.W = p->W, a.H = p->H, a.C = p->C, a.npos = p->npos, a.hidden = p->hidden;
    a.terrain = p->d_terrain, a.zero_value = p->d_zero_value;
    blob_of(p, 0, 0, &a.blob_bytes);
    const size_t units = a.blob_bytes / 16;
    const unsigned bx = (unsigned)(units < (size_t)kPackThreads * kPackMaxBlocks ? (units + kPackThreads - 1) / kPackThreads
                                                                                  : kPackMaxBlocks);
    for (int i0 = 0; i0 < n; i0 += kPackMax) {
        a.n = n - i0 < kPackMax ? n - i0 : kPackMax;
        for (int j = 0; j < a.n; ++j) {
            const ocb_weight_src& w = src[i0 + j];
            PackDesc& d = a.d[j];
            size_t bytes;
            d.dst = blob_of(p, w.policy, w.net, &bytes);
            d.conv_w = w.conv_w, d.conv_b = w.conv_b, d.fc1_w = w.fc1_w, d.fc1_b = w.fc1_b;
            d.fc2_w = w.fc2_w, d.fc2_b = w.fc2_b, d.head_w = w.head_w, d.head_b = w.head_b;
            d.policy = w.policy, d.net = w.net;
        }
        policy_pack_kernel<<<dim3(bx + 1, (unsigned)a.n), kPackThreads, 0, (cudaStream_t)stream>>>(a);
        const cudaError_t err = cudaGetLastError();
        if (err != cudaSuccess) return fail(OCB_ERR_CUDA, "ocb_policy_set_weights_device: %s", cudaGetErrorString(err));
    }
    return OCB_OK;
}

extern "C" int ocb_policy_read_blob(ocb_policy* p, int policy, int net, void* dst, size_t bytes, void* stream) {
    if (p == nullptr) return fail(OCB_ERR_INVALID_ARG, "NULL handle");
    if (policy < 0 || policy >= p->n_policies || net < 0 || net > 1) return fail(OCB_ERR_INVALID_ARG, "bad policy / net index");
    size_t total;
    const uint8_t* blob = blob_of(p, policy, net, &total);
    if (dst == nullptr) return (int)total;
    if (bytes < total) return fail(OCB_ERR_INVALID_ARG, "ocb_policy_read_blob: dst holds %zu bytes, the blob has %zu", bytes, total);
    DeviceGuard guard(p->device);
    const cudaError_t err = cudaMemcpyAsync(dst, blob, total, cudaMemcpyDeviceToDevice, (cudaStream_t)stream);
    if (err != cudaSuccess) {
        cudaGetLastError();
        return fail(OCB_ERR_CUDA, "ocb_policy_read_blob: %s", cudaGetErrorString(err));
    }
    return (int)total;
}

// evaluate_actions extras of ocb_policy_evaluate
struct EvalArgs {
    const int32_t* row_index;
    const int32_t* given_actions;
    float* entropy;
};

static int policy_launch(ocb_policy* p, int net_mask, const int8_t* obs, int M, const int32_t* tile_policy, float* logits,
                         int32_t* actions, float* logp, float* values, int deterministic, uint64_t seed, uint64_t offset,
                         const uint64_t* d_offset, void* stream, long long* prof = nullptr, int* ctas_out = nullptr,
                         const EvalArgs* ev = nullptr, int policy_index = 0) {
    if (p == nullptr || obs == nullptr) return fail(OCB_ERR_INVALID_ARG, "NULL argument");
    if (M < 1) return fail(OCB_ERR_INVALID_ARG, "M must be >= 1");
    if (!p->generic && (reinterpret_cast<uintptr_t>(obs) & 3u) != 0) return fail(OCB_ERR_INVALID_ARG, "obs must be 4-byte aligned");
    DeviceGuard guard(p->device);
    PolicyParams prm;
    memset(&prm, 0, sizeof(prm));
    prm.blobs = p->d_blobs + (size_t)policy_index * 2 * (size_t)p->L.total, prm.blob_stride = (size_t)p->L.total;
    prm.W = p->W, prm.H = p->H, prm.S = p->S, prm.SC = p->SC, prm.npos = p->npos;
    prm.obs = obs, prm.M = M, prm.tiles = (M + kRows - 1) / kRows, prm.tile_policy = tile_policy;
    prm.logits = logits, prm.actions = actions, prm.logp = logp, prm.values = values;
    prm.deterministic = deterministic, prm.seed = seed, prm.offset = offset;
    prm.rng_rows_per_seat = p->rng_rows_per_seat, prm.rng_add0 = p->rng_add0, prm.rng_add1 = p->rng_add1;
    prm.d_offset = reinterpret_cast<const unsigned long long*>(d_offset);
    prm.net_mask = net_mask, prm.pair_ring = p->pair_ring, prm.stage_stride = p->stage_stride;
    prm.prof = prof;
    if (ev != nullptr) prm.row_index = ev->row_index, prm.given_actions = ev->given_actions, prm.entropy = ev->entropy;
    if (p->generic) {
        if (prof != nullptr) return fail(OCB_ERR_UNSUPPORTED, "the role profile exists for the tensor-core kernels only");
        GParams gp;
        gp.base = prm, gp.blobs = p->d_gblobs, gp.C = p->C, gp.hidden = p->hidden;
        const int ctas = (M + kGRows - 1) / kGRows;
        const size_t smem = generic_smem_bytes(p->SC, p->hidden);
        if (ctas_out) *ctas_out = ctas;
        if (p->hidden == kHid)
            policy_generic_kernel<kHid><<<ctas, kGenThreads, smem, (cudaStream_t)stream>>>(gp);
        else
            policy_generic_kernel<kH5><<<ctas, kGenThreads, smem, (cudaStream_t)stream>>>(gp);
        cudaError_t gerr = cudaGetLastError();
        if (gerr != cudaSuccess) return fail(OCB_ERR_CUDA, "generic policy kernel launch failed: %s", cudaGetErrorString(gerr));
        p->calls += 1;
        return OCB_OK;
    }
    if (p->hidden == kH5) {
        if (prof != nullptr) return fail(OCB_ERR_UNSUPPORTED, "the role profile exists for hidden 64 only");
        if (ctas_out) *ctas_out = 0;
        return policy_launch512(p, prm, (cudaStream_t)stream);
    }
    // persistent grid, one CTA per SM: both networks of a tile in one CTA, or the one asked for as one stream
    prm.single = net_mask == 3 ? 0 : net_mask;
    const int ctas = prm.tiles < p->sm_count ? prm.tiles : p->sm_count;
    if (ctas_out) *ctas_out = ctas;
    if (prof != nullptr)
        policy_pair_kernel<true><<<ctas, kPThreads, p->pair_smem_bytes, (cudaStream_t)stream>>>(prm);
    else
        policy_pair_kernel<false><<<ctas, kPThreads, p->pair_smem_bytes, (cudaStream_t)stream>>>(prm);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return fail(OCB_ERR_CUDA, "policy kernel launch failed: %s", cudaGetErrorString(err));
    p->calls += 1;
    return OCB_OK;
}

extern "C" int ocb_policy_act(ocb_policy* p, const int8_t* obs, int M, const int32_t* tile_policy, int32_t* actions,
                              float* logp, float* logits, int deterministic, uint64_t seed, uint64_t offset,
                              void* stream) {
    return policy_launch(p, 1, obs, M, tile_policy, logits, actions, logp, nullptr, deterministic, seed, offset, nullptr, stream);
}

extern "C" int ocb_policy_act_ex(ocb_policy* p, const int8_t* obs, int M, const int32_t* tile_policy, int32_t* actions,
                                 float* logp, float* logits, int deterministic, uint64_t seed, uint64_t offset,
                                 const uint64_t* d_offset, void* stream) {
    return policy_launch(p, 1, obs, M, tile_policy, logits, actions, logp, nullptr, deterministic, seed, offset, d_offset, stream);
}

extern "C" int ocb_policy_value(ocb_policy* p, const int8_t* obs, int M, const int32_t* tile_policy, float* values,
                                void* stream) {
    if (values == nullptr) return fail(OCB_ERR_INVALID_ARG, "values is NULL");
    return policy_launch(p, 2, obs, M, tile_policy, nullptr, nullptr, nullptr, values, 0, 0, 0, nullptr, stream);
}

extern "C" int ocb_policy_forward(ocb_policy* p, const int8_t* obs, int M, const int32_t* tile_policy, int32_t* actions,
                                  float* logp, float* logits, float* values, int deterministic, uint64_t seed,
                                  uint64_t offset, const uint64_t* d_offset, void* stream) {
    if (values == nullptr) return fail(OCB_ERR_INVALID_ARG, "values is NULL");
    return policy_launch(p, 3, obs, M, tile_policy, logits, actions, logp, values, deterministic, seed, offset, d_offset, stream);
}

// evaluate_actions over minibatch rows picked out of the rollout buffer in place (R_Actor.evaluate_actions
// r_actor_critic.py:73-109 + R_Critic.forward 178-197): same kernels as ocb_policy_forward, the loader follows `rows`,
// the actor epilogue scores the stored action and emits the entropy instead of sampling
extern "C" int ocb_policy_evaluate(ocb_policy* p, const int8_t* obs, const int32_t* rows, int B, const int32_t* tile_policy,
                                   const int32_t* actions_src, float* logp, float* entropy, float* logits, float* values,
                                   void* stream) {
    if (actions_src == nullptr || logp == nullptr) return fail(OCB_ERR_INVALID_ARG, "actions_src and logp are required");
    const EvalArgs ev = {rows, actions_src, entropy};
    return policy_launch(p, values != nullptr ? 3 : 1, obs, B, tile_policy, logits, nullptr, logp, values, 0, 0, 0, nullptr, stream,
                         nullptr, nullptr, &ev);
}

extern "C" int ocb_policy_set_sampling_rows(ocb_policy* p, uint32_t rows_per_seat, uint32_t add_seat0, uint32_t add_seat1) {
    if (p == nullptr) return fail(OCB_ERR_INVALID_ARG, "NULL handle");
    p->rng_rows_per_seat = rows_per_seat, p->rng_add0 = add_seat0, p->rng_add1 = add_seat1;
    return OCB_OK;
}

extern "C" int ocb_policy_info(const ocb_policy* p, int* ring_slots, int* chunks_per_unit, int* smem_bytes) {
    if (p == nullptr) return fail(OCB_ERR_INVALID_ARG, "policy is NULL");
    if (ring_slots) *ring_slots = p->pair_ring;
    if (chunks_per_unit) *chunks_per_unit = 2 * p->L.chunks;
    if (smem_bytes) *smem_bytes = (int)p->pair_smem_bytes;
    return OCB_OK;
}

int ocb_policy_value_of(ocb_policy* p, int policy_index, const int8_t* obs, int M, float* values, void* stream) {
    if (p == nullptr || values == nullptr) return fail(OCB_ERR_INVALID_ARG, "NULL argument");
    if (p->generic || p->hidden != kHid) return fail(OCB_ERR_UNSUPPORTED, "ocb_policy_value_of exists for the hidden-64 tensor-core path");
    if (policy_index < 0 || policy_index >= p->n_policies) return fail(OCB_ERR_INVALID_ARG, "policy index out of range");
    return policy_launch(p, 2, obs, M, nullptr, nullptr, nullptr, nullptr, values, 0, 0, 0, nullptr, stream, nullptr, nullptr,
                         nullptr, policy_index);
}

int ocb_policy_value_slab(ocb_policy* p, const int8_t* obs_slab, int steps, int seat_tiles, const int32_t* critic_policy,
                          float* values, void* stream) {
    if (p == nullptr || obs_slab == nullptr || critic_policy == nullptr || values == nullptr)
        return fail(OCB_ERR_INVALID_ARG, "NULL argument");
    if (p->generic || p->hidden != kHid) return fail(OCB_ERR_UNSUPPORTED, "the slab critic pass exists for the hidden-64 tensor-core path");
    if (steps < 1 || seat_tiles < 1) return fail(OCB_ERR_INVALID_ARG, "steps and seat_tiles must be >= 1");
    if ((long long)steps * seat_tiles * kRows > kSlabMaxRows)
        return fail(OCB_ERR_UNSUPPORTED, "the slab critic pass covers at most %d rows (got %d steps of %d rows)", kSlabMaxRows, steps,
                    seat_tiles * kRows);
    if ((reinterpret_cast<uintptr_t>(obs_slab) & 3u) != 0) return fail(OCB_ERR_INVALID_ARG, "obs_slab must be 4-byte aligned");
    DeviceGuard guard(p->device);
    PolicyParams prm;
    memset(&prm, 0, sizeof(prm));
    prm.blobs = p->d_blobs, prm.blob_stride = (size_t)p->L.total;
    prm.W = p->W, prm.H = p->H, prm.S = p->S, prm.SC = p->SC, prm.npos = p->npos;
    prm.obs = obs_slab, prm.M = steps * seat_tiles * kRows, prm.tiles = seat_tiles, prm.tile_policy = critic_policy;
    prm.values = values, prm.f_slots = steps;
    prm.net_mask = 2, prm.single = 2, prm.pair_ring = p->pair_ring, prm.stage_stride = p->stage_stride;
    const long long units = (long long)steps * seat_tiles;  // an upper bound: the table is only read on the device
    const int ctas = units < p->sm_count ? (int)units : p->sm_count;
    policy_pair_kernel<false, true><<<ctas, kPThreads, p->pair_smem_bytes, (cudaStream_t)stream>>>(prm);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return fail(OCB_ERR_CUDA, "slab critic pass launch failed: %s", cudaGetErrorString(err));
    p->calls += 1;
    return OCB_OK;
}

// Diagnostic: one fused forward with the instrumented build of the kernel.  h_prof (HOST, int64
// [max_ctas][4 roles: epilogue, loader, MMA, producer][16]) receives per role the total cycles ([0])
// and the cycles stalled on each hand-off (enum PW_* in policy_kernels.cu).  Returns the CTA count.
extern "C" int ocb_policy_debug_profile(ocb_policy* p, const int8_t* obs, int M, const int32_t* tile_policy, float* values,
                                        int32_t* actions, int64_t* h_prof, int max_ctas) {
    if (p == nullptr || h_prof == nullptr || values == nullptr) return fail(OCB_ERR_INVALID_ARG, "NULL argument");
    DeviceGuard guard(p->device);
    long long* d_prof = nullptr;
    const size_t n = (size_t)p->sm_count * 4 * PW_COUNT;
    if (max_ctas < p->sm_count) return fail(OCB_ERR_INVALID_ARG, "h_prof too small (%d CTAs needed)", p->sm_count);
    cudaError_t err = cudaMalloc(&d_prof, n * sizeof(long long));
    if (err == cudaSuccess) err = cudaMemset(d_prof, 0, n * sizeof(long long));
    int ctas = 0;
    int rc = OCB_OK;
    int mask = 3;  // OCB_PROFILE_MASK=1 / 2: the single-network mode (actor / critic)
    if (const char* e = getenv("OCB_PROFILE_MASK")) mask = (e[0] == '1') ? 1 : (e[0] == '2') ? 2 : 3;
    if (err == cudaSuccess)
        rc = policy_launch(p, mask, obs, M, tile_policy, nullptr, mask == 2 ? nullptr : actions, nullptr, mask == 1 ? nullptr : values, 1, 0, 0,
                           nullptr, nullptr, d_prof, &ctas);
    if (err == cudaSuccess && rc == OCB_OK) err = cudaMemcpy(h_prof, d_prof, n * sizeof(long long), cudaMemcpyDeviceToHost);
    cudaFree(d_prof);
    if (rc != OCB_OK) return rc;
    if (err != cudaSuccess) {
        cudaGetLastError();
        return fail(OCB_ERR_CUDA, "ocb_policy_debug_profile: %s", cudaGetErrorString(err));
    }
    return ctas;
}

// ---------------------------------------------------------------- fused rollout (rollout_fused.cuh)
// tile_policy == nullptr: self-play of weight set `policy_index` with its critic (obs_slab, actions and values required).
// tile_policy != nullptr: cross-play, the per-step path's seat-major table (int32 [2 N / 128], device); actors only, every
// output buffer optional.
// population: tile_policy is a table by 128-world slice (int32 [N / 128], device); slice s is self-play of weight set
// tile_policy[s] with its critic (obs_slab, actions and values required).
// mix != nullptr: mixed play of the actors of weight sets policy_index (main) and mix->partner_policy over T = 2 L steps,
// only the forced worlds recorded into [L, 2, N] buffers (obs_slab and actions required, no critic: values must be NULL).
int ocb_policy_rollout_fused_launch(ocb_policy* p, int policy_index, const int32_t* tile_policy, bool population,
                                    const RolloutParams& envp, int env_w, int env_h, int T, int8_t* obs_slab, int32_t* actions,
                                    float* logp, float* values, int32_t* reward, int32_t* done, int deterministic, uint64_t seed,
                                    const uint64_t* d_offset, uint64_t* d_counter, void* stream, long long* d_trace, int trace_u0,
                                    int trace_n, const FusedMixArgs* mix) {
    if (p == nullptr) return fail(OCB_ERR_INVALID_ARG, "policy is NULL");
    if (p->generic) return fail(OCB_ERR_UNSUPPORTED, "the fused rollout kernel needs the tensor-core policy path (2 players, grids up to %d rows)", kMaxH);
    if (p->hidden != kHid) return fail(OCB_ERR_UNSUPPORTED, "the fused rollout kernel exists for hidden_size 64 only");
    if (population && tile_policy == nullptr) return fail(OCB_ERR_INVALID_ARG, "slice_policy is NULL");
    const bool cross = tile_policy != nullptr && !population;
    const bool mixed = mix != nullptr;
    if (mixed && (tile_policy != nullptr || population || values != nullptr || d_trace != nullptr))
        return fail(OCB_ERR_INVALID_ARG, "mixed play takes no table, no critic and no trace");
    if (tile_policy == nullptr && (policy_index < 0 || policy_index >= p->n_policies)) return fail(OCB_ERR_INVALID_ARG, "policy index out of range");
    if (mixed && (mix->partner_policy < 0 || mix->partner_policy >= p->n_policies))
        return fail(OCB_ERR_INVALID_ARG, "policy index out of range");
    if (env_w != p->W || env_h != p->H) return fail(OCB_ERR_INVALID_ARG, "env and policy were built for different layouts");
    if (T < 1) return fail(OCB_ERR_INVALID_ARG, "T must be >= 1");
    if (mixed && (mix->L < 2 || T != 2 * mix->L || envp.N % (mix->L - 1) != 0))
        return fail(OCB_ERR_INVALID_ARG, "mixed play runs T = 2 L steps over a multiple of L - 1 worlds");
    if (mixed && (obs_slab == nullptr || actions == nullptr)) return fail(OCB_ERR_INVALID_ARG, "obs_buf and actions are required");
    if (!cross && !mixed && (obs_slab == nullptr || actions == nullptr || values == nullptr))
        return fail(OCB_ERR_INVALID_ARG, "obs_slab, actions and values are required");
    if (cross && (envp.N % kRows) != 0)
        return fail(OCB_ERR_INVALID_ARG, "cross-play needs a multiple of %d worlds (one weight set per 128-row tile of a seat), got %d", kRows, envp.N);
    if (population && (envp.N % kRows) != 0)
        return fail(OCB_ERR_INVALID_ARG, "population self-play needs a multiple of %d worlds (one weight set per slice), got %d", kRows, envp.N);
    if (cross && values != nullptr) return fail(OCB_ERR_INVALID_ARG, "the cross-play rollout runs no critic: values must be NULL");
    const int wtiles = (envp.N + kFWorlds - 1) / kFWorlds;
    // two tiles in flight when there are more tiles than SMs and the second tile's planes leave a usable weight ring
    int slots = 1;
    {
        const int fixed2 = fused_smem_layout(p->npos, 0, p->S, p->SC, 2).total;
        const bool fits2 = fixed2 <= kSmemBudget && (kSmemBudget - fixed2) / kChunk >= 4;
        const char* e = getenv("OCB_FUSED_SLOTS");
        const bool want2 = e != nullptr ? (e[0] == '2') : (wtiles > p->sm_count);
        if (want2 && fits2) slots = 2;
    }
    const int fixed = fused_smem_layout(p->npos, 0, p->S, p->SC, slots).total;
    int ring = (kSmemBudget - fixed) / kChunk;
    if (ring > kPMaxRing) ring = kPMaxRing;
    if (ring > 2 * p->L.chunks) ring = 2 * p->L.chunks;
    if (fixed > kSmemBudget || ring < 4)
        return fail(OCB_ERR_UNSUPPORTED, "layout too large for the fused rollout kernel (%d x %d)", p->W, p->H);
    DeviceGuard guard(p->device);
    FusedParams fp;
    memset(&fp, 0, sizeof(fp));
    fp.pol.blobs = tile_policy != nullptr ? p->d_blobs : p->d_blobs + (size_t)policy_index * 2 * (size_t)p->L.total;
    fp.pol.blob_stride = (size_t)p->L.total;
    fp.pol.W = p->W, fp.pol.H = p->H, fp.pol.S = p->S, fp.pol.SC = p->SC, fp.pol.npos = p->npos;
    fp.pol.M = kRows, fp.pol.tiles = 1;
    fp.pol.deterministic = deterministic, fp.pol.seed = seed, fp.pol.offset = 0;
    fp.pol.rng_rows_per_seat = p->rng_rows_per_seat, fp.pol.rng_add0 = p->rng_add0, fp.pol.rng_add1 = p->rng_add1;
    fp.pol.d_offset = reinterpret_cast<const unsigned long long*>(d_offset);
    fp.pol.net_mask = 3, fp.pol.pair_ring = ring, fp.pol.stage_stride = p->stage_stride;
    // a round's world tiles (2 c, 2 c + 1 with two in flight) lie in one 128-world slice, so weights change only between rounds
    fp.pol.tile_policy = tile_policy, fp.pol.f_vt_round = slots * (T + 1), fp.pol.f_slots = slots;
    fp.pol.f_seat1_tiles = population ? 0 : envp.N / kRows;
    fp.env = envp;
    fp.T = T, fp.wtiles = wtiles, fp.slots = slots, fp.cross = cross ? 1 : 0;
    fp.obs_slab = obs_slab, fp.actions = actions, fp.logp = logp, fp.values = values, fp.reward = reward, fp.done = done;
    if (mixed) {
        fp.mix_L = mix->L, fp.mix_seed = mix->mix_seed, fp.mix_partner_seed = mix->partner_seed;
        fp.mix_partner_blobs = p->d_blobs + (size_t)mix->partner_policy * 2 * (size_t)p->L.total;
    }
    const int groups = (wtiles + slots - 1) / slots;
    const int ctas = groups < p->sm_count ? groups : p->sm_count;
    const size_t smem = (size_t)fused_smem_layout(p->npos, ring, p->S, p->SC, slots).total;
    fp.pol.trace = d_trace, fp.pol.trace_u0 = trace_u0, fp.pol.trace_n = trace_n;
    {   // 16-byte plane reads pay when the rows are 16-byte aligned (cramped_room, counter_circuit); OCB_FUSED_VEC_LOADER overrides
        const char* e = getenv("OCB_FUSED_VEC_LOADER");
        fp.vec_loader = e != nullptr ? (e[0] != '0') : (p->SC % 16 == 0);
    }
    {   // split mode (the critic's conv stream deferred behind the actor's): needs every grid column of a tile resident, one
        // tile in flight and a critic.  Population self-play takes it too: a change of weights between rounds waits, like
        // every head reload, for the previous tile's head-empty barrier, which counts the deferred critic conv's commit
        const int cols = 192 / (kCellCols * p->H);
        const char* e = getenv("OCB_FUSED_SPLIT");
        const bool want = e != nullptr ? (e[0] != '0') : true;
        fp.col_ring = (want && slots == 1 && !cross && !mixed && cols >= p->W) ? (p->W < kFMaxColRing ? p->W : kFMaxColRing) : 0;
        if (fp.col_ring < p->W) fp.col_ring = 0;
    }
    const cudaStream_t st = (cudaStream_t)stream;
    if (mixed) {  // its own instances, like population: both actors are needed before the env step, so no split mode
        fp.col_ring = kColRing;
        if (slots == 2)
            rollout_fused_kernel<false, false, 2, false, true><<<ctas, kFThreads, smem, st>>>(fp);
        else
            rollout_fused_kernel<false, false, 1, false, true><<<ctas, kFThreads, smem, st>>>(fp);
    } else if (population) {  // its own instances: the self-play and cross-play launches keep the code they had without this mode
        if (fp.col_ring > 0) {
            rollout_fused_kernel<false, true, 1, true><<<ctas, kFThreads, smem, st>>>(fp);
        } else {
            fp.col_ring = kColRing;
            if (slots == 2)
                rollout_fused_kernel<false, false, 2, true><<<ctas, kFThreads, smem, st>>>(fp);
            else
                rollout_fused_kernel<false, false, 1, true><<<ctas, kFThreads, smem, st>>>(fp);
        }
    } else if (fp.col_ring > 0) {
        if (d_trace != nullptr)
            rollout_fused_kernel<true, true, 1><<<ctas, kFThreads, smem, st>>>(fp);
        else
            rollout_fused_kernel<false, true, 1><<<ctas, kFThreads, smem, st>>>(fp);
    } else {
        fp.col_ring = kColRing;
        if (slots == 2) {
            if (d_trace != nullptr)
                rollout_fused_kernel<true, false, 2><<<ctas, kFThreads, smem, st>>>(fp);
            else
                rollout_fused_kernel<false, false, 2><<<ctas, kFThreads, smem, st>>>(fp);
        } else {
            if (d_trace != nullptr)
                rollout_fused_kernel<true, false, 1><<<ctas, kFThreads, smem, st>>>(fp);
            else
                rollout_fused_kernel<false, false, 1><<<ctas, kFThreads, smem, st>>>(fp);
        }
    }
    if (d_counter != nullptr)
        counter_add_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(reinterpret_cast<unsigned long long*>(d_counter), (unsigned long long)T);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return fail(OCB_ERR_CUDA, "fused rollout launch failed: %s", cudaGetErrorString(err));
    p->calls += 1;
    return OCB_OK;
}
