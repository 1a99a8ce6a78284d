// BezKick task-side kernels for B200 (sm_100a): K0 pre-physics, the fused post-physics tile kernel
// (bookkeeping + masked reset + observations + reward/termination; also instantiated as the separate
// observation / reward kernels), explicit-id reset, and the Philox uniform dump.
//
// Layout facts (Isaac Gym AoS, SURVEY App. D): per env, dof_state is 36 contiguous floats, root_states
// 26 contiguous floats (2 actors x 13); rigid_body / net_contact are sparse (10 of 286 resp. 6 of 66
// floats used).  One thread per env; every WARP owns a sub-tile of 32 consecutive envs (its own shared-memory
// slice, mbarrier and bulk copies -- the kernel has no CTA-wide barrier):
//   * the two dense inputs of the sub-tile are contiguous byte ranges -> two cp.async.bulk (TMA 1-D)
//     copies into shared memory, completion on the warp's mbarrier;
//   * the sparse rows are gathered with per-thread sector-aligned vector loads issued BEFORE the
//     barrier wait, so they fly together with the bulk copies;
//   * each thread reads its rows out of shared memory with bank-conflict-free 128-bit loads (row stride
//     36 words), computes everything in registers, then the 54-float observation rows are written
//     back into the SAME shared region (after a warp barrier) and leave as one cp.async.bulk store of
//     32*216 contiguous bytes per warp.
// Kernels are launched with the programmatic-dependent-launch attribute (prologue overlaps the previous kernel's
// drain; griddepcontrol.wait precedes the first global access).
// HBM-bound: 656-680 algorithmic B/env-step, no tensor cores.
#include "bezk_common.cuh"
#include "bezk_internal.h"
#include "bezk_task_math.cuh"
#include <math.h>
#include <stdlib.h>
#include <atomic>
#include <type_traits>

namespace bezk {

#ifndef BEZK_TILE
#define BEZK_TILE 128               // envs (= threads) per CTA
#endif
#ifndef BEZK_TILE_CTAS
#define BEZK_TILE_CTAS 4            // resident one-tile CTAs per SM the register allocation is tuned for: 4 (122 registers, no
                                    // spills, 100 KB left to L1 for the multi-load gathers) beats 5 (96 registers, 28 B of
                                    // spills) by 2-10 % at every size and 6 (80 registers) loses 22 % -- profiles/r01_kernels.md
#endif
// envs per CTA = threads per CTA is a template parameter (TILE).  128 is what ships: 64 was 3 % slower, a persistent 2-stage
// pipelined variant (12 warps/SM) 28 % slower and cross-CTA L2 prefetch 15 % slower -- measured, profiles/r01_kernels.md.
// per-tile shared memory: the observation rows alias the input tiles, so the region is the larger of the two
__host__ __device__ constexpr int smem_in_floats(int tile, int task = BEZK_TASK_KICK) {
    return tile * (DOF_ROW + root_row(task)) > tile * obs_row(task) ? tile * (DOF_ROW + root_row(task)) : tile * obs_row(task);
}
__host__ __device__ constexpr int smem_obs_floats(int tile, int task = BEZK_TASK_KICK) { return tile * obs_row(task); }


// ------------------------------------------------------------------------------------------------
// K0: pre-physics.  Pure streaming elementwise pass over (n,18): 72 B read + 72 B written per env.
// ------------------------------------------------------------------------------------------------
constexpr int K0_THREADS = 288;         // 9 column pairs x 32 rows: a thread keeps ONE column pair -> its constants live in registers
constexpr int K0_ROWS = K0_THREADS / 9;  // rows per block iteration
constexpr int K0_UNROLL = 8;            // independent 8-byte loads in flight per thread

__global__ void __launch_bounds__(K0_THREADS) pre_physics_kernel(const float* __restrict__ actions, float* __restrict__ actions_out,
                                                                 float* __restrict__ targets, const __grid_constant__ BezkTaskCfg cfg,
                                                                 int64_t n, int vec2) {
    const float clip = cfg.clip_actions;
    pdl_launch_dependents();
    pdl_wait();
    if (vec2) {
        const int pair = threadIdx.x % 9, rsub = threadIdx.x / 9;
        const int c0 = 2 * pair;
        const float d0 = cfg.default_dof_pos[c0], d1 = cfg.default_dof_pos[c0 + 1];
        const float l0 = cfg.dof_lower[c0], l1 = cfg.dof_lower[c0 + 1];
        const float h0 = cfg.dof_upper[c0], h1 = cfg.dof_upper[c0 + 1];
        const bool head = (pair == 0);
        const int64_t row0 = (int64_t)blockIdx.x * (K0_ROWS * K0_UNROLL) + rsub;
        float2 in[K0_UNROLL];
#pragma unroll
        for (int u = 0; u < K0_UNROLL; ++u) {
            const int64_t r = row0 + u * K0_ROWS;
            if (r < n) {
                const float2* p = reinterpret_cast<const float2*>(actions) + r * 9 + pair;
                asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(in[u].x), "=f"(in[u].y) : "l"(p));
            }
        }
#pragma unroll
        for (int u = 0; u < K0_UNROLL; ++u) {
            const int64_t r = row0 + u * K0_ROWS;
            if (r >= n) continue;
            float s0, s1;
            const float t0 = k0_target(in[u].x, head, clip, d0, l0, h0, &s0);
            const float t1 = k0_target(in[u].y, head, clip, d1, l1, h1, &s1);
            __stcs(reinterpret_cast<float2*>(targets) + r * 9 + pair, make_float2(t0, t1));
            if (actions_out) __stcs(reinterpret_cast<float2*>(actions_out) + r * 9 + pair, make_float2(s0, s1));
        }
    } else {                                       // pointers not 8-byte aligned: scalar grid-stride path
        const int64_t total = n * 18;
        const int64_t stride = (int64_t)gridDim.x * blockDim.x;
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
            const int col = (int)(i % 18);
            float st;
            targets[i] = k0_target(actions[i], col < 2, clip, cfg.default_dof_pos[col], cfg.dof_lower[col], cfg.dof_upper[col], &st);
            if (actions_out) actions_out[i] = st;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Per-env inputs that do not come through the dense TMA tiles: the IMU-link slice of rigid_body, the foot forces of
// net_contact (sparse AoS gathers) and the small per-env scalars.  Kept in registers; all loads are independent, so a
// caller can issue them long before the values are consumed.
// ------------------------------------------------------------------------------------------------
// the per-step goal draw of the walk / orient reset: counter (2^32-1, 2^32-1, step_lo, step_hi*16 + 15) never collides with
// an env's reset counters (env ids are < 2^63, sub-counter 0..8)
__device__ __forceinline__ Philox4 philox_goal(uint64_t seed, uint64_t step) {
    return philox4x32_10(0xFFFFFFFFu, 0xFFFFFFFFu, (uint32_t)step, ((uint32_t)(step >> 32) << 4) + 15u, (uint32_t)seed,
                         (uint32_t)(seed >> 32));
}

// L2H: the hinted variant (task_tile_l2_kernel) -- the call with the cache policy; otherwise the plain call, so that the unhinted
// kernel is the same code as without the hints (the policy descriptors cost ~9 % at 65 536 envs, where nothing is hinted)
#define L2HINT(f, pol, ...) (L2H ? f(__VA_ARGS__, pol) : f(__VA_ARGS__))

template <bool CLEATS>
struct Gathered {
    // raw load results: NOTHING depends on them until consume(), so issuing gather_env() never stalls the warp
    float raw[10];                       // the 40-byte IMU-link slice in LOAD order (vector path: 8 B, 16 B, 16 B pieces)
    float win[6];                        // window path only: floats 10..15 of the 16-byte aligned window around the slice
    float fl[CLEATS ? 12 : 3], fr[CLEATS ? 12 : 3];
    float goal[2], binit[2], prev[3];
    float gang;                          // orient task: goal angle
    float value;                         // critic value of this step (rollout epilogue only)
    long long reset_prev, progress;
};

// rb: this env's IMU-link slice (10 floats); cf_l / cf_r: its foot (first cleat) force rows.  The caller forms them as a
// warp-uniform 64-bit base plus a 32-bit lane offset.
template <bool OBS, bool BOOKREW, bool CLEATS, int TASK, bool L2H>
__device__ __forceinline__ void gather_env(const TaskArgs& a, const BezkTaskCfg& cfg, int64_t e, bool valid, const float* rb,
                                           float* cf_l, float* cf_r, Gathered<CLEATS>& g) {
    constexpr int NFORCE = CLEATS ? 12 : 3;
#pragma unroll
    for (int k = 0; k < NFORCE; ++k) { g.fl[k] = 0.0f; g.fr[k] = 0.0f; }
    g.goal[0] = g.goal[1] = g.binit[0] = g.binit[1] = 0.0f;
    g.prev[0] = g.prev[1] = g.prev[2] = 0.0f;
    g.gang = 0.0f;
    g.value = 0.0f;
    g.reset_prev = 0; g.progress = 0;
#pragma unroll
    for (int k = 0; k < 10; ++k) g.raw[k] = 0.0f;
#pragma unroll
    for (int k = 0; k < 6; ++k) g.win[k] = 0.0f;
    if (valid) {
        const uint64_t ps = L2H ? policy_evict_first() : 0;     // the simulator's rows: read once per step
        if (a.rb_vec2) {
            // 40 bytes at an 8-byte aligned address: one 8 B + two 16 B loads, order chosen per lane by bit 3
            const char* p = reinterpret_cast<const char*>(rb);
            const bool hi = (reinterpret_cast<uintptr_t>(p) & 8u) != 0;
            // request count matters as much as bytes (profiles/r01_fetch_granularity.md): when the 40-byte span straddles a
            // 64-byte boundary but stays inside one 128-byte line, ONE full-line fill replaces two 64-byte ones
            const uint32_t s128 = (uint32_t)(reinterpret_cast<uintptr_t>(p) & 127u);
            const bool one_line = (a.smart_granule == 2 && s128 + 40u <= 128u) ||
                                  (a.smart_granule && ((s128 & 63u) + 40u > 64u) && (s128 + 40u <= 128u));
            float2 a2; float4 b4, c4;
            if (one_line) {
                a2 = L2HINT(ldg128B_nc_v2, ps, p + (hi ? 0 : 32)); b4 = L2HINT(ldg128B_nc_v4, ps, p + (hi ? 8 : 0));
                c4 = L2HINT(ldg128B_nc_v4, ps, p + (hi ? 24 : 16));
            } else {
                a2 = L2HINT(ldg64B_nc_v2, ps, p + (hi ? 0 : 32)); b4 = L2HINT(ldg64B_nc_v4, ps, p + (hi ? 8 : 0));
                c4 = L2HINT(ldg64B_nc_v4, ps, p + (hi ? 24 : 16));
            }
            g.raw[0] = a2.x; g.raw[1] = a2.y; g.raw[2] = b4.x; g.raw[3] = b4.y; g.raw[4] = b4.z; g.raw[5] = b4.w;
            g.raw[6] = c4.x; g.raw[7] = c4.y; g.raw[8] = c4.z; g.raw[9] = c4.w;
        } else if (TASK != BEZK_TASK_KICK && a.rb_win) {       // BezKick's 22-body rows are 8-byte aligned: the branch is compiled out
            // slice only 4-byte aligned (21-body walk / orient rows): 3 (4 when the slice starts at +12) aligned 16-byte loads
            // of the window around it instead of 10 scalar loads; consume() rotates by the start offset
            const char* p = reinterpret_cast<const char*>(rb);
            const uint32_t o = (uint32_t)(reinterpret_cast<uintptr_t>(p) & 15u);
            const float4 c0 = L2HINT(ldg64B_nc_v4, ps, p - o), c1 = L2HINT(ldg64B_nc_v4, ps, p - o + 16);
            const float4 c2 = L2HINT(ldg64B_nc_v4, ps, p - o + 32);
            float4 c3 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (o == 12u) c3 = L2HINT(ldg64B_nc_v4, ps, p - o + 48);
            g.raw[0] = c0.x; g.raw[1] = c0.y; g.raw[2] = c0.z; g.raw[3] = c0.w; g.raw[4] = c1.x; g.raw[5] = c1.y; g.raw[6] = c1.z;
            g.raw[7] = c1.w; g.raw[8] = c2.x; g.raw[9] = c2.y;
            g.win[0] = c2.z; g.win[1] = c2.w; g.win[2] = c3.x; g.win[3] = c3.y; g.win[4] = c3.z; g.win[5] = c3.w;
        } else {
#pragma unroll
            for (int k = 0; k < 10; ++k) g.raw[k] = L2HINT(ldg64B_nc, ps, rb + k);
        }
        if (OBS) {
            if (!CLEATS && a.cf_vec2) {
                // same idea for the feet: a full-line fill when both feet (or a foot straddling a 64-byte boundary) sit
                // inside one 128-byte line, 64-byte granules otherwise
                const uint32_t sl = (uint32_t)(reinterpret_cast<uintptr_t>(cf_l) & 127u);
                const uint32_t sr = (uint32_t)(reinterpret_cast<uintptr_t>(cf_r) & 127u);
                const bool same_line = ((reinterpret_cast<uintptr_t>(cf_l) ^ (reinterpret_cast<uintptr_t>(cf_r) + 11u)) & ~(uintptr_t)127u) == 0;
                const bool l_line = a.smart_granule == 2 || (a.smart_granule && (same_line || (((sl & 63u) + 12u > 64u) && (sl + 12u <= 128u))));
                const bool r_line = a.smart_granule == 2 || (a.smart_granule && !same_line && (((sr & 63u) + 12u > 64u) && (sr + 12u <= 128u)));
                const float2 l2 = l_line ? L2HINT(ldg128B_v2, ps, cf_l) : L2HINT(ldg64B_v2, ps, cf_l);
                const float2 r2 = r_line ? L2HINT(ldg128B_v2, ps, cf_r) : L2HINT(ldg64B_v2, ps, cf_r);
                g.fl[0] = l2.x; g.fl[1] = l2.y; g.fl[2] = L2HINT(ldg64B, ps, cf_l + 2);
                g.fr[0] = r2.x; g.fr[1] = r2.y; g.fr[2] = L2HINT(ldg64B, ps, cf_r + 2);
            } else {
#pragma unroll
                for (int k = 0; k < NFORCE; ++k) { g.fl[k] = L2HINT(ldg64B, ps, cf_l + k); g.fr[k] = L2HINT(ldg64B, ps, cf_r + k); }
            }
        }
        // the carried per-env state: the same addresses every step
        const uint64_t pk = L2H ? policy_evict_last() : 0;
        if (OBS && a.prev_lin_vel) {
#pragma unroll
            for (int k = 0; k < 3; ++k) g.prev[k] = L2HINT(ld_f32, pk, a.prev_lin_vel + e * 3 + k);
        }
        if (TASK == BEZK_TASK_KICK) {
            const float2 g2 = L2HINT(ld_nc_v2, pk, reinterpret_cast<const float2*>(a.goal) + e);
            const float2 b2 = L2HINT(ld_nc_v2, pk, reinterpret_cast<const float2*>(a.ball_init) + e);
            g.goal[0] = g2.x; g.goal[1] = g2.y; g.binit[0] = b2.x; g.binit[1] = b2.y;
        } else if (TASK == BEZK_TASK_WALK) {      // goal is rewritten by this kernel on reset: coherent load
            const float2 g2 = L2HINT(ldg128B_v2, pk, reinterpret_cast<const float2*>(a.goal) + e);
            g.goal[0] = g2.x; g.goal[1] = g2.y;
        } else {
            g.gang = L2HINT(ld_f32, pk, a.goal_angle + e);
        }
        if (BOOKREW) {
            g.reset_prev = L2HINT(ld_i64, pk, a.reset_in + e);
            g.progress = L2HINT(ld_i64, pk, a.progress_in + e);
            if (a.values) g.value = ld_f32(a.values + e * a.values_stride);
        }
    }
}

// First use of a gathered set: pin the raw registers behind an (empty) volatile asm so that the compiler cannot
// hoist the unpacking selects up to the loads (which would stall the warp at issue time), then unpack.
template <bool CLEATS, int TASK>
__device__ __forceinline__ void consume(const TaskArgs& a, const float* rb, Gathered<CLEATS>& g, float (&imu)[10]) {
    asm volatile("" : "+f"(g.raw[0]), "+f"(g.raw[1]), "+f"(g.raw[2]), "+f"(g.raw[3]), "+f"(g.raw[4]), "+f"(g.raw[5]),
                      "+f"(g.raw[6]), "+f"(g.raw[7]), "+f"(g.raw[8]), "+f"(g.raw[9]));
    asm volatile("" : "+l"(g.reset_prev), "+l"(g.progress));
    // vector path, slice NOT 16-byte aligned (hi): pieces were loaded in memory order (8,16,16) -> raw is already in order;
    // 16-byte aligned: pieces were loaded as (tail 8 B, first 16 B, second 16 B) -> rotate
    if (TASK != BEZK_TASK_KICK && !a.rb_vec2 && a.rb_win) {
        asm volatile("" : "+f"(g.win[0]), "+f"(g.win[1]), "+f"(g.win[2]), "+f"(g.win[3]), "+f"(g.win[4]), "+f"(g.win[5]));
        const uint32_t sh = (uint32_t)(reinterpret_cast<uintptr_t>(rb) & 15u) >> 2;     // slice starts at window float 0..3
#pragma unroll
        for (int k = 0; k < 10; ++k) {
            // window float k + sh, statically indexed: floats 0..9 live in raw, 10..15 in win
            const float w0 = g.raw[k];
            const float w1 = (k + 1 < 10) ? g.raw[k + 1] : g.win[k + 1 - 10];
            const float w2 = (k + 2 < 10) ? g.raw[k + 2] : g.win[k + 2 - 10];
            const float w3 = (k + 3 < 10) ? g.raw[k + 3] : g.win[k + 3 - 10];
            imu[k] = sh == 0 ? w0 : (sh == 1 ? w1 : (sh == 2 ? w2 : w3));
        }
        return;
    }
    const bool rot = a.rb_vec2 && ((reinterpret_cast<uintptr_t>(rb) & 8u) == 0);
#pragma unroll
    for (int k = 0; k < 10; ++k) imu[k] = rot ? g.raw[(k + 2) % 10] : g.raw[k];
}

// ------------------------------------------------------------------------------------------------
// The fused tile kernel.  PARTS: 1 bookkeeping+masked reset, 2 observations, 4 reward/termination.
// ------------------------------------------------------------------------------------------------
// rl_games' episode bookkeeping of one env in the reward epilogue (episode_step), its carried values stored like the bookkeeping
template <bool L2H>
__device__ __forceinline__ void episode_epilogue(const EpArgs& ep, int64_t e, float rew, int64_t reset, float ret, float len, bool& done,
                                                 float& r, float& l) {
    float ret_out, len_out;
    episode_step(ret, len, rew, reset, r, l, ret_out, len_out);
    const uint64_t pk = L2H ? policy_evict_last() : 0;
    L2HINT(st_f32, pk, ep.ret + e, ret_out);
    L2HINT(st_f32, pk, ep.len + e, len_out);
    done = reset != 0;
}

// the game term returns of one env in the reward epilogue: episode_step's recurrence on each term's accumulator.  acc holds the
// carried values on entry and r_k = acc_k + term_k on return; the carried values are stored as multiplies by (1 - done)
template <bool L2H, int K>
__device__ __forceinline__ void game_terms_epilogue(const GameTermArgs& ga, int64_t n, int64_t e, int64_t reset, const float (&tm)[K],
                                                    float (&acc)[K]) {
    const float not_done = 1.0f - (reset != 0 ? 1.0f : 0.0f);
    const uint64_t pk = L2H ? policy_evict_last() : 0;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        acc[k] = acc[k] + tm[k];
        L2HINT(st_f32, pk, ga.acc + k * n + e, acc[k] * not_done);
    }
}

// the pack element of type T
template <typename T, typename P0, typename... P>
__device__ __forceinline__ const T& arg_of(const P0& p0, const P&... p) {
    if constexpr (std::is_same<T, P0>::value) return p0;
    else return arg_of<T>(p...);
}
template <typename T, typename... P>
constexpr bool has_arg = (std::is_same<T, P>::value || ...);

// Ep: empty, or one EpArgs -- then EP is on and the episode accumulators ride along (task_tile_ep_kernel / task_tile_ep_l2_kernel;
// whole step only) -- or EpArgs and NormArgs: the eval-mode observation normaliser too (task_tile_obsnorm_kernel /
// task_tile_obsnorm_l2_kernel).  Either EP pack may end in OutArgs: the per-warp episode outcome counts too
// (task_tile_outcome_kernel / task_tile_obsnorm_outcome_kernel and their _l2 forms).  EpArgs (and OutArgs) may be followed by
// TermArgs: the per-warp reward term sums too (task_tile_terms_kernel / task_tile_outcome_terms_kernel and their _l2 forms).  Any of
// these packs may end in GameTermArgs: the carried game term returns too (task_tile_game_kernel / task_tile_game_l2_kernel).  A
// parameter pack rather than always-present arguments: the kernels without accumulators make exactly the call they made before the
// accumulators existed (an unused EpArgs argument alone changes their register allocation).
template <int PARTS, bool CLEATS, int TILE, int TASK, bool L2H, typename... Ep>
__device__ __forceinline__ void task_tile(const TaskArgs& a, const BezkTaskCfg& cfg, const Ep&... eps) {
    constexpr bool EP = sizeof...(Ep) >= 1;
    constexpr bool NORM = has_arg<NormArgs, Ep...>;
    constexpr bool OUT = has_arg<OutArgs, Ep...>;
    constexpr bool TERMS = has_arg<TermArgs, Ep...>;
    constexpr bool GAME = has_arg<GameTermArgs, Ep...>;
    constexpr int K_TERMS = reward_terms(TASK);
    static_assert(!EP || PARTS == 7, "the episode accumulators ride in the whole step");
    constexpr int ROOT_ROW = root_row(TASK);
    constexpr int OBS_ROW = obs_row(TASK);
    constexpr bool BOOK = (PARTS & BEZK_PART_BOOKKEEP) != 0;
    constexpr bool OBS = (PARTS & BEZK_PART_OBS) != 0;
    constexpr bool REW = (PARTS & BEZK_PART_REWARD) != 0;
    constexpr int NFORCE = CLEATS ? 12 : 3;

    // Every WARP owns a sub-tile of 32 consecutive envs: its own slice of shared memory, its own mbarrier, its own bulk
    // copies and bulk store.  Nothing in the kernel is CTA-wide (no __syncthreads): a warp whose data has arrived never
    // waits for a sibling whose gathers are still in flight.
    constexpr int WT = 32;
    constexpr int WARPS = TILE / WT;
    extern __shared__ __align__(128) float smem[];
    __shared__ __align__(8) uint64_t s_bars[WARPS];

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    float* s_dof = smem + warp * smem_in_floats(WT, TASK);                         // [32][36]
    float* s_root = s_dof + WT * DOF_ROW;                                          // [32][26 | 13]
    float* s_obs = s_dof;                                                          // [32][54 | 52], aliases this warp's input tiles
    float* s_obs_clip = smem + smem_in_floats(TILE, TASK) + warp * smem_obs_floats(WT, TASK);   // only when a.obs_clipped
    uint64_t* s_bar = &s_bars[warp];

    const int64_t e0 = (int64_t)blockIdx.x * TILE + warp * WT;                     // first env of this warp's sub-tile
    const int64_t left = a.n - e0;
    const int nv = (int)(left < 0 ? 0 : (left < (int64_t)WT ? left : (int64_t)WT));
    const bool full = (nv == WT) && a.use_tma;
    const int64_t e = e0 + lane;
    const bool valid = lane < nv;

    pdl_launch_dependents();               // the next kernel on the stream may be scheduled as our CTAs retire
    if (full && lane == 0) {
        mbar_init(s_bar, 1);
        fence_mbar_init();
    }
    pdl_wait();                            // nothing above touches global memory

    // ---- 1. sparse gathers first: they are the slow requests (one 64-byte granule each), the dense tiles follow ----
    // per-env row pointers: warp-uniform 64-bit base + 32-bit lane offset
    const float* rb = a.rigid_body + (e0 * a.rb_stride + a.rb_off) + lane * a.rb_stride;
    float* cf_env = a.net_contact ? a.net_contact + e0 * a.cf_stride + lane * a.cf_stride : nullptr;
    float* cf_l = cf_env ? cf_env + a.cf_l_off : nullptr;
    float* cf_r = cf_env ? cf_env + a.cf_r_off : nullptr;
    Gathered<CLEATS> g;
    gather_env<OBS, (BOOK || REW), CLEATS, TASK, L2H>(a, cfg, e, valid, rb, cf_l, cf_r, g);
    float ep_ret = 0.0f, ep_len = 0.0f;    // carried like the bookkeeping: the same addresses every step
    if constexpr (EP) {
        const EpArgs& ep = arg_of<EpArgs>(eps...);
        if (valid) {
            const uint64_t pk = L2H ? policy_evict_last() : 0;
            ep_ret = L2HINT(ld_f32, pk, ep.ret + e);
            ep_len = L2HINT(ld_f32, pk, ep.len + e);
        }
    }
    float gacc[K_TERMS] = {};              // GAME: the carried game term returns, then this step's r_k (0 in lanes past the last env)
    if constexpr (GAME) {
        const GameTermArgs& ga = arg_of<GameTermArgs>(eps...);
        if (valid) {
            const uint64_t pk = L2H ? policy_evict_last() : 0;
#pragma unroll
            for (int k = 0; k < K_TERMS; ++k) gacc[k] = L2HINT(ld_f32, pk, ga.acc + k * a.n + e);
        }
    }
    bool ep_done = false;                  // this env's episode ended in this step, with return ep_r and length ep_l
    float ep_r = 0.0f, ep_l = 0.0f;
    int ep_oc = OUTCOME_NONE;              // OUT: the rule that ended it (the outcome class), from the reward call whose rew is stored
    float tm[K_TERMS] = {};                // TERMS / GAME: this env's reward terms, from the same call (0 in lanes past the last env)
    constexpr bool TM = TERMS || GAME;


    // ---- 2. dense tiles: TMA bulk copies (full sub-tiles) or cooperative coalesced loads (tail) ----
    if (full) {
        if (lane == 0) {
            mbar_arrive_expect_tx(s_bar, WT * (DOF_ROW + ROOT_ROW) * 4);
            const uint64_t ps = L2H ? policy_evict_first() : 0;
            L2HINT(bulk_g2s, ps, s_dof, a.dof_state + e0 * DOF_ROW, WT * DOF_ROW * 4, s_bar);
            L2HINT(bulk_g2s, ps, s_root, a.root_states + e0 * ROOT_ROW, WT * ROOT_ROW * 4, s_bar);
        }
    } else {
        for (int i = lane; i < nv * DOF_ROW; i += WT) s_dof[i] = a.dof_state[e0 * DOF_ROW + i];
        for (int i = lane; i < nv * ROOT_ROW; i += WT) s_root[i] = a.root_states[e0 * ROOT_ROW + i];
    }

    float imu_in[10];
    consume<CLEATS, TASK>(a, rb, g, imu_in);
    float (&fl)[NFORCE] = g.fl;
    float (&fr)[NFORCE] = g.fr;
    float (&goal)[2] = g.goal;
    float (&binit)[2] = g.binit;
    float (&prev)[3] = g.prev;
    const int64_t reset_prev = (int64_t)g.reset_prev;
    int64_t progress = (int64_t)g.progress;
    const float q[4] = {imu_in[0], imu_in[1], imu_in[2], imu_in[3]};
    const float v[3] = {imu_in[4], imu_in[5], imu_in[6]};
    const float w[3] = {imu_in[7], imu_in[8], imu_in[9]};

    // ---- 3. wait for the dense tiles ----
    __syncwarp();                          // mbarrier init / cooperative stores visible to the whole warp
    if (full) mbar_wait(s_bar, 0);

    // ---- 4. bookkeeping + masked reset (vec_task.py:331-332, kick_env.py:429-435, 779-850) ----
    // The reset of an env is done by its WARP: lanes 0..8 each run one Philox4x32 block (4 of the 36 draws),
    // patch the env's row in shared memory and write it back to dof_state as 9 float4 stores; lanes 0..25 copy
    // the initial root-state row.  No divergent 36-draw loop in the per-thread path.
    int64_t timeout = 0, reset_cur = reset_prev;
    if (BOOK) {
        unsigned pending = __ballot_sync(0xffffffffu, valid && reset_prev != 0);
        while (pending) {
            const int r = __ffs(pending) - 1;
            pending &= pending - 1;
            const int64_t env = e0 + r;
            if (lane < 9) {
                float u4[4];
                if (a.uniforms) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) u4[k] = a.uniforms[env * 36 + 4 * lane + k];
                } else {
                    const int64_t genv = a.env_base + env;         // Philox is keyed by the GLOBAL env id
                    const Philox4 x = philox4x32_10((uint32_t)genv, (uint32_t)((uint64_t)genv >> 32), (uint32_t)a.step,
                                                    ((uint32_t)(a.step >> 32) << 4) + (uint32_t)lane, (uint32_t)a.seed,
                                                    (uint32_t)(a.seed >> 32));
                    u4[0] = u01(x.x); u4[1] = u01(x.y); u4[2] = u01(x.z); u4[3] = u01(x.w);
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int d = 4 * lane + k;              // draw index: 0..17 positions, 18..35 velocities
                    if (d < 18) {
                        const float off = cfg.reset_pos_span * u4[k] + cfg.reset_pos_lo;
                        s_dof[r * DOF_ROW + 2 * d] = tensor_clamp(cfg.default_dof_pos[d] + off, cfg.dof_lower[d], cfg.dof_upper[d]);
                    } else {
                        s_dof[r * DOF_ROW + 2 * (d - 18) + 1] = cfg.reset_vel_span * u4[k] + cfg.reset_vel_lo;
                    }
                }
            }
            __syncwarp();
            if (lane < 9) {
                if (a.use_tma) {
                    reinterpret_cast<float4*>(a.dof_state_wb + env * DOF_ROW)[lane] = reinterpret_cast<const float4*>(s_dof + r * DOF_ROW)[lane];
                } else {
#pragma unroll
                    for (int k = 0; k < 4; ++k) a.dof_state_wb[env * DOF_ROW + 4 * lane + k] = s_dof[r * DOF_ROW + 4 * lane + k];
                }
            }
            if ((cfg.flags & BEZK_F_RESET_ROOT_STATES) && lane < ROOT_ROW) {
                const float t = a.initial_root[env * ROOT_ROW + lane];
                s_root[r * ROOT_ROW + lane] = t;
                a.root_states_wb[env * ROOT_ROW + lane] = t;
            }
            __syncwarp();
        }
        if (valid) {
            timeout = (progress >= (int64_t)cfg.max_episode_length - 1) ? 1 : 0;
            progress += 1;
            if (a.randomize_buf) a.randomize_buf[e] += 1;
            if (reset_prev != 0) {
                progress = 0; reset_cur = 0;
                if (TASK != BEZK_TASK_KICK) {
                    // goal randomisation (walk_env.py:566-574): ONE draw per reset batch, i.e. per step
                    float ux, uy;
                    if (a.goal_uniforms) { ux = a.goal_uniforms[0]; uy = a.goal_uniforms[1]; }
                    else { const Philox4 x = philox_goal(a.seed, a.step); ux = u01(x.x); uy = u01(x.y); }
                    goal[0] = 4.0f * ux + -2.0f;                 // torch_rand_float(-2, 2): (hi - lo) * u + lo
                    goal[1] = 4.0f * uy + -2.0f;
                    L2HINT(st_v2, L2H ? policy_evict_last() : 0, reinterpret_cast<float2*>(a.goal) + e, make_float2(goal[0], goal[1]));
                }
            }
            L2HINT(st_i64, L2H ? policy_evict_last() : 0, a.timeout_buf + e, timeout);
            if (!REW) {
                L2HINT(st_i64, L2H ? policy_evict_last() : 0, a.progress_out + e, progress);
                L2HINT(st_i64, L2H ? policy_evict_last() : 0, a.reset_out + e, reset_cur);
            }
        }
    }

    // ---- 5. this env's rows: shared -> registers (conflict-free 128-bit reads, row stride 36 words) ----
    float row[36];
    float bez[3] = {0.f, 0.f, 0.f}, ball_xy[2] = {0.f, 0.f}, ball_vxy[2] = {0.f, 0.f};
    if (valid) {
        const float4* r4 = reinterpret_cast<const float4*>(s_dof + lane * DOF_ROW);
#pragma unroll
        for (int k = 0; k < 9; ++k) {
            const float4 t = r4[k];
            row[4 * k] = t.x; row[4 * k + 1] = t.y; row[4 * k + 2] = t.z; row[4 * k + 3] = t.w;
        }
        const float* rr = s_root + lane * ROOT_ROW;
        bez[0] = rr[0]; bez[1] = rr[1]; bez[2] = rr[2];
        if (TASK == BEZK_TASK_KICK) {
            ball_xy[0] = rr[13]; ball_xy[1] = rr[14];
            ball_vxy[0] = rr[20]; ball_vxy[1] = rr[21];
        }
    }

    // ---- 5b. the dof half of the observation row leaves the registers NOW: pos_sq (the only other use of the 36 dof values) is
    // formed first, then -- once every lane has read its rows -- the de-interleaved [pos 18, vel 18] columns are written into the
    // aliased output tile, so the long dependent chains below (IMU, heading, reward) run without 36 live registers ----
    float pos_sq = 0.0f;
    if (REW && valid) {
#pragma unroll
        for (int j = 0; j < 18; ++j) {
            const float d = cfg.default_dof_pos[j] - row[2 * j];
            pos_sq += d * d;
        }
    }
    if (OBS) {
        __syncwarp();                      // every lane has finished reading its s_dof / s_root rows
        if (valid) {
            float2* o2 = reinterpret_cast<float2*>(s_obs + lane * OBS_ROW);
#pragma unroll
            for (int k = 0; k < 9; ++k) {  // dof_pos 0:18, dof_vel 18:36 (de-interleave of [pos, vel] pairs)
                o2[k] = make_float2(row[4 * k], row[4 * k + 2]);
                o2[9 + k] = make_float2(row[4 * k + 1], row[4 * k + 3]);
            }
        }
    }

    // ---- 6. observations (kick_env.py:749-777) ----
    float imu6[6], orn2[2], feet[8];
    if (OBS && valid) {
        float pv[3];
        if (a.prev_lin_vel) { pv[0] = prev[0]; pv[1] = prev[1]; pv[2] = prev[2]; }
        else { pv[0] = v[0]; pv[1] = v[1]; pv[2] = v[2]; }                  // aliasing, kick_env.py:930
        // the per-env math runs on the branch-free exact operators (Mth<true>); an env with an operand outside their
        // validity range is recomputed once with the plain operators -- same bits either way
        Mth<true> mo;
        imu_term(q, v, w, pv, cfg, imu6, mo);
        if (a.prev_lin_vel) {
#pragma unroll
            for (int k = 0; k < 3; ++k) L2HINT(st_f32, L2H ? policy_evict_last() : 0, a.prev_lin_vel + e * 3 + k, v[k]);
        }
        if (TASK == BEZK_TASK_ORIENT) {                                    // compute_off_angle, orient_env.py:720-733
            const float d = angle_to_goal(q, g.gang);
            sincosf(d, &orn2[1], &orn2[0]);
        } else {
            off_orn_term(bez[0], bez[1], q, goal[0], goal[1], orn2, mo);
        }
        if (mo.bad()) {
            Mth<false> mp;
            imu_term(q, v, w, pv, cfg, imu6, mp);
            if (TASK != BEZK_TASK_ORIENT) off_orn_term(bez[0], bez[1], q, goal[0], goal[1], orn2, mp);
        }
        if (CLEATS) {                                                      // kick_env.py:1053-1061
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int b = CLEATS ? 3 * k : 0;
                const float nl = sqrtf((fl[b] * fl[b] + fl[b + 1] * fl[b + 1]) + fl[b + 2] * fl[b + 2]);
                const float nr = sqrtf((fr[b] * fr[b] + fr[b + 1] * fr[b + 1]) + fr[b + 2] * fr[b + 2]);
                feet[k] = (nl > 1.0f) ? 1.0f : -1.0f;
                feet[4 + k] = (nr > 1.0f) ? 1.0f : -1.0f;
            }
        } else {
            float l3[3] = {fl[0], fl[1], fl[2]}, r3[3] = {fr[0], fr[1], fr[2]};
            float lb[4], rbits[4];
            foot_bits(l3, lb);
            foot_bits(r3, rbits);
#pragma unroll
            for (int k = 0; k < 4; ++k) { feet[k] = lb[k]; feet[4 + k] = rbits[k]; }
            if (cfg.flags & BEZK_F_WRITE_CONTACT_FILTER) {                 // in-place filter, :987-990
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    if (__float_as_uint(l3[k]) != __float_as_uint(fl[k])) cf_l[k] = l3[k];
                    if (__float_as_uint(r3[k]) != __float_as_uint(fr[k])) cf_r[k] = r3[k];
                }
            }
        }
    }

    // ---- 7. remaining observation columns -> shared (aliasing the input tiles) -> one bulk store ----
    if (OBS) {
        if (valid) {
            float2* o2 = reinterpret_cast<float2*>(s_obs + lane * OBS_ROW);
            o2[18] = make_float2(imu6[0], imu6[1]); o2[19] = make_float2(imu6[2], imu6[3]); o2[20] = make_float2(imu6[4], imu6[5]);
            o2[21] = make_float2(orn2[0], orn2[1]);
            o2[22] = make_float2(feet[0], feet[1]); o2[23] = make_float2(feet[2], feet[3]);
            o2[24] = make_float2(feet[4], feet[5]); o2[25] = make_float2(feet[6], feet[7]);
            if (TASK == BEZK_TASK_KICK) o2[26] = make_float2(binit[0], binit[1]);
            if (a.obs_clipped) {           // vec_task.py:343 clamp(obs_buf, -clip_obs, clip_obs)
                float2* c2 = reinterpret_cast<float2*>(s_obs_clip + lane * OBS_ROW);
                const float lim = cfg.clip_obs;
#pragma unroll
                for (int k = 0; k < OBS_ROW / 2; ++k) {
                    const float2 t = o2[k];
                    c2[k] = make_float2(clamp_nan(t.x, -lim, lim), clamp_nan(t.y, -lim, lim));
                }
            }
        }
        if (full) {
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
                const uint64_t po = L2H ? policy_keep(!(cfg.flags & BEZK_F_OBS_STREAMED)) : 0;
                L2HINT(bulk_s2g, po, a.obs + e0 * OBS_ROW, s_obs, WT * OBS_ROW * 4);
                if (a.obs_clipped) L2HINT(bulk_s2g, po, a.obs_clipped + e0 * OBS_ROW, s_obs_clip, WT * OBS_ROW * 4);
                bulk_commit();
            }
        } else {
            __syncwarp();
            for (int i = lane; i < nv * OBS_ROW; i += WT) a.obs[e0 * OBS_ROW + i] = s_obs[i];
            if (a.obs_clipped)
                for (int i = lane; i < nv * OBS_ROW; i += WT) a.obs_clipped[e0 * OBS_ROW + i] = s_obs_clip[i];
        }
    }

    // ---- 8. reward / termination (overlaps the bulk store) ----
    if (REW && valid) {
        float rew;
        int64_t reset;
        if constexpr (TASK == BEZK_TASK_KICK) {
            RewardIn s;
            s.bez[0] = bez[0]; s.bez[1] = bez[1]; s.bez[2] = bez[2];
            s.ball_xy[0] = ball_xy[0]; s.ball_xy[1] = ball_xy[1];
            s.ball_vxy[0] = ball_vxy[0]; s.ball_vxy[1] = ball_vxy[1];
            s.goal[0] = goal[0]; s.goal[1] = goal[1];
            s.ball_init[0] = binit[0]; s.ball_init[1] = binit[1];
#pragma unroll
            for (int k = 0; k < 3; ++k) { s.v[k] = v[k]; s.w[k] = w[k]; }
            s.pos_sq = pos_sq;
            Mth<true> mr;
            reward_term<true, OUT, TM>(s, cfg, progress, reset_cur, &rew, &reset, mr, &ep_oc, tm);
            if (mr.bad()) {
                Mth<false> mp;
                reward_term<false, OUT, TM>(s, cfg, progress, reset_cur, &rew, &reset, mp, &ep_oc, tm);
            }
        } else {
            Mth<true> mr;
            if (TASK == BEZK_TASK_WALK)
                reward_walk<true, OUT, TM>(bez, q, v, w, pos_sq, goal, cfg, progress, reset_cur, &rew, &reset, mr, &ep_oc, tm);
            else reward_orient<true, OUT, TM>(bez, q, v, w, pos_sq, g.gang, cfg, progress, reset_cur, &rew, &reset, mr, &ep_oc, tm);
            if (mr.bad()) {
                Mth<false> mp;
                if (TASK == BEZK_TASK_WALK)
                    reward_walk<false, OUT, TM>(bez, q, v, w, pos_sq, goal, cfg, progress, reset_cur, &rew, &reset, mp, &ep_oc, tm);
                else reward_orient<false, OUT, TM>(bez, q, v, w, pos_sq, g.gang, cfg, progress, reset_cur, &rew, &reset, mp, &ep_oc, tm);
            }
        }
        L2HINT(st_f32, L2H ? policy_evict_last() : 0, a.rew + e, rew);
        L2HINT(st_i64, L2H ? policy_evict_last() : 0, a.reset_out + e, reset);
        if (BOOK) { L2HINT(st_i64, L2H ? policy_evict_last() : 0, a.progress_out + e, progress); rollout_epilogue(a, e, rew, reset, timeout, g.value); }
        if constexpr (EP) episode_epilogue<L2H>(arg_of<EpArgs>(eps...), e, rew, reset, ep_ret, ep_len, ep_done, ep_r, ep_l);
        if constexpr (GAME) game_terms_epilogue<L2H>(arg_of<GameTermArgs>(eps...), a.n, e, reset, tm, gacc);
    }

    // ---- 9. this warp's slot of the per-step episode statistics: [count of done envs, sum of their returns, sum of their
    // lengths] at (k, env / 32).  Fixed-order shuffle tree, one store per value, every step (zeros included): nothing needs
    // zeroing, no atomics, and the sums are the same bits from run to run ----
    if constexpr (EP) if (nv > 0) {
        const EpArgs& ep = arg_of<EpArgs>(eps...);
        const unsigned done_mask = __ballot_sync(0xffffffffu, ep_done);
        double sr = ep_done ? (double)ep_r : 0.0, sl = ep_done ? (double)ep_l : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            sr += __shfl_down_sync(0xffffffffu, sr, o);
            sl += __shfl_down_sync(0xffffffffu, sl, o);
        }
        if (lane == 0) {
            const int64_t slot = e0 / WT;
            ep.partials[slot] = (double)__popc(done_mask);
            ep.partials[ep.w + slot] = sr;
            ep.partials[2 * ep.w + slot] = sl;
        }
        if constexpr (OUT) {
            // ... and the count of its done envs per outcome class at (k, env / 32): one ballot per class, lane k stores class k.
            // In the whole step an env is done exactly when a rule fired (reset_cur is 0 on entry), so the K counts sum to the
            // done count above
            const OutArgs& oa = arg_of<OutArgs>(eps...);
            constexpr int K = outcome_classes(TASK);
            unsigned mine = 0;
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const unsigned m = __ballot_sync(0xffffffffu, ep_oc == k);
                if (lane == k) mine = m;
            }
            if (lane < K) oa.partials[lane * oa.w + e0 / WT] = __popc(mine);
        }
        if constexpr (TERMS) {
            // ... and the fp64 sum of each reward term over its envs at (k, env / 32), with the same fixed-order tree
            const TermArgs& ta = arg_of<TermArgs>(eps...);
#pragma unroll
            for (int k = 0; k < reward_terms(TASK); ++k) {
                double s = (double)tm[k];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
                if (lane == 0) ta.partials[k * ta.w + e0 / WT] = s;
            }
        }
        if constexpr (GAME) {
            // ... and the fp64 sum of each term's episode return over its done envs at (k, env / 32), with the same tree
            const GameTermArgs& ga = arg_of<GameTermArgs>(eps...);
#pragma unroll
            for (int k = 0; k < K_TERMS; ++k) {
                double s = ep_done ? (double)gacc[k] : 0.0;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
                if (lane == 0) ga.partials[k * ga.w + e0 / WT] = s;
            }
        }
    }

    if constexpr (NORM) {
        // ---- 10. rl_games RunningMeanStd.forward in eval mode on the row step() returns (the clipped one when a.obs_clipped),
        // with rms_normalize_kernel's arithmetic: mean.float(), sqrtf(var.float() + eps), IEEE division (Mth fast sequence,
        // plain operator for a chunk with an operand outside its range), clamp to +-5 with NaN propagating.  Lane j holds the
        // statistics of columns j and 32 + j, read from the device every launch.  The tile is normalised in place once the
        // stores above have read it, then leaves as one more bulk store (normal L2 priority: not part of the carried set) ----
        const NormArgs& nm = arg_of<NormArgs>(eps...);
        if (nv == 0) return;                             // warp-uniform: a warp past the last env
        const float m_lo = (float)nm.mean[lane], d_lo = sqrtf((float)nm.var[lane] + nm.eps);
        float m_hi = 0.0f, d_hi = 1.0f;
        if (32 + lane < OBS_ROW) { m_hi = (float)nm.mean[32 + lane]; d_hi = sqrtf((float)nm.var[32 + lane] + nm.eps); }
        if (full && lane == 0) bulk_wait_read0();       // the obs (and clipped) stores have read the tile
        __syncwarp();
        float* x = a.obs_clipped ? s_obs_clip : s_obs;
        float2* r2 = reinterpret_cast<float2*>(x + lane * OBS_ROW);
        // every lane runs the loop (the statistics are shuffled across the warp); a tail warp's lanes >= nv work on rows that
        // are never stored
        constexpr int NF2 = OBS_ROW / 2, CH = 9;         // float2 per row, float2 per chunk
#pragma unroll
        for (int k0 = 0; k0 < NF2; k0 += CH) {
            float in[2 * CH], mean[2 * CH], den[2 * CH], out[2 * CH];
            Mth<true> mq;
#pragma unroll
            for (int k = 0; k < CH; ++k) {
                if (k0 + k >= NF2) break;
                const float2 t = r2[k0 + k];
                in[2 * k] = t.x; in[2 * k + 1] = t.y;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int c = 2 * (k0 + k) + h;
                    mean[2 * k + h] = __shfl_sync(0xffffffffu, c < 32 ? m_lo : m_hi, c & 31);
                    den[2 * k + h] = __shfl_sync(0xffffffffu, c < 32 ? d_lo : d_hi, c & 31);
                    out[2 * k + h] = clamp_nan(mq.div(in[2 * k + h] - mean[2 * k + h], den[2 * k + h]), -5.0f, 5.0f);
                }
            }
            if (mq.bad()) {
#pragma unroll
                for (int j = 0; j < 2 * CH; ++j)
                    if (2 * k0 + j < OBS_ROW) out[j] = clamp_nan((in[j] - mean[j]) / den[j], -5.0f, 5.0f);
            }
#pragma unroll
            for (int k = 0; k < CH; ++k) {
                if (k0 + k >= NF2) break;
                r2[k0 + k] = make_float2(out[2 * k], out[2 * k + 1]);
            }
        }
        if (full) {
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
                bulk_s2g(nm.out + e0 * OBS_ROW, x, WT * OBS_ROW * 4);
                bulk_commit();
                bulk_wait_read0();
            }
        } else {
            __syncwarp();
            for (int i = lane; i < nv * OBS_ROW; i += WT) nm.out[e0 * OBS_ROW + i] = x[i];
        }
        return;
    }
    if (OBS && full && lane == 0) bulk_wait_read0();   // shared memory must outlive the bulk store's reads
}

template <int PARTS, bool CLEATS, int TILE, int TASK>
__global__ void __launch_bounds__(TILE, BEZK_TILE_CTAS * 128 / TILE) task_tile_kernel(const TaskArgs a, const __grid_constant__ BezkTaskCfg cfg) {
    task_tile<PARTS, CLEATS, TILE, TASK, false>(a, cfg);
}
// the same step with the L2 policy of set_l2_policy: carried state evict_last, simulator tensors evict_first
template <int PARTS, bool CLEATS, int TILE, int TASK>
__global__ void __launch_bounds__(TILE, BEZK_TILE_CTAS * 128 / TILE) task_tile_l2_kernel(const TaskArgs a, const __grid_constant__ BezkTaskCfg cfg) {
    task_tile<PARTS, CLEATS, TILE, TASK, true>(a, cfg);
}
// the whole step with the episode accumulators (bezk_post_physics_rollout_ep), plain and with the L2 policy
template <bool CLEATS, int TILE, int TASK>
__global__ void __launch_bounds__(TILE, BEZK_TILE_CTAS * 128 / TILE) task_tile_ep_kernel(const TaskArgs a, const __grid_constant__ BezkTaskCfg cfg,
                                                                                         const EpArgs ep) {
    task_tile<7, CLEATS, TILE, TASK, false>(a, cfg, ep);
}
template <bool CLEATS, int TILE, int TASK>
__global__ void __launch_bounds__(TILE, BEZK_TILE_CTAS * 128 / TILE) task_tile_ep_l2_kernel(const TaskArgs a, const __grid_constant__ BezkTaskCfg cfg,
                                                                                            const EpArgs ep) {
    task_tile<7, CLEATS, TILE, TASK, true>(a, cfg, ep);
}
// the whole step with the episode accumulators and the eval-mode observation normaliser (bezk_post_physics_rollout_ep_norm)
template <bool CLEATS, int TILE, int TASK>
__global__ void __launch_bounds__(TILE, BEZK_TILE_CTAS * 128 / TILE) task_tile_obsnorm_kernel(const TaskArgs a,
                                                                                              const __grid_constant__ BezkTaskCfg cfg,
                                                                                              const EpArgs ep, const NormArgs nm) {
    task_tile<7, CLEATS, TILE, TASK, false>(a, cfg, ep, nm);
}
template <bool CLEATS, int TILE, int TASK>
__global__ void __launch_bounds__(TILE, BEZK_TILE_CTAS * 128 / TILE) task_tile_obsnorm_l2_kernel(const TaskArgs a,
                                                                                                 const __grid_constant__ BezkTaskCfg cfg,
                                                                                                 const EpArgs ep, const NormArgs nm) {
    task_tile<7, CLEATS, TILE, TASK, true>(a, cfg, ep, nm);
}
// the EP and the EP + normaliser steps that also count their done envs per outcome class (bezk_post_physics_rollout_ep_outcome)
template <bool CLEATS, int TILE, int TASK>
__global__ void __launch_bounds__(TILE, BEZK_TILE_CTAS * 128 / TILE) task_tile_outcome_kernel(const TaskArgs a,
                                                                                              const __grid_constant__ BezkTaskCfg cfg,
                                                                                              const EpArgs ep, const OutArgs oa) {
    task_tile<7, CLEATS, TILE, TASK, false>(a, cfg, ep, oa);
}
template <bool CLEATS, int TILE, int TASK>
__global__ void __launch_bounds__(TILE, BEZK_TILE_CTAS * 128 / TILE) task_tile_outcome_l2_kernel(const TaskArgs a,
                                                                                                 const __grid_constant__ BezkTaskCfg cfg,
                                                                                                 const EpArgs ep, const OutArgs oa) {
    task_tile<7, CLEATS, TILE, TASK, true>(a, cfg, ep, oa);
}
template <bool CLEATS, int TILE, int TASK>
__global__ void __launch_bounds__(TILE, BEZK_TILE_CTAS * 128 / TILE) task_tile_obsnorm_outcome_kernel(
    const TaskArgs a, const __grid_constant__ BezkTaskCfg cfg, const EpArgs ep, const NormArgs nm, const OutArgs oa) {
    task_tile<7, CLEATS, TILE, TASK, false>(a, cfg, ep, nm, oa);
}
template <bool CLEATS, int TILE, int TASK>
__global__ void __launch_bounds__(TILE, BEZK_TILE_CTAS * 128 / TILE) task_tile_obsnorm_outcome_l2_kernel(
    const TaskArgs a, const __grid_constant__ BezkTaskCfg cfg, const EpArgs ep, const NormArgs nm, const OutArgs oa) {
    task_tile<7, CLEATS, TILE, TASK, true>(a, cfg, ep, nm, oa);
}
// the EP and the EP + outcome steps that also sum their envs' reward terms per warp (bezk_post_physics_rollout_ep_terms)
template <bool CLEATS, int TILE, int TASK>
__global__ void __launch_bounds__(TILE, BEZK_TILE_CTAS * 128 / TILE) task_tile_terms_kernel(const TaskArgs a,
                                                                                            const __grid_constant__ BezkTaskCfg cfg,
                                                                                            const EpArgs ep, const TermArgs ta) {
    task_tile<7, CLEATS, TILE, TASK, false>(a, cfg, ep, ta);
}
template <bool CLEATS, int TILE, int TASK>
__global__ void __launch_bounds__(TILE, BEZK_TILE_CTAS * 128 / TILE) task_tile_terms_l2_kernel(const TaskArgs a,
                                                                                               const __grid_constant__ BezkTaskCfg cfg,
                                                                                               const EpArgs ep, const TermArgs ta) {
    task_tile<7, CLEATS, TILE, TASK, true>(a, cfg, ep, ta);
}
template <bool CLEATS, int TILE, int TASK>
__global__ void __launch_bounds__(TILE, BEZK_TILE_CTAS * 128 / TILE) task_tile_outcome_terms_kernel(
    const TaskArgs a, const __grid_constant__ BezkTaskCfg cfg, const EpArgs ep, const OutArgs oa, const TermArgs ta) {
    task_tile<7, CLEATS, TILE, TASK, false>(a, cfg, ep, oa, ta);
}
template <bool CLEATS, int TILE, int TASK>
__global__ void __launch_bounds__(TILE, BEZK_TILE_CTAS * 128 / TILE) task_tile_outcome_terms_l2_kernel(
    const TaskArgs a, const __grid_constant__ BezkTaskCfg cfg, const EpArgs ep, const OutArgs oa, const TermArgs ta) {
    task_tile<7, CLEATS, TILE, TASK, true>(a, cfg, ep, oa, ta);
}
// every EP step above that also carries the game term returns (bezk_post_physics_rollout_ep_game_terms): Ep is that step's pack
// followed by GameTermArgs
template <bool CLEATS, int TILE, int TASK, typename... Ep>
__global__ void __launch_bounds__(TILE, BEZK_TILE_CTAS * 128 / TILE) task_tile_game_kernel(const TaskArgs a,
                                                                                           const __grid_constant__ BezkTaskCfg cfg,
                                                                                           const Ep... eps) {
    task_tile<7, CLEATS, TILE, TASK, false>(a, cfg, eps...);
}
template <bool CLEATS, int TILE, int TASK, typename... Ep>
__global__ void __launch_bounds__(TILE, BEZK_TILE_CTAS * 128 / TILE) task_tile_game_l2_kernel(const TaskArgs a,
                                                                                              const __grid_constant__ BezkTaskCfg cfg,
                                                                                              const Ep... eps) {
    task_tile<7, CLEATS, TILE, TASK, true>(a, cfg, eps...);
}

// ------------------------------------------------------------------------------------------------
// K3 (function level): reset_idx over an explicit id list; one thread per (id, dof) pair + root rows.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) reset_idx_kernel(const int64_t* __restrict__ env_ids, int64_t k, const float* __restrict__ uniforms,
                                                        uint64_t seed, uint64_t step, float* dof_state, float* root_states,
                                                        const float* __restrict__ initial_root, int64_t* progress, int64_t* reset,
                                                        const __grid_constant__ BezkTaskCfg cfg, int64_t n, int root_floats,
                                                        float* goal, const float* __restrict__ goal_uniforms, int64_t env_base) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= k) return;
    const int64_t e = env_ids[i];
    if (e < 0 || e >= n) return;
    float u[36], row[36];
    if (uniforms) {
#pragma unroll
        for (int c = 0; c < 36; ++c) u[c] = uniforms[i * 36 + c];
    } else {
        philox_reset_uniforms(seed, step, env_base + e, u);          // keyed by the GLOBAL env id
    }
    reset_dof_row(u, cfg, row);
#pragma unroll
    for (int c = 0; c < 36; ++c) dof_state[e * DOF_ROW + c] = row[c];
    if (cfg.flags & BEZK_F_RESET_ROOT_STATES) {
        for (int c = 0; c < root_floats; ++c) root_states[e * root_floats + c] = initial_root[e * root_floats + c];
    }
    if (goal) {                                    // walk / orient: one goal draw per reset batch (walk_env.py:566-574)
        float ux, uy;
        if (goal_uniforms) { ux = goal_uniforms[0]; uy = goal_uniforms[1]; }
        else { const Philox4 x = philox_goal(seed, step); ux = u01(x.x); uy = u01(x.y); }
        goal[e * 2] = 4.0f * ux + -2.0f;
        goal[e * 2 + 1] = 4.0f * uy + -2.0f;
    }
    progress[e] = 0;
    reset[e] = 0;
}

__global__ void philox_uniforms_kernel(uint64_t seed, uint64_t step, float* out, int64_t n) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    float u[36];
    philox_reset_uniforms(seed, step, e, u);
#pragma unroll
    for (int c = 0; c < 36; ++c) out[e * 36 + c] = u[c];
}

// ------------------------------------------------------------------------------------------------
// host launchers
// ------------------------------------------------------------------------------------------------
static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
static inline bool aligned8(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 7u) == 0; }

// Ep: empty (task_tile_kernel / task_tile_l2_kernel), the episode accumulators (task_tile_ep_kernel / task_tile_ep_l2_kernel) or
// those and the observation normaliser (task_tile_obsnorm_kernel / task_tile_obsnorm_l2_kernel), either EP pack followed by the
// outcome counts (task_tile_outcome_kernel / task_tile_obsnorm_outcome_kernel and their _l2 forms), the EP or EP + outcome pack
// followed by the reward terms (task_tile_terms_kernel / task_tile_outcome_terms_kernel and their _l2 forms), any of those packs
// followed by the game term returns (task_tile_game_kernel / task_tile_game_l2_kernel); a.l2_resident picks the L2 variant.  Every
// variant has the same shared memory: the normaliser works in the observation tile.
template <int PARTS, bool CLEATS, int TILE, int TASK, typename... Ep>
static cudaError_t launch_tile(const TaskArgs& a, const BezkTaskCfg& cfg, cudaStream_t st, const Ep&... eps) {
    static_assert(sizeof...(Ep) == 0 || PARTS == 7, "the episode accumulators ride in the whole step");
    const auto kernel = [&] {
        constexpr bool NORM = has_arg<NormArgs, Ep...>, OUT = has_arg<OutArgs, Ep...>, TERMS = has_arg<TermArgs, Ep...>;
        if constexpr (sizeof...(Ep) == 0)
            return a.l2_resident ? task_tile_l2_kernel<PARTS, CLEATS, TILE, TASK> : task_tile_kernel<PARTS, CLEATS, TILE, TASK>;
        else if constexpr (has_arg<GameTermArgs, Ep...>)
            return a.l2_resident ? task_tile_game_l2_kernel<CLEATS, TILE, TASK, Ep...> : task_tile_game_kernel<CLEATS, TILE, TASK, Ep...>;
        else if constexpr (TERMS && OUT)
            return a.l2_resident ? task_tile_outcome_terms_l2_kernel<CLEATS, TILE, TASK> : task_tile_outcome_terms_kernel<CLEATS, TILE, TASK>;
        else if constexpr (TERMS)
            return a.l2_resident ? task_tile_terms_l2_kernel<CLEATS, TILE, TASK> : task_tile_terms_kernel<CLEATS, TILE, TASK>;
        else if constexpr (NORM && OUT)
            return a.l2_resident ? task_tile_obsnorm_outcome_l2_kernel<CLEATS, TILE, TASK> : task_tile_obsnorm_outcome_kernel<CLEATS, TILE, TASK>;
        else if constexpr (OUT)
            return a.l2_resident ? task_tile_outcome_l2_kernel<CLEATS, TILE, TASK> : task_tile_outcome_kernel<CLEATS, TILE, TASK>;
        else if constexpr (NORM)
            return a.l2_resident ? task_tile_obsnorm_l2_kernel<CLEATS, TILE, TASK> : task_tile_obsnorm_kernel<CLEATS, TILE, TASK>;
        else
            return a.l2_resident ? task_tile_ep_l2_kernel<CLEATS, TILE, TASK> : task_tile_ep_kernel<CLEATS, TILE, TASK>;
    }();
    const size_t smem = (size_t)(smem_in_floats(TILE, TASK) + (a.obs_clipped ? smem_obs_floats(TILE, TASK) : 0)) * sizeof(float);
    static SmemOptIn opt_in, opt_in_l2;    // per instantiation, per device
    if (cudaError_t err = (a.l2_resident ? opt_in_l2 : opt_in).ensure(kernel, (smem_in_floats(TILE, TASK) + smem_obs_floats(TILE, TASK)) * sizeof(float)))
        return err;
    const int64_t tiles = (a.n + TILE - 1) / TILE;
    return launch_ex(kernel, dim3((unsigned)tiles), dim3(TILE), smem, st, a, cfg, eps...);
}

template <int V>
using Int = std::integral_constant<int, V>;

cudaError_t launch_task(int task, int parts, const TaskArgs& a, const BezkTaskCfg& cfg, const EpArgs* ep, cudaStream_t st,
                        const NormArgs* nm, const OutArgs* oa, const TermArgs* ta, const GameTermArgs* ga) {
    const bool cleats = (cfg.flags & BEZK_F_CLEATS) != 0;
    if ((nm || oa || ta || ga) && !ep) return cudaErrorInvalidValue;
    if (ta && nm) return cudaErrorInvalidValue;
    // one (TASK, PARTS) pair, with or without cleats; the episode accumulators (and the normaliser / outcome counts / reward terms /
    // game term returns) only with the whole step
    const auto tile = [&](auto task_c, auto parts_c) -> cudaError_t {
        constexpr int TASK = decltype(task_c)::value, PARTS = decltype(parts_c)::value;
        if constexpr (PARTS == 7) {
            // the EP pack, followed by the game term returns when they are armed
            const auto whole = [&](const auto&... pk) -> cudaError_t {
                if (ga)
                    return cleats ? launch_tile<7, true, BEZK_TILE, TASK>(a, cfg, st, pk..., *ga)
                                  : launch_tile<7, false, BEZK_TILE, TASK>(a, cfg, st, pk..., *ga);
                return cleats ? launch_tile<7, true, BEZK_TILE, TASK>(a, cfg, st, pk...) : launch_tile<7, false, BEZK_TILE, TASK>(a, cfg, st, pk...);
            };
            if (ta && oa) return whole(*ep, *oa, *ta);
            if (ta) return whole(*ep, *ta);
            if (nm && oa) return whole(*ep, *nm, *oa);
            if (oa) return whole(*ep, *oa);
            if (nm) return whole(*ep, *nm);
            if (ep) return whole(*ep);
        }
        if (ep) return cudaErrorInvalidValue;
        return cleats ? launch_tile<PARTS, true, BEZK_TILE, TASK>(a, cfg, st) : launch_tile<PARTS, false, BEZK_TILE, TASK>(a, cfg, st);
    };
    // walk / orient: the fused step (7), the observation kernel (2 or 3) and the reward kernel (4)
    const auto sibling = [&](auto task_c) -> cudaError_t {
        switch (parts) {
            case 2: return tile(task_c, Int<2>{});
            case 3: return tile(task_c, Int<3>{});
            case 4: return tile(task_c, Int<4>{});
            case 7: return tile(task_c, Int<7>{});
            default: return cudaErrorInvalidValue;
        }
    };
    switch (task) {
        case BEZK_TASK_WALK: return sibling(Int<BEZK_TASK_WALK>{});
        case BEZK_TASK_ORIENT: return sibling(Int<BEZK_TASK_ORIENT>{});
        case BEZK_TASK_KICK: break;
        default: return cudaErrorInvalidValue;
    }
    // BezKick: every non-empty subset of the three parts
    constexpr Int<BEZK_TASK_KICK> kick{};
    switch (parts) {
        case 1: return tile(kick, Int<1>{});
        case 2: return tile(kick, Int<2>{});
        case 3: return tile(kick, Int<3>{});
        case 4: return tile(kick, Int<4>{});
        case 5: return tile(kick, Int<5>{});
        case 6: return tile(kick, Int<6>{});
        case 7: return tile(kick, Int<7>{});
        default: return cudaErrorInvalidValue;
    }
}

__global__ void goal_uniforms_kernel(uint64_t seed, uint64_t step, float* out2) {
    const Philox4 x = philox_goal(seed, step);
    out2[0] = u01(x.x); out2[1] = u01(x.y);
}
cudaError_t launch_goal_uniforms(uint64_t seed, uint64_t step, float* out2, cudaStream_t st) {
    goal_uniforms_kernel<<<1, 1, 0, st>>>(seed, step, out2);
    return cudaGetLastError();
}

void fill_alignment(TaskArgs& a, const BezkTaskCfg& cfg) {
    if (a.dof_state_wb == nullptr) a.dof_state_wb = a.dof_state;
    if (a.root_states_wb == nullptr) a.root_states_wb = a.root_states;
    if (a.values_stride <= 0) a.values_stride = 1;
    a.use_tma = aligned16(a.dof_state) && aligned16(a.root_states) && aligned16(a.dof_state_wb) && (a.obs == nullptr || aligned16(a.obs)) &&
                (a.obs_clipped == nullptr || aligned16(a.obs_clipped));
    if (a.rb_stride == 0) { a.rb_stride = cfg.num_bodies * 13; a.rb_off = cfg.imu_body * 13 + 3; }
    if (a.cf_stride == 0) { a.cf_stride = cfg.num_bodies * 3; a.cf_l_off = cfg.left_foot_body * 3; a.cf_r_off = cfg.right_foot_body * 3; }
    a.rb_vec2 = aligned8(a.rigid_body) && (a.rb_stride % 2 == 0) && (a.rb_off % 2 == 0);
    // window path for slices that are only 4-byte aligned: needs a 16-byte aligned base and 12 readable bytes either side of
    // the slice inside the tensor (the slice starts >= 3 floats into its body row; it must not sit in the last body)
    a.rb_win = !a.rb_vec2 && aligned16(a.rigid_body) && a.rb_off >= 3 && a.rb_stride == cfg.num_bodies * 13 &&
               cfg.imu_body + 1 < cfg.num_bodies;
    // 0: 64-byte granules only; 1 (default): per-lane 64 / 128-byte choice; 2: full 128-byte lines wherever the span allows.
    // Read ONCE per process (A/B measurement knob, profiles/r01_fetch_granularity.md), never on the launch path.
    static const int smart_granule = env_int("BEZK_SMART_GRANULE", 1);
    a.smart_granule = smart_granule;
    a.cf_vec2 = a.net_contact != nullptr && aligned8(a.net_contact) && (a.cf_stride % 2 == 0) && (a.cf_l_off % 2 == 0) &&
                (a.cf_r_off % 2 == 0);
}

// L2 residency of the carried per-env state.  Between two steps the fused kernel streams ~650 B/env of simulator tensors through
// L2 (dense tiles, 64-byte gathers) next to K0 and the rollout slots; at normal priority that evicts the ~270 B/env the step
// re-reads or overwrites at the SAME address every step (obs rows, bookkeeping, prev_lin_vel, goal / ball_init), so each step paid
// HBM for that state twice (write-back, re-fetch).  When the carried state of all n envs fits BEZK_L2_BUDGET_PCT of the device's
// L2 and the step's streamed + carried bytes do not (below that L2 keeps both anyway, and the hints only cost K0 and GAE their hits),
// the carried state is accessed with evict_last and the streams with evict_first; otherwise nothing is hinted.  Measured on B200
// (profiles/r03_l2_resident.md): a partial set -- envs [0, k) resident at 1 048 576 envs -- and the hints at 65 536 envs were
// both slower than no hints.  Launches whose carried buffers are not all device memory (host pipelines) are not hinted.
#ifndef BEZK_L2_BUDGET_PCT
#define BEZK_L2_BUDGET_PCT 75
#endif
static int64_t l2_bytes_of_device() {
    static std::atomic<int64_t> bytes[64];          // per device, 0 = not read yet
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 0;
    int64_t b = bytes[dev].load(std::memory_order_relaxed);
    if (b == 0) {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrL2CacheSize, dev) != cudaSuccess) return 0;
        b = v;
        bytes[dev].store(b, std::memory_order_relaxed);
    }
    return b;
}
static bool on_device(const void* p) {
    if (p == nullptr) return true;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { (void)cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeDevice;
}
void set_l2_policy(int task, uint32_t flags, TaskArgs& a, const EpArgs* ep, const GameTermArgs* ga) {
    a.l2_resident = 0;
    if (!l2_resident_enabled()) return;
    const void* carried[] = {a.obs, a.obs_clipped, a.reset_out, a.progress_out, a.timeout_buf, a.rew, a.prev_lin_vel, a.goal,
                             a.ball_init, a.goal_angle, ep ? ep->ret : nullptr, ep ? ep->len : nullptr, ga ? ga->acc : nullptr};
    int64_t per_env = ep ? 8 : 0;          // the two episode accumulators, when armed
    if (ga) per_env += 4 * reward_terms(task);   // and the K game term accumulators
    for (const void* p : carried)
        if (!on_device(p)) return;
    const bool obs_kept = !(flags & BEZK_F_OBS_STREAMED);
    if (a.obs && obs_kept) per_env += obs_row(task) * 4;
    if (a.obs_clipped && obs_kept) per_env += obs_row(task) * 4;
    if (a.reset_out) per_env += 8;
    if (a.progress_out) per_env += 8;
    if (a.timeout_buf) per_env += 8;
    if (a.rew) per_env += 4;
    if (a.prev_lin_vel) per_env += 12;
    if (a.goal) per_env += 8;
    if (a.ball_init && task == BEZK_TASK_KICK) per_env += 8;
    if (a.goal_angle && task == BEZK_TASK_ORIENT) per_env += 4;
    const int64_t l2 = l2_bytes_of_device();
    // per env and step the simulator tensors cost the two dense rows and at least three 64-byte granules (IMU slice, two feet)
    const int64_t streamed = (DOF_ROW + root_row(task)) * 4 + 3 * 64;
    if (per_env == 0 || a.n * per_env > l2 * BEZK_L2_BUDGET_PCT / 100 || a.n * (per_env + streamed) <= l2) return;
    a.l2_resident = 1;
}

// applypriority works on one 128-byte line: only the lines entirely inside the range are touched
__global__ void __launch_bounds__(256) l2_release_kernel(const char* base, int64_t lines) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < lines; i += (int64_t)gridDim.x * blockDim.x)
        asm volatile("applypriority.global.L2::evict_normal [%0], 128;" ::"l"(base + i * 128) : "memory");
}
cudaError_t launch_l2_release(const void* ptr, uint64_t bytes, cudaStream_t st) {
    const uintptr_t lo = (reinterpret_cast<uintptr_t>(ptr) + 127) & ~(uintptr_t)127;
    const uintptr_t hi = (reinterpret_cast<uintptr_t>(ptr) + bytes) & ~(uintptr_t)127;
    if (hi <= lo) return cudaSuccess;
    const int64_t lines = (int64_t)((hi - lo) / 128);
    int64_t blocks = (lines + 255) / 256;
    if (blocks > 148LL * 16) blocks = 148LL * 16;
    l2_release_kernel<<<(unsigned)blocks, 256, 0, st>>>(reinterpret_cast<const char*>(lo), lines);
    return cudaGetLastError();
}

// Host pipeline: the sparse Isaac Gym rows leave PINNED HOST memory through the copy engines -- strided cudaMemcpy2DAsync
// pulls into compact device staging -- instead of 64-byte zero-copy reads issued by the SMs (profiles/r02_host_link.md).
//   imu_stage  (n, 10)                    <- rigid_body row (env, imu_body), floats 3..12                       (40 B of 52 * num_bodies)
//   feet_stage (n, 8)  [l xyz _ r xyz _]  <- net_contact rows (env, left_foot_body), (env, right_foot_body)     (2 x 12 B of 12 * num_bodies)
//   cleats:    (n, 24) [l 12, r 12]       <- the two runs of 4 cleat bodies                                     (2 x 48 B)
cudaError_t stage_sparse_rows(const float* rigid_body, const float* net_contact, const BezkTaskCfg& cfg, float* imu_stage,
                              float* feet_stage, int64_t env0, int64_t n, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    const size_t rb_pitch = (size_t)cfg.num_bodies * 13 * sizeof(float), cf_pitch = (size_t)cfg.num_bodies * 3 * sizeof(float);
    const bool cleats = (cfg.flags & BEZK_F_CLEATS) != 0;
    const size_t fw = cleats ? 48 : 12, fpitch = cleats ? 96 : 32, roff = cleats ? 48 : 16;
    cudaError_t e = cudaMemcpy2DAsync(imu_stage + env0 * 10, 40, rigid_body + (env0 * cfg.num_bodies + cfg.imu_body) * 13 + 3, rb_pitch,
                                      40, (size_t)n, cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) return e;
    char* fs = reinterpret_cast<char*>(feet_stage) + env0 * fpitch;
    e = cudaMemcpy2DAsync(fs, fpitch, net_contact + (env0 * cfg.num_bodies + cfg.left_foot_body) * 3, cf_pitch, fw, (size_t)n,
                          cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) return e;
    return cudaMemcpy2DAsync(fs + roff, fpitch, net_contact + (env0 * cfg.num_bodies + cfg.right_foot_body) * 3, cf_pitch, fw, (size_t)n,
                             cudaMemcpyHostToDevice, st);
}

// The foot rows of bezk_stage_sparse_rows pulled by the SMs instead (zero-copy reads of pinned host memory): the copy engine
// that serves the H2D direction is row-rate-bound on the strided pulls (1.4 ns per row), so letting a small gather kernel fetch
// the two foot rows over PCIe WHILE the engine moves the dense tensors and the IMU slices shortens the H2D critical path.
__global__ void __launch_bounds__(256) stage_feet_kernel(const float* __restrict__ net_contact, float* __restrict__ feet_stage,
                                                         const __grid_constant__ BezkTaskCfg cfg, int64_t env0, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t e = env0 + i;
    const bool cleats = (cfg.flags & BEZK_F_CLEATS) != 0;
    const int w = cleats ? 12 : 3, pitch = cleats ? 24 : 8, roff = cleats ? 12 : 4;
    const float* l = net_contact + (e * cfg.num_bodies + cfg.left_foot_body) * 3;
    const float* r = net_contact + (e * cfg.num_bodies + cfg.right_foot_body) * 3;
    float* d = feet_stage + e * pitch;
    for (int k = 0; k < w; ++k) { d[k] = ldg64B_nc(l + k); d[roff + k] = ldg64B_nc(r + k); }
}

cudaError_t stage_feet_gather(const float* net_contact, const BezkTaskCfg& cfg, float* feet_stage, int64_t env0, int64_t n,
                              cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    stage_feet_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(net_contact, feet_stage, cfg, env0, n);
    return cudaGetLastError();
}

cudaError_t stage_imu_rows(const float* rigid_body, const BezkTaskCfg& cfg, float* imu_stage, int64_t env0, int64_t n, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    const size_t rb_pitch = (size_t)cfg.num_bodies * 13 * sizeof(float);
    return cudaMemcpy2DAsync(imu_stage + env0 * 10, 40, rigid_body + (env0 * cfg.num_bodies + cfg.imu_body) * 13 + 3, rb_pitch, 40,
                             (size_t)n, cudaMemcpyHostToDevice, st);
}

// Host pipeline, packed records (bezk_host_pack.cu): the 3 (7) root-state floats the step reads travel inside the per-env record;
// this scatters them into the columns of the device image of root_states the tile kernel's dense bulk copy expects (the other
// columns are never read).  28 B per env, a few microseconds per chunk.
__global__ void __launch_bounds__(256) unpack_root_kernel(const float* __restrict__ records, PackLayout L, float* __restrict__ root_states,
                                                          int root_row_floats, int64_t n) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const float* q = records + e * L.stride + L.root_off;
    float* r = root_states + e * root_row_floats;
    r[0] = q[0]; r[1] = q[1]; r[2] = q[2];
    if (L.root_n == 7) { r[13] = q[3]; r[14] = q[4]; r[20] = q[5]; r[21] = q[6]; }
}

cudaError_t launch_unpack_root(int task, const float* records, PackLayout L, float* root_states, int64_t n, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    unpack_root_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(records, L, root_states, root_row(task), n);
    return cudaGetLastError();
}

cudaError_t launch_pre_physics(const float* actions, float* actions_out, float* targets, const BezkTaskCfg& cfg,
                               int64_t n, cudaStream_t st) {
    const int vec2 = aligned8(actions) && aligned8(targets) && (actions_out == nullptr || aligned8(actions_out));
    const int64_t per_block = (int64_t)K0_ROWS * K0_UNROLL;
    int64_t blocks = vec2 ? (n + per_block - 1) / per_block : (n * 18 + K0_THREADS - 1) / K0_THREADS;
    if (blocks < 1) blocks = 1;
    if (!vec2 && blocks > 148LL * 64) blocks = 148LL * 64;      // scalar path is grid-strided
    return launch_ex(pre_physics_kernel, dim3((unsigned)blocks), dim3(K0_THREADS), 0, st, actions, actions_out, targets, cfg, n, vec2);
}

cudaError_t launch_reset_idx(const int64_t* env_ids, int64_t k, const float* uniforms, uint64_t seed, uint64_t step,
                             float* dof_state, float* root_states, const float* initial_root, int64_t* progress,
                             int64_t* reset, const BezkTaskCfg& cfg, int64_t n, int task, float* goal, const float* goal_uniforms,
                             int64_t env_base, cudaStream_t st) {
    if (k == 0) return cudaSuccess;
    reset_idx_kernel<<<(unsigned)((k + 127) / 128), 128, 0, st>>>(env_ids, k, uniforms, seed, step, dof_state, root_states,
                                                                  initial_root, progress, reset, cfg, n, root_row(task),
                                                                  task == BEZK_TASK_KICK ? nullptr : goal, goal_uniforms, env_base);
    return cudaGetLastError();
}

cudaError_t launch_philox_uniforms(uint64_t seed, uint64_t step, float* out, int64_t n, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    philox_uniforms_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(seed, step, out, n);
    return cudaGetLastError();
}

}  // namespace bezk
