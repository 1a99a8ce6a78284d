// Rollout plumbing either side of the task step (SURVEY 8f rows 1-2) for B200 (sm_100a):
//   * swap_and_flatten01 -- rl_games' (T, N, ...) -> (N*T, ...) env-major flattening as ONE tiled shared-memory
//     transposition per tensor (the slab-addressed learner kernels in bezk_learner.cu need no flattening pass at all;
//     this entry exists for callers that want rl_games' exact dataset layout);
//   * policy_head -- everything rl_games does between the policy MLP and the simulator in play_steps: Normal sampling,
//     neglogp, value un-normalisation, the experience-buffer writes (actions / neglogpacs / values / mus / sigmas slot t),
//     preprocess_actions' clamp and K0's PD targets, in one pass over the (N,18) network output.
// Both are HBM-bound streaming kernels.
#include "bezk_common.cuh"
#include "bezk_internal.h"
#include <math.h>
#include <string.h>

namespace bezk {

// ------------------------------------------------------------------------------------------------
// swap_and_flatten01: dst[(e - env0) * T + t][:] = src[t * N + e][:],  rows of `w` elements of type E.
// CTA tile = tb timesteps x eb envs: coalesced reads of eb*w-element runs (one per t), transposed placement in shared
// memory, then the tile leaves as eb runs of tb*w elements (ONE contiguous run when tb == T).
// ------------------------------------------------------------------------------------------------
template <typename E>
__global__ void __launch_bounds__(256) swap_flatten_kernel(const E* __restrict__ src, E* __restrict__ dst, int horizon, int64_t n,
                                                           int64_t env0, int64_t envs, int w, int eb, int tb) {
    extern __shared__ __align__(16) unsigned char sf_smem[];
    E* tile = reinterpret_cast<E*>(sf_smem);                    // [eb][tb][w]
    pdl_launch_dependents();
    pdl_wait();
    const int64_t eblk0 = (int64_t)blockIdx.x * eb;
    const int t0 = blockIdx.y * tb;
    const int ebc = (int)((envs - eblk0) < (int64_t)eb ? (envs - eblk0) : (int64_t)eb);
    const int tbc = (horizon - t0) < tb ? (horizon - t0) : tb;
    const int run = ebc * w;                                     // contiguous source elements per timestep
    const int total = tbc * run;
    const int orun = tbc * w;                                    // contiguous destination elements per env
    // narrow rows walk a COLUMN of the tile in the placement below: give them an odd row pitch (no bank conflicts).  Wide rows
    // (observations, actions) keep the dense pitch, so that the tile leaves as one linear run
    const int pitch = (w * (int)sizeof(E) <= 16) ? (orun | 1) : orun;
    for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
        const int t = idx / run, rem = idx - t * run;
        const int e = rem / w, c = rem - e * w;
        tile[e * pitch + t * w + c] = src[((int64_t)(t0 + t) * n + env0 + eblk0) * w + rem];
    }
    __syncthreads();
    E* d = dst + (eblk0 * (int64_t)horizon + t0) * w;
    if (pitch == orun && tbc == horizon) {                       // whole horizon in the tile, dense pitch: one linear run
        for (int idx = threadIdx.x; idx < total; idx += blockDim.x) d[idx] = tile[idx];
    } else {
        const int64_t dpitch = (int64_t)horizon * w;
        for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
            const int e = idx / orun, rem = idx - e * orun;
            d[e * dpitch + rem] = tile[e * pitch + rem];
        }
    }
}

// One-element rows (values, returns, neglogpacs, rewards, uint8 dones): the classic padded 32 x 128 transposition tile, indexed
// with shifts and masks only -- the generic kernel's per-element divisions made these the slowest rows (0.30 of the HBM peak).
constexpr int SFS_EB = 128;               // envs per tile
template <typename E>
__global__ void __launch_bounds__(256) swap_flatten_scalar_kernel(const E* __restrict__ src, E* __restrict__ dst, int horizon, int64_t n,
                                                                  int64_t env0, int64_t envs) {
    __shared__ E tile[SFS_EB][33];
    pdl_launch_dependents();
    pdl_wait();
    const int64_t eblk0 = (int64_t)blockIdx.x * SFS_EB;
    const int t0 = blockIdx.y * 32;
    const int ebc = (int)((envs - eblk0) < (int64_t)SFS_EB ? (envs - eblk0) : (int64_t)SFS_EB);
    const int tbc = (horizon - t0) < 32 ? (horizon - t0) : 32;
    for (int i = threadIdx.x; i < 32 * SFS_EB; i += 256) {       // reads: 128 consecutive envs of one timestep per 128 threads
        const int t = i >> 7, e = i & (SFS_EB - 1);
        if (t < tbc && e < ebc) tile[e][t] = src[(int64_t)(t0 + t) * n + env0 + eblk0 + e];
    }
    __syncthreads();
    E* d = dst + eblk0 * (int64_t)horizon + t0;
    for (int i = threadIdx.x; i < 32 * SFS_EB; i += 256) {       // writes: the 32 timesteps of one env per warp
        const int e = i >> 5, t = i & 31;
        if (t < tbc && e < ebc) d[(int64_t)e * horizon + t] = tile[e][t];
    }
}

template <typename E>
static cudaError_t launch_sf(const void* src, void* dst, int horizon, int64_t n, int64_t env0, int64_t envs, int w, cudaStream_t st) {
    if (w == 1) {
        const dim3 grid((unsigned)((envs + SFS_EB - 1) / SFS_EB), (unsigned)((horizon + 31) / 32));
        return launch_ex(swap_flatten_scalar_kernel<E>, grid, dim3(256), 0, st, (const E*)src, (E*)dst, horizon, n, env0, envs);
    }
    const int tb = horizon < 32 ? horizon : 32;
    int64_t eb = 32768 / ((int64_t)tb * w * (int64_t)sizeof(E));
    if (eb < 1) eb = 1;
    if (eb > 256) eb = 256;
    if (eb > envs) eb = envs;
    const size_t smem = (size_t)(((int64_t)tb * w) | 1) * eb * sizeof(E);      // covers both pitches
    if (smem > 200 * 1024) return cudaErrorInvalidValue;         // rows wider than 6 KB are not rollout tensors
    static SmemOptIn opt_in;                                      // per element type, per device
    if (smem > 48 * 1024) {
        if (cudaError_t e = opt_in.ensure(swap_flatten_kernel<E>, 200 * 1024)) return e;
    }
    const dim3 grid((unsigned)((envs + eb - 1) / eb), (unsigned)((horizon + tb - 1) / tb));
    return launch_ex(swap_flatten_kernel<E>, grid, dim3(256), smem, st, (const E*)src, (E*)dst, horizon, n, env0, envs, w, (int)eb, tb);
}

cudaError_t launch_swap_flatten(const void* src, void* dst, int horizon, int64_t n, int64_t env0, int64_t envs, int row_bytes,
                                cudaStream_t st) {
    if (envs == 0 || horizon == 0 || row_bytes == 0) return cudaSuccess;
    const uintptr_t al = reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst);
    if (row_bytes % 8 == 0 && (al & 7u) == 0) return launch_sf<uint64_t>(src, dst, horizon, n, env0, envs, row_bytes / 8, st);
    if (row_bytes % 4 == 0 && (al & 3u) == 0) return launch_sf<uint32_t>(src, dst, horizon, n, env0, envs, row_bytes / 4, st);
    return launch_sf<uint8_t>(src, dst, horizon, n, env0, envs, row_bytes, st);
}

// ------------------------------------------------------------------------------------------------
// policy_head.  rl_games ModelA2CContinuousLogStd.forward (is_train=False) + A2CBase.get_action_values (value
// un-normalisation) + play_steps' experience-buffer writes + preprocess_actions + (optionally) K0.
//   sigma = exp(logstd);  action = mu + sigma * eps;  neglogp = 0.5*sum(((a-mu)/sigma)^2) + 0.5*log(2pi)*18 + sum(logstd)
//   value = sqrt(var.float() + eps_v) * clamp(v, -5, 5) + mean.float()
//   env action = clamp(action, -1, 1) * 1 + 0  -> K0 (clip, zero head, + default pose, joint limits) -> targets
// eps: caller's N(0,1) draws, or Philox4x32-10 keyed (seed, step, env) + Box-Muller (5 blocks -> 9 pairs per env).
// One thread per env; the (128,18) tiles move by cp.async.bulk like the PPO-loss kernel's.
// ------------------------------------------------------------------------------------------------
constexpr int PH_TILE = 128;

// Box-Muller on the special-function unit: lg2 / sin / cos / sqrt approximations (absolute error of a draw <= ~1e-5).  The
// draws are NOISE (DR white noise, the policy's exploration noise): nothing downstream depends on their last bits -- neglogp is
// computed from the action actually sampled -- and the device functions that must agree bit for bit (bezk_dr_fill /
// bezk_normal_noise, used by the checkers) share this code.  Exact logf / sincosf / sqrtf cost ~120 of the DR
// kernel's ~250 instructions per quad and made a 12 B/element streaming pass issue-bound (0.61 -> 0.91 of the HBM peak).
__device__ __forceinline__ void box_muller_sfu(uint32_t a, uint32_t b, float* z0, float* z1) {
    const float u1 = (float)((a >> 8) + 1u) * (1.0f / 16777216.0f);       // (0, 1]
    const float u2 = (float)(b >> 8) * (1.0f / 16777216.0f);              // [0, 1)
    float r;
    const float t = -2.0f * __logf(u1);                                   // >= 0 (and -0 -> sqrt gives -0 -> draws of 0)
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(t));
    float sn, cs;
    __sincosf(6.283185307179586f * u2, &sn, &cs);
    *z0 = r * cs;
    *z1 = r * sn;
}

// the 18 standard normals of env `e` at (seed, step): blocks j = 0..4 -> uniforms (x,y), (z,w) -> pairs 2j, 2j+1
__device__ __forceinline__ void philox_normals18(uint64_t seed, uint64_t step, int64_t e, float (&z)[18]) {
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    const uint32_t c0 = (uint32_t)e, c1 = (uint32_t)((uint64_t)e >> 32);
    const uint32_t c2 = (uint32_t)step, c3h = ((uint32_t)(step >> 32) << 4);
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        const Philox4 r = philox4x32_10(c0, c1, c2, c3h + (uint32_t)j, k0 ^ 0x5851F42Du, k1);     // key tweak: stream distinct from the reset draws
        float a, b;
        box_muller_sfu(r.x, r.y, &a, &b);
        if (4 * j < 18) { z[4 * j] = a; z[4 * j + 1] = b; }
        box_muller_sfu(r.z, r.w, &a, &b);
        if (4 * j + 2 < 18) { z[4 * j + 2] = a; z[4 * j + 3] = b; }
    }
}

struct HeadArgs {
    const float *mu, *logstd, *value_norm, *noise;
    const double *value_mean, *value_var;
    float value_eps;
    uint64_t seed, step;
    int64_t env_base;            // global id of row 0 (Philox key): non-zero on env-sharded ranks
    float *actions, *neglogp, *values, *mus, *sigmas, *env_actions, *targets;
    int64_t n;
    int use_tma, has_task;
};

__global__ void __launch_bounds__(PH_TILE) policy_head_kernel(const HeadArgs a, const __grid_constant__ BezkTaskCfg cfg) {
    __shared__ __align__(128) float s_mu[PH_TILE * 18];
    __shared__ __align__(128) float s_eps[PH_TILE * 18];       // noise in, then env actions out
    __shared__ __align__(128) float s_act[PH_TILE * 18];
    __shared__ __align__(128) float s_tgt[PH_TILE * 18];
    __shared__ __align__(8) uint64_t s_bar;
    __shared__ float s_sigma[18], s_logstd[18], s_ry[18];
    const int tid = threadIdx.x;
    constexpr uint32_t TILE_BYTES = PH_TILE * 18 * 4;
    const int64_t i0 = (int64_t)blockIdx.x * PH_TILE;
    const int nv = (int)((a.n - i0) < (int64_t)PH_TILE ? (a.n - i0) : (int64_t)PH_TILE);
    const bool full = (nv == PH_TILE) && a.use_tma;
    const int64_t i = i0 + tid;
    const bool valid = tid < nv;

    pdl_launch_dependents();
    if (tid == 0) { mbar_init(&s_bar, 1); fence_mbar_init(); }
    pdl_wait();
    if (tid < 18) {
        const float ls = a.logstd[tid];
        const float sg = expf(ls);
        s_logstd[tid] = ls; s_sigma[tid] = sg; s_ry[tid] = Mth<true>::rcp_refined(sg);     // the divisor of every row's neglogp
    }
    __syncthreads();
    if (full) {
        if (tid == 0) {
            mbar_arrive_expect_tx(&s_bar, a.noise ? 2 * TILE_BYTES : TILE_BYTES);
            bulk_g2s(s_mu, a.mu + i0 * 18, TILE_BYTES, &s_bar);
            if (a.noise) bulk_g2s(s_eps, a.noise + i0 * 18, TILE_BYTES, &s_bar);
        }
    } else {
        for (int k = tid; k < nv * 18; k += PH_TILE) {
            s_mu[k] = a.mu[i0 * 18 + k];
            if (a.noise) s_eps[k] = a.noise[i0 * 18 + k];
        }
    }
    float vnorm = 0.0f;
    if (valid && a.value_norm) vnorm = a.value_norm[i];
    float z[18];
    if (!a.noise && valid) philox_normals18(a.seed, a.step, a.env_base + i, z);       // keyed by the GLOBAL env id; overlaps the tile load
    if (full) mbar_wait(&s_bar, 0);
    else __syncthreads();

    if (valid) {
        float lsum = 0.0f;
#pragma unroll
        for (int j = 0; j < 18; ++j) lsum += s_logstd[j];
        float sq = 0.0f;
        Mth<true> mq;                                                    // exact division without a branch per dimension
#pragma unroll
        for (int j = 0; j < 18; ++j) mq.check_divisor(s_sigma[j]);       // per-column constants: range-checked once per thread
        float2* mu2 = reinterpret_cast<float2*>(s_mu + tid * 18);
        float2* eps2 = reinterpret_cast<float2*>(s_eps + tid * 18);
        float2* act2 = reinterpret_cast<float2*>(s_act + tid * 18);
        float2* tgt2 = reinterpret_cast<float2*>(s_tgt + tid * 18);
#pragma unroll
        for (int h = 0; h < 9; ++h) {
            const float2 M = mu2[h];
            float2 E;
            if (a.noise) E = eps2[h]; else E = make_float2(z[2 * h], z[2 * h + 1]);
            const float mv[2] = {M.x, M.y}, ev[2] = {E.x, E.y};
            float av[2], cv[2], tv[2];
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const int j = 2 * h + q;
                const float sg = s_sigma[j];
                av[q] = mv[q] + sg * ev[q];                              // Normal(mu, sigma).sample()
                const float zz = mq.div_by(av[q] - mv[q], sg, s_ry[j]);  // models.py neglogp: the reference divides by sigma
                sq += zz * zz;
                cv[q] = clamp_nan(av[q], -1.0f, 1.0f) * 1.0f + 0.0f;     // preprocess_actions: clamp, rescale_actions(-1, 1)
                float stored;
                tv[q] = a.has_task ? k0_target(cv[q], j < 2, cfg.clip_actions, cfg.default_dof_pos[j], cfg.dof_lower[j],
                                                   cfg.dof_upper[j], &stored) : 0.0f;
            }
            act2[h] = make_float2(av[0], av[1]);
            eps2[h] = make_float2(cv[0], cv[1]);                         // s_eps now holds the env actions
            tgt2[h] = make_float2(tv[0], tv[1]);
        }
        if (mq.bad()) {                                                  // operands outside the fast sequence's range: plain operator
            sq = 0.0f;
            for (int j = 0; j < 18; ++j) {
                const float zz = (s_act[tid * 18 + j] - s_mu[tid * 18 + j]) / s_sigma[j];
                sq += zz * zz;
            }
        }
        if (a.neglogp) a.neglogp[i] = (0.5f * sq + (float)(0.5 * 1.8378770664093453 * 18.0)) + lsum;
        if (a.values) {
            float v = vnorm;
            if (a.value_mean) {
                const float mean = (float)a.value_mean[0];
                const float den = sqrtf((float)a.value_var[0] + a.value_eps);
                v = den * clamp_nan(vnorm, -5.0f, 5.0f) + mean;          // RunningMeanStd(unnorm=True)
            }
            a.values[i] = v;
        }
    }
    // ---- tiles out ----
    if (full) {
        fence_proxy_async_smem();
        __syncthreads();
        if (tid == 0) {
            if (a.actions) bulk_s2g(a.actions + i0 * 18, s_act, TILE_BYTES);
            if (a.mus) bulk_s2g(a.mus + i0 * 18, s_mu, TILE_BYTES);
            if (a.env_actions) bulk_s2g(a.env_actions + i0 * 18, s_eps, TILE_BYTES);
            if (a.targets) bulk_s2g(a.targets + i0 * 18, s_tgt, TILE_BYTES);
            bulk_commit();
        }
        // sigmas rows are all the same 18 values: the tile is an 18-periodic pattern, written as coalesced float4 stores
        if (a.sigmas) {
            float4* d4 = reinterpret_cast<float4*>(a.sigmas + i0 * 18);
            for (int k = tid; k < PH_TILE * 18 / 4; k += PH_TILE) {
                const int c = (4 * k) % 18;
                __stcs(d4 + k, make_float4(s_sigma[c], s_sigma[(c + 1) % 18], s_sigma[(c + 2) % 18], s_sigma[(c + 3) % 18]));
            }
        }
        if (tid == 0) bulk_wait_read0();
    } else {
        __syncthreads();
        for (int k = tid; k < nv * 18; k += PH_TILE) {
            if (a.actions) a.actions[i0 * 18 + k] = s_act[k];
            if (a.mus) a.mus[i0 * 18 + k] = s_mu[k];
            if (a.sigmas) a.sigmas[i0 * 18 + k] = s_sigma[k % 18];
            if (a.env_actions) a.env_actions[i0 * 18 + k] = s_eps[k];
            if (a.targets) a.targets[i0 * 18 + k] = s_tgt[k];
        }
    }
}

__global__ void normal_noise_kernel(uint64_t seed, uint64_t step, float* out, int64_t n, int64_t env_base) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    float z[18];
    philox_normals18(seed, step, env_base + e, z);
#pragma unroll
    for (int c = 0; c < 18; ++c) out[e * 18 + c] = z[c];
}

static inline bool al16(const void* p) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

cudaError_t launch_policy_head(const float* mu, const float* logstd, const float* value_norm, const double* value_mean,
                               const double* value_var, float value_eps, const float* noise, uint64_t seed, uint64_t step,
                               float* actions, float* neglogp, float* values, float* mus, float* sigmas, const BezkTaskCfg* cfg,
                               float* env_actions, float* targets, int64_t env_base, int64_t n, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    HeadArgs a;
    a.env_base = env_base;
    a.mu = mu; a.logstd = logstd; a.value_norm = value_norm; a.noise = noise; a.value_mean = value_mean; a.value_var = value_var;
    a.value_eps = value_eps; a.seed = seed; a.step = step; a.actions = actions; a.neglogp = neglogp; a.values = values;
    a.mus = mus; a.sigmas = sigmas; a.env_actions = env_actions; a.targets = cfg ? targets : nullptr; a.n = n;
    a.has_task = cfg != nullptr;
    a.use_tma = al16(mu) && al16(noise) && al16(actions) && al16(mus) && al16(sigmas) && al16(env_actions) && al16(targets);
    BezkTaskCfg c;
    if (cfg) c = *cfg; else memset(&c, 0, sizeof(c));
    return launch_ex(policy_head_kernel, dim3((unsigned)((n + PH_TILE - 1) / PH_TILE)), dim3(PH_TILE), 0, st, a, c);
}

cudaError_t launch_normal_noise(uint64_t seed, uint64_t step, float* out, int64_t n, int64_t env_base, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    normal_noise_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(seed, step, out, n, env_base);
    return cudaGetLastError();
}

}  // namespace bezk

// ------------------------------------------------------------------------------------------------
// Domain-randomisation noise lambdas (SURVEY 8f row 4; tasks/base/vec_task.py:562-618, applied at :314-315 to the actions
// and at :338-339 to obs_buf):   y = op(x, (corr * a_corr + b_corr) + w * a + b)
// with corr a persistent N(0,1) tensor (drawn once per randomisation period), w fresh N(0,1) ("gaussian") or U[0,1)
// ("uniform") noise per call, op = + ("additive") or * ("scaling").  Evaluation order as the reference's Python expression:
// ((corr' + w * a) + b).  w: caller's tensor, or Philox4x32-10 keyed (seed, step, element/4) -- 4 draws per block, one
// float4 of elements per thread -- so the pass moves 12 B/element (x, corr in; y out) and generates its noise in registers.
// ------------------------------------------------------------------------------------------------
namespace bezk {

__device__ __forceinline__ float dr_one(float x, float corr, float w, const BezkNoiseCfg& c) {
    const float cc = corr * c.a_corr + c.b_corr;
    const float nz = (cc + w * c.a) + c.b;
    return c.operation == 0 ? x + nz : x * nz;
}

// One quad (4 consecutive elements, one Philox counter).  FULL: all four exist and the pointers are 16-byte aligned -> float4
// accesses.  Otherwise every element is handled by fully unrolled, predicated scalar code: no array is ever indexed with a
// run-time value, so nothing lives in local memory (round 1's ragged-tail loops cost 77 STL in the SASS).
template <bool FULL>
__device__ __forceinline__ void dr_quad(const float* __restrict__ x, const float* __restrict__ corr, const float* __restrict__ white,
                                        uint64_t seed, uint64_t step, const BezkNoiseCfg& cfg, float* __restrict__ y,
                                        float* __restrict__ y_clip, float clip, int64_t q, int64_t total) {
    const int64_t i0 = q * 4;
    float x0 = 0.f, x1 = 0.f, x2 = 0.f, x3 = 0.f, c0 = 0.f, c1 = 0.f, c2 = 0.f, c3 = 0.f, w0, w1, w2, w3;
    const bool e1 = FULL || i0 + 1 < total, e2 = FULL || i0 + 2 < total, e3 = FULL || i0 + 3 < total;
    if (FULL) {
        const float4 t = ldg_stream4(reinterpret_cast<const float4*>(x) + q);
        x0 = t.x; x1 = t.y; x2 = t.z; x3 = t.w;
        if (corr) { const float4 u = ldg_stream4(reinterpret_cast<const float4*>(corr) + q); c0 = u.x; c1 = u.y; c2 = u.z; c3 = u.w; }
    } else {
        x0 = x[i0]; if (e1) x1 = x[i0 + 1]; if (e2) x2 = x[i0 + 2]; if (e3) x3 = x[i0 + 3];
        if (corr) { c0 = corr[i0]; if (e1) c1 = corr[i0 + 1]; if (e2) c2 = corr[i0 + 2]; if (e3) c3 = corr[i0 + 3]; }
    }
    if (white) {
        if (FULL) { const float4 t = ldg_stream4(reinterpret_cast<const float4*>(white) + q); w0 = t.x; w1 = t.y; w2 = t.z; w3 = t.w; }
        else { w0 = white[i0]; w1 = e1 ? white[i0 + 1] : 0.f; w2 = e2 ? white[i0 + 2] : 0.f; w3 = e3 ? white[i0 + 3] : 0.f; }
    } else {
        const Philox4 r = philox4x32_10((uint32_t)q, (uint32_t)((uint64_t)q >> 32), (uint32_t)step, (uint32_t)(step >> 32),
                                        (uint32_t)seed ^ 0x2545F491u, (uint32_t)(seed >> 32));
        if (cfg.distribution == 0) { box_muller_sfu(r.x, r.y, &w0, &w1); box_muller_sfu(r.z, r.w, &w2, &w3); }
        else { w0 = u01(r.x); w1 = u01(r.y); w2 = u01(r.z); w3 = u01(r.w); }
    }
    const float o0 = dr_one(x0, c0, w0, cfg), o1 = dr_one(x1, c1, w1, cfg), o2 = dr_one(x2, c2, w2, cfg), o3 = dr_one(x3, c3, w3, cfg);
    if (FULL) {
        __stcs(reinterpret_cast<float4*>(y) + q, make_float4(o0, o1, o2, o3));
        if (y_clip) __stcs(reinterpret_cast<float4*>(y_clip) + q, make_float4(clamp_nan(o0, -clip, clip), clamp_nan(o1, -clip, clip),
                                                                              clamp_nan(o2, -clip, clip), clamp_nan(o3, -clip, clip)));
    } else {
        y[i0] = o0; if (e1) y[i0 + 1] = o1; if (e2) y[i0 + 2] = o2; if (e3) y[i0 + 3] = o3;
        if (y_clip) {
            y_clip[i0] = clamp_nan(o0, -clip, clip);
            if (e1) y_clip[i0 + 1] = clamp_nan(o1, -clip, clip);
            if (e2) y_clip[i0 + 2] = clamp_nan(o2, -clip, clip);
            if (e3) y_clip[i0 + 3] = clamp_nan(o3, -clip, clip);
        }
    }
}

// y_clip != nullptr: also write clamp(y, -clip, clip) -- VecTask.step clamps the observations AFTER the noise (vec_task.py:338-343),
// so the clipped copy the step kernel produced from the noise-free rows is refreshed in the same pass.
__global__ void __launch_bounds__(256) dr_noise_kernel(const float* __restrict__ x, const float* __restrict__ corr,
                                                       const float* __restrict__ white, uint64_t seed, uint64_t step,
                                                       const __grid_constant__ BezkNoiseCfg cfg, float* __restrict__ y,
                                                       float* __restrict__ y_clip, float clip, int64_t total, int vec4) {
    pdl_launch_dependents();
    pdl_wait();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t nq = (total + 3) >> 2;                         // quads of elements; quad q owns Philox counter q
    const int64_t nfull = vec4 ? (total >> 2) : 0;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += stride) {
        if (q < nfull) dr_quad<true>(x, corr, white, seed, step, cfg, y, y_clip, clip, q, total);
        else dr_quad<false>(x, corr, white, seed, step, cfg, y, y_clip, clip, q, total);
    }
}

// white noise exactly as the Philox path above draws it (checker / corr initialisation): gaussian (0) or uniform (1)
__global__ void __launch_bounds__(256) dr_fill_kernel(uint64_t seed, uint64_t step, int distribution, float* __restrict__ out, int64_t total) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t nq = (total + 3) >> 2;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += stride) {
        const Philox4 r = philox4x32_10((uint32_t)q, (uint32_t)((uint64_t)q >> 32), (uint32_t)step, (uint32_t)(step >> 32),
                                        (uint32_t)seed ^ 0x2545F491u, (uint32_t)(seed >> 32));
        float wv[4];
        if (distribution == 0) { box_muller_sfu(r.x, r.y, &wv[0], &wv[1]); box_muller_sfu(r.z, r.w, &wv[2], &wv[3]); }
        else { wv[0] = u01(r.x); wv[1] = u01(r.y); wv[2] = u01(r.z); wv[3] = u01(r.w); }
        for (int k = 0; k < 4 && q * 4 + k < total; ++k) out[q * 4 + k] = wv[k];
    }
}

static inline int dr_blocks(int64_t total) {
    int64_t b = ((total + 3) / 4 + 255) / 256;
    if (b < 1) b = 1;
    const int64_t cap = 148LL * 8;
    return (int)(b > cap ? cap : b);
}

cudaError_t launch_dr_noise(const float* x, const float* corr, const float* white, uint64_t seed, uint64_t step,
                            const BezkNoiseCfg& cfg, float* y, float* y_clip, float clip, int64_t total, cudaStream_t st) {
    if (total == 0) return cudaSuccess;
    const int vec4 = al16(x) && al16(corr) && al16(white) && al16(y) && al16(y_clip);
    return launch_ex(dr_noise_kernel, dim3((unsigned)dr_blocks(total)), dim3(256), 0, st, x, corr, white, seed, step, cfg, y, y_clip, clip,
                     total, vec4);
}

cudaError_t launch_dr_fill(uint64_t seed, uint64_t step, int distribution, float* out, int64_t total, cudaStream_t st) {
    if (total == 0) return cudaSuccess;
    dr_fill_kernel<<<dr_blocks(total), 256, 0, st>>>(seed, step, distribution, out, total);
    return cudaGetLastError();
}

}  // namespace bezk

// ------------------------------------------------------------------------------------------------
// Self-test of Mth<true> (bezk_common.cuh) against the built-in IEEE operators.
//   sqrt: every 2^32 bit pattern.   div: `pairs` Philox-random (a, b) bit patterns, a quarter of them drawn from the
//   2^-70 .. 2^70 exponent window the task math lives in, plus an exhaustive cross of special values (0, -0, denormals, the
//   guard-range edges, FLT_MAX, inf, NaN).  Wherever the fast path reports `!bad` its bits must equal the operator's.
// counts[0] = sqrt mismatches, [1] = div mismatches, [2] = sqrt inputs accepted by the fast path, [3] = div pairs accepted.
// ------------------------------------------------------------------------------------------------
namespace bezk {

__device__ __forceinline__ bool same_bits(float a, float b) {
    return __float_as_uint(a) == __float_as_uint(b) || (a != a && b != b);
}

__global__ void __launch_bounds__(256) selftest_sqrt_kernel(unsigned long long* counts) {
    unsigned long long bad_cnt = 0, ok_cnt = 0;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (1ull << 32); i += stride) {
        const float x = __uint_as_float((uint32_t)i);
        Mth<true> m;
        const float f = m.sqr(x);
        if (!m.bad()) { ++ok_cnt; if (!same_bits(f, sqrtf(x))) ++bad_cnt; }
    }
    if (bad_cnt) atomicAdd(&counts[0], bad_cnt);
    atomicAdd(&counts[2], ok_cnt);
}

__device__ __forceinline__ float special_value(int k) {
    const uint32_t v[] = {0x00000000u, 0x80000000u, 0x00000001u, 0x007FFFFFu, 0x00800000u, 0x21800000u, 0x217FFFFFu, 0x5D800000u,
                          0x5D800001u, 0x3F800000u, 0xBF800000u, 0x3F7FFFFFu, 0x3F800001u, 0x7F7FFFFFu, 0x7F800000u, 0xFF800000u,
                          0x7FC00000u, 0x3C888889u /* ~dt */, 0x40000000u, 0x34000000u, 0x4B800000u, 0x3FFFFFFFu, 0x00FFFFFFu, 0xDD800000u};
    return __uint_as_float(v[k]);
}

__global__ void __launch_bounds__(256) selftest_div_kernel(uint64_t pairs, uint64_t seed, unsigned long long* counts) {
    unsigned long long bad_cnt = 0, ok_cnt = 0;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (uint64_t i = tid; i < pairs / 2; i += stride) {
        const Philox4 r = philox4x32_10((uint32_t)i, (uint32_t)(i >> 32), 0x5E1F7E57u, 0u, (uint32_t)seed, (uint32_t)(seed >> 32));
        uint32_t w[4] = {r.x, r.y, r.z, r.w};
        if ((i & 3) == 0) {              // squeeze the exponents into 2^-70 .. 2^70 so that most pairs take the fast path
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint32_t e = 57u + ((w[k] >> 23) & 0xFFu) % 141u;
                w[k] = (w[k] & 0x807FFFFFu) | (e << 23);
            }
        }
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const float a = __uint_as_float(w[2 * k]), b = __uint_as_float(w[2 * k + 1]);
            Mth<true> m;
            const float f = m.div(a, b);
            if (!m.bad()) { ++ok_cnt; if (!same_bits(f, a / b)) ++bad_cnt; }
        }
    }
    if (tid < 24 * 24) {
        const float a = special_value((int)(tid / 24)), b = special_value((int)(tid % 24));
        Mth<true> m;
        const float f = m.div(a, b);
        if (!m.bad()) { ++ok_cnt; if (!same_bits(f, a / b)) ++bad_cnt; }
    }
    if (bad_cnt) atomicAdd(&counts[1], bad_cnt);
    atomicAdd(&counts[3], ok_cnt);
}

cudaError_t launch_selftest_fastmath(uint64_t pairs, uint64_t seed, unsigned long long* counts, cudaStream_t st) {
    cudaError_t e = cudaMemsetAsync(counts, 0, 4 * sizeof(unsigned long long), st);
    if (e != cudaSuccess) return e;
    selftest_sqrt_kernel<<<148 * 8, 256, 0, st>>>(counts);
    selftest_div_kernel<<<148 * 8, 256, 0, st>>>(pairs, seed, counts);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Episode meters: rl_games' game_rewards / game_lengths (torch_ext.AverageMeter, games_to_track) fed by the per-step partials of
// the fused step with episode accumulators ((T, 3, W): per warp of 32 envs the count of done envs, the sum of their returns and
// of their lengths).  One launch, no host round trip: CTA t reduces step t's 3 x W partials in a fixed order (the same bits every
// run), and the last CTA to finish (ticket) runs the AverageMeter recurrence over the steps in order in one warp:
//   new_mean = sum / count (fp64, rounded to fp32); size = min(count, max_size); old_size = min(max_size - size, current_size)
//   current_size = old_size + size; mean = (mean * old_size + new_mean * size) / current_size    (fp32, rl_games' order)
// No CTA-wide barrier: the warps of a CTA meet through a ticket as well.
// ------------------------------------------------------------------------------------------------
constexpr int EPM_THREADS = 256;
constexpr int EPM_WARPS = EPM_THREADS / 32;

struct EpmScratch {
    double* warp_sums;     // (steps, EPM_WARPS, 3)
    double* step_sums;     // (steps, 3)
    unsigned* tickets;     // (steps + 1,) zeroed: per step (its warps), then the steps
};

__global__ void __launch_bounds__(EPM_THREADS) episode_meter_kernel(const double* __restrict__ partials, int steps, int64_t w,
                                                                    int64_t max_size, EpmScratch sc, float* mean2, int64_t* size2) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int step = blockIdx.x;
    pdl_launch_dependents();
    pdl_wait();
    const double* p = partials + (int64_t)step * 3 * w;
    double acc[3] = {0.0, 0.0, 0.0};
    for (int64_t i = threadIdx.x; i < w; i += EPM_THREADS) {
#pragma unroll
        for (int k = 0; k < 3; ++k) acc[k] += p[k * w + i];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int k = 0; k < 3; ++k) acc[k] += __shfl_down_sync(0xffffffffu, acc[k], o);
    }
    const unsigned full = 0xffffffffu;
    int last = 0;
    if (lane == 0) {
        double* ws = sc.warp_sums + ((int64_t)step * EPM_WARPS + warp) * 3;
#pragma unroll
        for (int k = 0; k < 3; ++k) ws[k] = acc[k];
        __threadfence();
        last = atomicAdd(&sc.tickets[step], 1u) == EPM_WARPS - 1;
    }
    if (!__shfl_sync(full, last, 0)) return;
    // the last warp of this CTA: the step's sums, warp by warp in order
    __threadfence();
    if (lane == 0) {
        const double* wsum = sc.warp_sums + (int64_t)step * EPM_WARPS * 3;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            double v = 0.0;
#pragma unroll
            for (int j = 0; j < EPM_WARPS; ++j) v += __ldcg(wsum + j * 3 + k);
            sc.step_sums[step * 3 + k] = v;
        }
        __threadfence();
        last = atomicAdd(&sc.tickets[steps], 1u) == (unsigned)steps - 1;
    }
    if (!__shfl_sync(full, last, 0)) return;
    // the last step to finish: the recurrence, step by step in order.  Lane j of the warp loads step t0 + j's sums, so the
    // loads of 32 steps are in flight together; every lane then runs the same recurrence on the shuffled values.
    __threadfence();
    float mean[2] = {mean2[0], mean2[1]};
    int64_t cur[2] = {size2[0], size2[1]};     // 0: game_rewards (returns), 1: game_lengths
    for (int t0 = 0; t0 < steps; t0 += 32) {
        double c = 0.0, s[2] = {0.0, 0.0};
        if (t0 + lane < steps) {
            c = __ldcg(sc.step_sums + 3 * (t0 + lane));
            s[0] = __ldcg(sc.step_sums + 3 * (t0 + lane) + 1);
            s[1] = __ldcg(sc.step_sums + 3 * (t0 + lane) + 2);
        }
        const int m = steps - t0 < 32 ? steps - t0 : 32;
        for (int j = 0; j < m; ++j) {
            const double cnt = __shfl_sync(full, c, j);
            const double sum[2] = {__shfl_sync(full, s[0], j), __shfl_sync(full, s[1], j)};
            if (!(cnt > 0.0)) continue;           // AverageMeter.update: size == 0 -> no-op
            const int64_t size = (int64_t)cnt < max_size ? (int64_t)cnt : max_size;
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const float new_mean = (float)(sum[k] / cnt);
                const int64_t old_size = (max_size - size) < cur[k] ? (max_size - size) : cur[k];
                const int64_t size_sum = old_size + size;
                cur[k] = size_sum;
                mean[k] = (mean[k] * (float)old_size + new_mean * (float)size) / (float)size_sum;
            }
        }
    }
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 2; ++k) { mean2[k] = mean[k]; size2[k] = cur[k]; }
    }
}

cudaError_t launch_episode_meter_update(const double* partials, int steps, int64_t n, int64_t games_to_track, float* mean2,
                                        int64_t* size2, cudaStream_t st) {
    if (steps == 0 || n == 0) return cudaSuccess;
    // the sums and tickets live for this launch only: stream-ordered scratch (capturable in a CUDA graph, no host synchronisation)
    const size_t nd = (size_t)steps * (EPM_WARPS + 1) * 3, bytes = nd * sizeof(double) + (size_t)(steps + 1) * sizeof(unsigned);
    void* buf = nullptr;
    cudaError_t e = cudaMallocAsync(&buf, bytes, st);
    if (e != cudaSuccess) return e;
    EpmScratch sc;
    sc.warp_sums = static_cast<double*>(buf);
    sc.step_sums = sc.warp_sums + (size_t)steps * EPM_WARPS * 3;
    sc.tickets = reinterpret_cast<unsigned*>(sc.warp_sums + nd);
    e = cudaMemsetAsync(sc.tickets, 0, (size_t)(steps + 1) * sizeof(unsigned), st);
    if (e == cudaSuccess)
        e = launch_ex(episode_meter_kernel, dim3((unsigned)steps), dim3(EPM_THREADS), 0, st, partials, steps, (n + 31) / 32,
                      games_to_track, sc, mean2, size2);
    const cudaError_t f = cudaFreeAsync(buf, st);
    return e != cudaSuccess ? e : f;
}

// ------------------------------------------------------------------------------------------------
// Player tally: rl_games BasePlayer.run's per-step bookkeeping (RECALLED, v1.1.x)
//   games_played += done_count; sum_rewards += cr[done].sum(); sum_steps += steps[done].sum(); stop once games_played >= games_num
// fed by the same per-step partials.  One warp per step sums the step's 3 x W slots in a fixed order: lane l adds slots
// l, l + 32, ... in order, then a shuffle-down tree (16, 8, 4, 2, 1) -- tests/rl_games_player_oracle.py restates it.  The last
// warp to finish (ticket) goes through the steps in order: a step that starts with games_played >= games_num adds nothing (and
// neither does any step of a later call, since the tally carries games_played), so the result does not depend on how the steps
// are chunked; the step that reaches the cutoff is added whole, as in rl_games.
//   tally (4,) f64 in/out: [games_played, sum_rewards, sum_steps, steps_folded];  per_step (steps, 3) f64 out (optional): each
//   folded step's [count, return sum, length sum], zeros after the cutoff.
// No barrier, no local memory, scratch from stream-ordered allocation: capturable in a CUDA graph.
// ------------------------------------------------------------------------------------------------
constexpr int PT_THREADS = 256;
constexpr int PT_WARPS = PT_THREADS / 32;

__global__ void __launch_bounds__(PT_THREADS) player_tally_kernel(const double* __restrict__ partials, int steps, int64_t w,
                                                                   double games_num, double* step_sums, unsigned* ticket, double* tally,
                                                                   double* per_step) {
    const int lane = threadIdx.x & 31;
    const int step = blockIdx.x * PT_WARPS + (threadIdx.x >> 5);
    const unsigned full = 0xffffffffu;
    pdl_launch_dependents();
    pdl_wait();
    if (step >= steps) return;                  // warp-uniform
    const double* p = partials + (int64_t)step * 3 * w;
    double acc[3] = {0.0, 0.0, 0.0};
    for (int64_t i = lane; i < w; i += 32) {
#pragma unroll
        for (int k = 0; k < 3; ++k) acc[k] += p[k * w + i];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int k = 0; k < 3; ++k) acc[k] += __shfl_down_sync(full, acc[k], o);
    }
    int last = 0;
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 3; ++k) step_sums[(int64_t)step * 3 + k] = acc[k];
        __threadfence();
        last = atomicAdd(ticket, 1u) == (unsigned)steps - 1;
    }
    if (!__shfl_sync(full, last, 0)) return;
    // the last step to finish: the fold, step by step in order.  Lane j loads step t0 + j's sums; every lane runs the same
    // recurrence on the shuffled values and lane j writes step t0 + j's per_step row.
    __threadfence();
    double games = __ldcg(tally), sr = __ldcg(tally + 1), sl = __ldcg(tally + 2), folded = __ldcg(tally + 3);
    for (int t0 = 0; t0 < steps; t0 += 32) {
        double c = 0.0, r = 0.0, l = 0.0;
        if (t0 + lane < steps) {
            c = __ldcg(step_sums + 3 * (t0 + lane));
            r = __ldcg(step_sums + 3 * (t0 + lane) + 1);
            l = __ldcg(step_sums + 3 * (t0 + lane) + 2);
        }
        bool mine = false;                      // this lane's step was folded
        const int m = steps - t0 < 32 ? steps - t0 : 32;
        for (int j = 0; j < m; ++j) {
            const double cj = __shfl_sync(full, c, j), rj = __shfl_sync(full, r, j), lj = __shfl_sync(full, l, j);
            if (games >= games_num) continue;   // the cutoff was reached by an earlier step
            folded += 1.0;
            if (lane == j) mine = true;
            if (cj > 0.0) { games += cj; sr += rj; sl += lj; }
        }
        if (per_step && t0 + lane < steps) {
            double* q = per_step + 3 * (int64_t)(t0 + lane);
            q[0] = mine ? c : 0.0; q[1] = mine ? r : 0.0; q[2] = mine ? l : 0.0;
        }
    }
    if (lane == 0) { tally[0] = games; tally[1] = sr; tally[2] = sl; tally[3] = folded; }
}

cudaError_t launch_player_tally_update(const double* partials, int steps, int64_t n, int64_t games_num, double* tally,
                                       double* per_step, cudaStream_t st) {
    if (steps == 0 || n == 0) return cudaSuccess;
    const size_t bytes = (size_t)steps * 3 * sizeof(double) + sizeof(unsigned);
    void* buf = nullptr;
    cudaError_t e = cudaMallocAsync(&buf, bytes, st);
    if (e != cudaSuccess) return e;
    double* step_sums = static_cast<double*>(buf);
    unsigned* ticket = reinterpret_cast<unsigned*>(step_sums + (size_t)steps * 3);
    e = cudaMemsetAsync(ticket, 0, sizeof(unsigned), st);
    if (e == cudaSuccess)
        e = launch_ex(player_tally_kernel, dim3((unsigned)((steps + PT_WARPS - 1) / PT_WARPS)), dim3(PT_THREADS), 0, st, partials, steps,
                      (n + 31) / 32, (double)games_num, step_sums, ticket, tally, per_step);
    const cudaError_t f = cudaFreeAsync(buf, st);
    return e != cudaSuccess ? e : f;
}

}  // namespace bezk
