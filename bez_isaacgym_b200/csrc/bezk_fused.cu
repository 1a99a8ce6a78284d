// Single-launch statistics kernels for the learner's LAUNCH-BOUND sizes (BASELINE configs[2]: 4096 x 32 rollout, minibatch
// 32 768 x 54 = 7 MB).  At these sizes the 4-5 kernel chains of bezk_learner.cu (pivot copy, moments, finalize, merge, normalise)
// cost 4-5 launch latencies for ~3 us of memory traffic.  Here ONE cooperative kernel does the whole train-mode forward:
//
//   phase 1  every CTA reads its contiguous block of rows ONCE from HBM, keeps it in shared memory, and accumulates pivoted fp64
//            moments (pivot = the old running mean, fixed reduction order) -> per-CTA partials
//   grid sync
//   phase 2  every CTA folds the partials in the same fixed order (so all CTAs hold bit-identical statistics), applies rl_games'
//            parallel-variance merge; CTA 0 writes running_mean / running_var / count back
//   phase 3  every CTA normalises its rows out of shared memory and writes y
//
// => 216 B read + 216 B written per 54-wide sample (the algorithmic minimum; the chain re-reads x), one launch, no host round trip.
// The multi-GPU path cannot use it (the all-reduce sits between phase 1 and phase 2) and keeps the moments -> all-reduce -> merge ->
// normalise chain.  Same arithmetic as rms_merge_kernel / rms_normalize_kernel (IEEE division through Mth).
#include "bezk_common.cuh"
#include "bezk_internal.h"
#include <cooperative_groups.h>
#include <math.h>

namespace cg = cooperative_groups;

namespace bezk {

constexpr int FUSED_THREADS = 256;
constexpr int FUSED_MAX_STAGE_BYTES = 160 * 1024;     // rows of one CTA kept in shared memory

__device__ __forceinline__ int64_t fused_src_row(int64_t r, int64_t slab_rows, int64_t slab_stride) {
    if (slab_stride == slab_rows) return r;
    const uint32_t s = (uint32_t)r / (uint32_t)slab_rows;             // launcher guarantees < 2^32 rows
    return (int64_t)s * slab_stride + ((uint32_t)r - s * (uint32_t)slab_rows);
}

// Fold of the per-CTA partials, fixed order, ALL loads of a chunk in flight at once.  A warp owns columns wid, wid + 8, ...;
// it takes them FOLD_COLS at a time: every lane first issues its (up to FOLD_MAXB / 32) x FOLD_COLS independent L2 loads, then
// adds them in a fixed order and the 32 lane sums go through a fixed shuffle tree.  (A plain loop over the columns costs one L2
// round trip per partial per column -- 40 us for 108 columns x 148 CTAs, measured -- instead of two round trips in total.)
constexpr int FOLD_COLS = 7;
constexpr int FOLD_MAXB = 160;          // grid <= 148 CTAs
__device__ __forceinline__ void fused_fold_all(const double* __restrict__ partials, int nblocks, int ncols, int wid, int lane,
                                               int warps, double* s_tot) {
    constexpr int PER_LANE = FOLD_MAXB / 32;
    for (int j0 = wid; j0 < ncols; j0 += warps * FOLD_COLS) {
        double v[FOLD_COLS][PER_LANE];
#pragma unroll
        for (int k = 0; k < FOLD_COLS; ++k) {
            const int j = j0 + k * warps;
#pragma unroll
            for (int u = 0; u < PER_LANE; ++u) {
                const int b = lane + 32 * u;
                v[k][u] = (j < ncols && b < nblocks) ? __ldcg(partials + (int64_t)b * ncols + j) : 0.0;
            }
        }
#pragma unroll
        for (int k = 0; k < FOLD_COLS; ++k) {
            const int j = j0 + k * warps;
            double t = 0.0;
#pragma unroll
            for (int u = 0; u < PER_LANE; ++u) t += v[k][u];
            t = warp_sum(t);
            if (lane == 0 && j < ncols) s_tot[j] = t;
        }
    }
}

struct FusedRmsArgs {
    const float* x;
    const float* x2;           // advantage mode: the statistics / output are over (x - x2)
    double *running_mean, *running_var, *count;     // RunningMeanStd mode
    double* partials;          // [grid][2c]
    float* y;
    int64_t m;
    int c;
    float eps;
    int64_t slab_rows, slab_stride;
    int rows_per_cta;
    int mode;                  // 0: RunningMeanStd train forward; 1: advantage normalisation (c == 1)
    int normalize;             // mode 1: 0 -> y = x - x2 only
};

template <int VEC>
__global__ void __launch_bounds__(FUSED_THREADS) fused_stats_kernel(const FusedRmsArgs a) {
    extern __shared__ __align__(16) unsigned char fsm[];
    const int c = a.c;
    const int cgs = c / VEC;                                  // column groups
    const int rpi = FUSED_THREADS / cgs;                      // rows per iteration
    double* s_red = reinterpret_cast<double*>(fsm);           // [2][rpi][c], then [2c] totals
    float* s_stat = reinterpret_cast<float*>(s_red + (size_t)2 * rpi * c);      // [2c]: mean.float(), sqrt(var.float() + eps)
    float* s_rows = s_stat + ((2 * c + 3) & ~3);              // [rows_per_cta][c]
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int rsub = tid / cgs, g = tid - rsub * cgs;
    const bool active = rsub < rpi;
    const int64_t r0 = (int64_t)blockIdx.x * a.rows_per_cta;
    const int64_t r1 = (r0 + a.rows_per_cta < a.m) ? r0 + a.rows_per_cta : a.m;
    const int nrows = (int)(r1 > r0 ? r1 - r0 : 0);

    // ---- phase 0: old statistics (read BEFORE the grid sync; CTA 0 overwrites them after it) ----
    double old_mean = 0.0, old_var = 1.0, old_cnt = 0.0;
    if (a.mode == 0 && tid < c) { old_mean = a.running_mean[tid]; old_var = a.running_var[tid]; old_cnt = a.count[0]; }
    double pv[VEC], s[VEC], ss[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k) { s[k] = 0.0; ss[k] = 0.0; pv[k] = (a.mode == 0 && active) ? a.running_mean[g * VEC + k] : 0.0; }

    // ---- phase 1: rows -> shared memory + pivoted moments ----
    if (active) {
        constexpr int U = 8;
        int r = rsub;
        for (; r + (U - 1) * rpi < nrows; r += U * rpi) {
            float v[U][VEC];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int64_t src = fused_src_row(r0 + r + u * rpi, a.slab_rows, a.slab_stride) * c + g * VEC;
                if (VEC == 2) {
                    const float2 t = __ldcs(reinterpret_cast<const float2*>(a.x + src));
                    v[u][0] = t.x; v[u][VEC - 1] = t.y;
                    if (a.x2) { const float2 w = __ldcs(reinterpret_cast<const float2*>(a.x2 + src)); v[u][0] -= w.x; v[u][VEC - 1] -= w.y; }
                } else {
                    v[u][0] = __ldcs(a.x + src);
                    if (a.x2) v[u][0] -= __ldcs(a.x2 + src);
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u)
#pragma unroll
                for (int k = 0; k < VEC; ++k) {
                    s_rows[(size_t)(r + u * rpi) * c + g * VEC + k] = v[u][k];
                    const double d = (double)v[u][k] - pv[k];
                    s[k] += d; ss[k] += d * d;
                }
        }
        for (; r < nrows; r += rpi) {
            const int64_t src = fused_src_row(r0 + r, a.slab_rows, a.slab_stride) * c + g * VEC;
#pragma unroll
            for (int k = 0; k < VEC; ++k) {
                float v = a.x[src + k];
                if (a.x2) v -= a.x2[src + k];
                s_rows[(size_t)r * c + g * VEC + k] = v;
                const double d = (double)v - pv[k];
                s[k] += d; ss[k] += d * d;
            }
        }
#pragma unroll
        for (int k = 0; k < VEC; ++k) {
            s_red[(0 * rpi + rsub) * c + g * VEC + k] = s[k];
            s_red[(1 * rpi + rsub) * c + g * VEC + k] = ss[k];
        }
    }
    __syncthreads();
    for (int j = tid; j < 2 * c; j += FUSED_THREADS) {        // fixed-order fold over the rpi row slots
        const int stat = j / c, col = j - stat * c;
        double acc = 0.0;
        for (int q = 0; q < rpi; ++q) acc += s_red[(stat * rpi + q) * c + col];
        a.partials[(int64_t)blockIdx.x * 2 * c + j] = acc;
    }
    __threadfence();
    cg::this_grid().sync();

    // ---- phase 2: every CTA folds the partials (identical order -> identical statistics), merges ----
    fused_fold_all(a.partials, (int)gridDim.x, 2 * c, wid, lane, FUSED_THREADS / 32, s_red);
    __syncthreads();
    const double B = (double)a.m;
    if (a.mode == 0) {
        if (tid < c) {
            // rl_games running_mean_std.py, training branch (fp64): unbiased batch variance, parallel-variance merge
            const double S = s_red[tid], SS = s_red[c + tid];
            const double mean_b = old_mean + S / B;                       // pivot = old running mean
            const double var_b = (SS - S * S / B) / (B - 1.0);            // NaN for B == 1, like torch.var
            const double delta = mean_b - old_mean;
            const double tot = old_cnt + B;
            const double new_mean = old_mean + delta * B / tot;
            const double new_var = (old_var * old_cnt + var_b * B + delta * delta * old_cnt * B / tot) / tot;
            s_stat[tid] = (float)new_mean;
            s_stat[c + tid] = sqrtf((float)new_var + a.eps);
            if (blockIdx.x == 0) {
                a.running_mean[tid] = new_mean; a.running_var[tid] = new_var;
                if (tid == 0) a.count[0] = tot;
            }
        }
    } else if (tid == 0) {
        // a2c_common.py prepare_dataset: (adv - adv.mean()) / (adv.std() + 1e-8), unbiased std
        const double S = s_red[0], SS = s_red[1];
        const double mu = S / B;
        const double var = (SS - S * mu) / (B - 1.0);
        s_stat[0] = (float)mu;
        s_stat[1] = (float)sqrt(var < 0.0 ? 0.0 : var) + 1e-8f;       // as adv_normalize_kernel: NaN passes, negatives are 0
    }
    __syncthreads();

    // ---- phase 3: normalise this CTA's rows out of shared memory ----
    const int total = nrows * c;
    float* yb = a.y + r0 * c;
    for (int i = tid * VEC; i < total; i += FUSED_THREADS * VEC) {
        float in[VEC], out[VEC];
        int col = i % c;
        const int col0 = col;
#pragma unroll
        for (int k = 0; k < VEC; ++k) in[k] = s_rows[i + k];
        if (a.mode == 0) {
            Mth<true> mq;
#pragma unroll
            for (int k = 0; k < VEC; ++k) { out[k] = clamp_nan(mq.div(in[k] - s_stat[col], s_stat[c + col]), -5.0f, 5.0f); col = (col + 1 == c) ? 0 : col + 1; }
            if (mq.bad()) {
                col = col0;
                for (int k = 0; k < VEC; ++k) { out[k] = clamp_nan((in[k] - s_stat[col]) / s_stat[c + col], -5.0f, 5.0f); col = (col + 1 == c) ? 0 : col + 1; }
            }
        } else {
#pragma unroll
            for (int k = 0; k < VEC; ++k) out[k] = a.normalize ? (in[k] - s_stat[0]) / s_stat[1] : in[k];
        }
        if (VEC == 2) __stcs(reinterpret_cast<float2*>(yb + i), make_float2(out[0], out[VEC - 1]));
        else __stcs(yb + i, out[0]);
    }
}

static inline bool f_aligned8(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 7u) == 0; }

// geometry shared by the eligibility test and the launcher
static bool fused_geometry(int64_t m, int c, int vec, int* grid, int* rows_per_cta, size_t* smem) {
    if (m < 2 || c < 1 || c > 128 || m >= (1LL << 31)) return false;
    // one CTA per SM of the CURRENT device (a cooperative grid must be co-resident): 148 on a full B200
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms < 1)
        return false;
    int g = sms < FOLD_MAXB ? sms : FOLD_MAXB;
    int64_t rpc = (m + g - 1) / g;
    rpc = (rpc + 1) & ~1LL;                                 // even: every CTA's output block stays 8-byte aligned
    if (rpc < 2) rpc = 2;
    g = (int)((m + rpc - 1) / rpc);
    const int rpi = FUSED_THREADS / (c / vec);
    const size_t bytes = (size_t)2 * rpi * c * sizeof(double) + (size_t)((2 * c + 3) & ~3) * sizeof(float) + (size_t)rpc * c * sizeof(float);
    if ((size_t)rpc * c * sizeof(float) > FUSED_MAX_STAGE_BYTES) return false;
    *grid = g; *rows_per_cta = (int)rpc; *smem = bytes;
    return true;
}

bool fused_stats_eligible(int64_t m, int c) {
    int g, r; size_t s;
    return fused_geometry(m, c, (c % 2 == 0) ? 2 : 1, &g, &r, &s);
}

static cudaError_t launch_fused(FusedRmsArgs& a, cudaStream_t st) {
    const bool v2 = (a.c % 2 == 0) && f_aligned8(a.x) && f_aligned8(a.y) && (a.x2 == nullptr || f_aligned8(a.x2));
    int grid, rpc; size_t smem;
    if (!fused_geometry(a.m, a.c, v2 ? 2 : 1, &grid, &rpc, &smem)) return cudaErrorInvalidValue;
    a.rows_per_cta = rpc;
    static SmemOptIn opt1, opt2;
    cudaLaunchConfig_t lc = {};
    lc.gridDim = dim3((unsigned)grid); lc.blockDim = dim3(FUSED_THREADS); lc.dynamicSmemBytes = smem; lc.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;
    attr[0].val.cooperative = 1;
    lc.attrs = attr; lc.numAttrs = 1;
    if (v2) {
        if (cudaError_t e = opt2.ensure(fused_stats_kernel<2>, 200 * 1024)) return e;
        return cudaLaunchKernelEx(&lc, fused_stats_kernel<2>, a);
    }
    if (cudaError_t e = opt1.ensure(fused_stats_kernel<1>, 200 * 1024)) return e;
    return cudaLaunchKernelEx(&lc, fused_stats_kernel<1>, a);
}

cudaError_t launch_rms_train_forward(const float* x, double* running_mean, double* running_var, double* count, float eps, float* y,
                                     double* partials, int64_t m, int c, int64_t slab_rows, int64_t slab_stride, cudaStream_t st) {
    if (slab_rows <= 0 || slab_rows >= m) { slab_rows = m; slab_stride = m; }
    if (m % slab_rows != 0) return cudaErrorInvalidValue;
    FusedRmsArgs a = {};
    a.x = x; a.running_mean = running_mean; a.running_var = running_var; a.count = count; a.partials = partials; a.y = y;
    a.m = m; a.c = c; a.eps = eps; a.slab_rows = slab_rows; a.slab_stride = slab_stride; a.mode = 0;
    return launch_fused(a, st);
}

cudaError_t launch_adv_fused(const float* returns, const float* values, float* adv, double* partials, int normalize, int64_t m,
                             cudaStream_t st) {
    FusedRmsArgs a = {};
    a.x = returns; a.x2 = values; a.partials = partials; a.y = adv; a.m = m; a.c = 1; a.slab_rows = m; a.slab_stride = m;
    a.mode = 1; a.normalize = normalize;
    return launch_fused(a, st);
}

}  // namespace bezk
