// rl_games rollout / learner math for B200 (sm_100a): GAE reverse scan, RunningMeanStd moments /
// merge / normalise, advantage statistics, fused PPO loss forward + backward.
// All HBM-bound streaming or reduction kernels; statistics are accumulated in fp64 with a fixed
// reduction order (thread -> fixed-order shared-memory fold -> per-block partial -> single-block
// finalize), so results are run-to-run deterministic and additive across ranks.
#include "bezk_common.cuh"
#include "bezk_internal.h"
#include <cooperative_groups.h>
#include <math.h>

namespace bezk {

// Slab addressing: a batch of m rows read straight out of time-major rollout storage.  Batch row r lives at source row
// (r / slab_rows) * slab_stride + r % slab_rows of the (already offset) base pointer; slab_rows == m means contiguous.
__device__ __forceinline__ int64_t slab_src_row(int64_t r, int64_t slab_rows, int64_t slab_stride) {
    if (slab_stride == slab_rows) return r;                // contiguous (the launchers pass slab_rows = slab_stride = m): no divide
    if ((uint64_t)(r | slab_rows) >> 32 == 0) {            // 32-bit divide when both fit (always, below 4 G rows)
        const uint32_t s = (uint32_t)r / (uint32_t)slab_rows;
        return (int64_t)s * slab_stride + ((uint32_t)r - s * (uint32_t)slab_rows);
    }
    const int64_t s = r / slab_rows;
    return s * slab_stride + (r - s * slab_rows);
}

// ------------------------------------------------------------------------------------------------
// K6: GAE.  One thread per env keeps (lastgaelam, next value, next non-terminal) in registers and
// walks the horizon backwards; for a fixed t a warp touches 32 consecutive floats of every array.
// rl_games a2c_common.py discount_values:
//   delta = r[t] + gamma * nextvalues * nextnonterminal - v[t]
//   adv[t] = lastgaelam = delta + gamma * tau * nextnonterminal * lastgaelam ;  ret = adv + v
// ------------------------------------------------------------------------------------------------
template <typename DoneT, int UNROLL>
__global__ void __launch_bounds__(256) gae_kernel(const float* __restrict__ rewards, const float* __restrict__ values,
                                                  const DoneT* __restrict__ dones, const float* __restrict__ last_values,
                                                  const DoneT* __restrict__ last_dones, float gamma, float gamma_tau,
                                                  float* __restrict__ advs, float* __restrict__ returns, int horizon, int64_t n) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    float next_v = last_values[e];
    float next_nt = 1.0f - (float)last_dones[e];
    float lam = 0.0f;
    int t = horizon - 1;
    for (; t >= UNROLL - 1; t -= UNROLL) {
        float r[UNROLL], v[UNROLL], d[UNROLL];
#pragma unroll
        for (int k = 0; k < UNROLL; ++k) {               // all loads of the chunk first (memory-level parallelism)
            const int64_t idx = (int64_t)(t - k) * n + e;
            r[k] = ldg_stream(rewards + idx);
            v[k] = ldg_stream(values + idx);
            d[k] = (float)dones[idx];
        }
#pragma unroll
        for (int k = 0; k < UNROLL; ++k) {
            const int64_t idx = (int64_t)(t - k) * n + e;
            const float delta = (r[k] + (gamma * next_v) * next_nt) - v[k];
            lam = delta + ((gamma_tau * next_nt) * lam);
            __stcs(advs + idx, lam);
            __stcs(returns + idx, lam + v[k]);
            next_v = v[k];
            next_nt = 1.0f - d[k];
        }
    }
    for (; t >= 0; --t) {
        const int64_t idx = (int64_t)t * n + e;
        const float r = rewards[idx], v = values[idx], d = (float)dones[idx];
        const float delta = (r + (gamma * next_v) * next_nt) - v;
        lam = delta + ((gamma_tau * next_nt) * lam);
        advs[idx] = lam;
        returns[idx] = lam + v;
        next_v = v;
        next_nt = 1.0f - d;
    }
}

cudaError_t launch_gae(const float* rewards, const float* values, const void* dones, const float* last_values,
                       const void* last_dones, int dones_kind, double gamma, double tau, float* advs, float* returns,
                       int horizon, int64_t n, cudaStream_t st) {
    if (n == 0 || horizon == 0) return cudaSuccess;
    const unsigned blocks = (unsigned)((n + 255) / 256);
    const float g = (float)gamma, gt = (float)(gamma * tau);
    if (dones_kind == 0)
        gae_kernel<uint8_t, 8><<<blocks, 256, 0, st>>>(rewards, values, (const uint8_t*)dones, last_values,
                                                       (const uint8_t*)last_dones, g, gt, advs, returns, horizon, n);
    else
        gae_kernel<float, 8><<<blocks, 256, 0, st>>>(rewards, values, (const float*)dones, last_values,
                                                     (const float*)last_dones, g, gt, advs, returns, horizon, n);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// K4: RunningMeanStd batch moments, pivoted: acc = [m, sum_j (x-p_j), sum_j (x-p_j)^2].
// Block of RMS_THREADS threads covers `rpi = RMS_THREADS / cg` consecutive rows per iteration
// (cg = column groups of VEC floats), so every thread keeps the same column(s) and every warp load
// is a contiguous 128 B * VEC segment.
// ------------------------------------------------------------------------------------------------
constexpr int RMS_THREADS = 256;
constexpr int RMS_MAX_BLOCKS = 148 * 8;
constexpr int RMS_UNROLL = 8;
constexpr int RMS_MAX_C = 256;                  // columns supported by the multi-column kernel

template <int VEC>
__global__ void __launch_bounds__(RMS_THREADS) rms_partials_kernel(const float* __restrict__ x, const double* __restrict__ pivot,
                                                                   double* __restrict__ partials, int64_t m, int c,
                                                                   int64_t slab_rows, int64_t slab_stride) {
    extern __shared__ double s_red[];           // [2][rpi][c]
    const int cg = c / VEC;
    const int rpi = RMS_THREADS / cg;           // rows per iteration (>= 1 because c <= RMS_MAX_C)
    const int tid = threadIdx.x;
    const int rsub = tid / cg, g = tid - rsub * cg;
    const bool active = rsub < rpi;
    double s[VEC], ss[VEC], pv[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k) { s[k] = 0.0; ss[k] = 0.0; pv[k] = (pivot && active) ? pivot[g * VEC + k] : 0.0; }
    if (active) {
        const int64_t row_stride = (int64_t)gridDim.x * rpi;
        int64_t r = (int64_t)blockIdx.x * rpi + rsub;
        // RMS_UNROLL independent loads in flight per thread
        for (; r + (RMS_UNROLL - 1) * row_stride < m; r += RMS_UNROLL * row_stride) {
            float xv[RMS_UNROLL][VEC];
#pragma unroll
            for (int u = 0; u < RMS_UNROLL; ++u) {
                const float* p = x + slab_src_row(r + u * row_stride, slab_rows, slab_stride) * c + g * VEC;
                // volatile asm loads: issued as one batch (the compiler otherwise interleaves load/use and keeps 1-2 in flight)
                if (VEC == 2) asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(xv[u][0]), "=f"(xv[u][VEC - 1]) : "l"(p));
                else xv[u][0] = ldg_stream(p);
            }
            // one opaque statement that "uses" every loaded register: nothing below can be scheduled between the loads
            static_assert(RMS_UNROLL == 8, "fence lists 8 rows");
            if (VEC == 2)
                asm volatile("" : "+f"(xv[0][0]), "+f"(xv[1][0]), "+f"(xv[2][0]), "+f"(xv[3][0]), "+f"(xv[4][0]), "+f"(xv[5][0]),
                                  "+f"(xv[6][0]), "+f"(xv[7][0]), "+f"(xv[0][VEC - 1]), "+f"(xv[1][VEC - 1]), "+f"(xv[2][VEC - 1]),
                                  "+f"(xv[3][VEC - 1]), "+f"(xv[4][VEC - 1]), "+f"(xv[5][VEC - 1]), "+f"(xv[6][VEC - 1]), "+f"(xv[7][VEC - 1]));
            else
                asm volatile("" : "+f"(xv[0][0]), "+f"(xv[1][0]), "+f"(xv[2][0]), "+f"(xv[3][0]), "+f"(xv[4][0]), "+f"(xv[5][0]),
                                  "+f"(xv[6][0]), "+f"(xv[7][0]));
#pragma unroll
            for (int u = 0; u < RMS_UNROLL; ++u)
#pragma unroll
                for (int k = 0; k < VEC; ++k) { const double d = (double)xv[u][k] - pv[k]; s[k] += d; ss[k] += d * d; }
        }
        for (; r < m; r += row_stride) {
            const float* p = x + slab_src_row(r, slab_rows, slab_stride) * c + g * VEC;
#pragma unroll
            for (int k = 0; k < VEC; ++k) { const double d = (double)p[k] - pv[k]; s[k] += d; ss[k] += d * d; }
        }
#pragma unroll
        for (int k = 0; k < VEC; ++k) {
            s_red[(0 * rpi + rsub) * c + g * VEC + k] = s[k];
            s_red[(1 * rpi + rsub) * c + g * VEC + k] = ss[k];
        }
    }
    __syncthreads();
    for (int j = tid; j < 2 * c; j += RMS_THREADS) {        // fixed-order fold over the rpi row slots
        const int stat = j / c, col = j - stat * c;
        double acc = 0.0;
        for (int q = 0; q < rpi; ++q) acc += s_red[(stat * rpi + q) * c + col];
        partials[(int64_t)blockIdx.x * 2 * c + j] = acc;
    }
}

// TMA variant of the multi-column moments kernel (used when x is 16-byte aligned and c*4*2 is a multiple of 16, i.e.
// always for the 54-wide observations).  The per-thread-load version above keeps only 1-2 loads per thread in flight
// (ptxas interleaves load/use whatever the source order; measured 2.6 TB/s); here persistent CTAs stream contiguous tiles
// of RMS_TR rows through a 4-stage ring of cp.async.bulk copies, so ~3 tiles (41 KB for c = 54) per CTA are always in
// flight, and the fp64 accumulation reads shared memory (consecutive threads = consecutive columns, conflict-free).
constexpr int RMS_TR = 64;                      // rows per tile
constexpr int RMS_STAGES = 4;

template <bool SLABS>       // the contiguous instantiation carries no slab arithmetic (32 registers; with it: 44, and 7 % slower)
__global__ void __launch_bounds__(RMS_THREADS) rms_partials_tma_kernel(const float* __restrict__ x, const double* __restrict__ pivot,
                                                                       double* __restrict__ partials, int64_t m, int c,
                                                                       int64_t slab_rows, int64_t slab_stride,
                                                                       int64_t x_batch_elems) {
    // blockIdx.y = batch (bezk_rms_moments_slabs_batched): its own rows and its own gridDim.x partial rows
    x += (int64_t)blockIdx.y * x_batch_elems;
    partials += (int64_t)blockIdx.y * gridDim.x * 2 * c;
    extern __shared__ __align__(128) unsigned char rms_smem[];
    __shared__ __align__(8) uint64_t s_full[RMS_STAGES];
    float* s_tile = reinterpret_cast<float*>(rms_smem);                       // [RMS_STAGES][RMS_TR * c]
    double* s_red = reinterpret_cast<double*>(rms_smem);                      // reused after the loop: [2][rpb][c]
    const int tid = threadIdx.x;
    const int rpb = RMS_THREADS / c;                                          // row groups per block (>= 1)
    const int rg = tid / c, col = tid - rg * c;
    const bool active = rg < rpb;
    const int64_t ntiles = (m + RMS_TR - 1) / RMS_TR;
    const int tile_floats = RMS_TR * c;
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < RMS_STAGES; ++s) mbar_init(&s_full[s], 1);
        fence_mbar_init();
    }
    pdl_wait();                                          // the prologue above overlaps the previous kernel's tail
    pdl_launch_dependents();
    const double pv = (pivot && active) ? pivot[col] : 0.0;
    __syncthreads();

    auto issue = [&](int64_t tile, int stage) {          // thread 0 only
        const int64_t r0 = tile * RMS_TR;
        const int64_t rows = (m - r0) < (int64_t)RMS_TR ? (m - r0) : (int64_t)RMS_TR;
        const uint32_t bytes = (uint32_t)(rows * c * 4);
        mbar_arrive_expect_tx(&s_full[stage], bytes);
        // slab mode: slab_rows is a multiple of RMS_TR (checked by the launcher), so a tile never straddles two slabs
        const int64_t src = SLABS ? slab_src_row(r0, slab_rows, slab_stride) : r0;
        bulk_g2s(s_tile + (size_t)stage * tile_floats, x + src * c, bytes, &s_full[stage]);
    };
    // this CTA's tiles: blockIdx.x, +gridDim.x, ...
    int64_t my_tiles = 0;
    if ((int64_t)blockIdx.x < ntiles) my_tiles = (ntiles - 1 - blockIdx.x) / gridDim.x + 1;
    if (tid == 0) {
        for (int k = 0; k < RMS_STAGES - 1 && k < my_tiles; ++k) issue((int64_t)blockIdx.x + (int64_t)k * gridDim.x, k);
    }
    double s = 0.0, ss = 0.0;
    for (int64_t k = 0; k < my_tiles; ++k) {
        const int stage = (int)(k % RMS_STAGES);
        const uint32_t parity = (uint32_t)((k / RMS_STAGES) & 1);
        // refill the stage that was consumed in the previous iteration (all threads passed the barrier below)
        if (tid == 0 && k + RMS_STAGES - 1 < my_tiles)
            issue((int64_t)blockIdx.x + (k + RMS_STAGES - 1) * gridDim.x, (int)((k + RMS_STAGES - 1) % RMS_STAGES));
        mbar_wait(&s_full[stage], parity);
        const int64_t r0 = ((int64_t)blockIdx.x + k * gridDim.x) * RMS_TR;
        const int rows = (int)((m - r0) < (int64_t)RMS_TR ? (m - r0) : (int64_t)RMS_TR);
        if (active) {
            const float* t = s_tile + (size_t)stage * tile_floats + col;
            for (int r = rg; r < rows; r += rpb) {
                const double d = (double)t[r * c] - pv;
                s += d;
                ss += d * d;
            }
        }
        __syncthreads();                                   // stage fully consumed before thread 0 may refill it
    }
    // fixed-order fold over the row groups (shared memory is free now)
    if (active) { s_red[(0 * rpb + rg) * c + col] = s; s_red[(1 * rpb + rg) * c + col] = ss; }
    __syncthreads();
    for (int j = tid; j < 2 * c; j += RMS_THREADS) {
        const int stat = j / c, cc = j - stat * c;
        double acc = 0.0;
        for (int q = 0; q < rpb; ++q) acc += s_red[(stat * rpb + q) * c + cc];
        partials[(int64_t)blockIdx.x * 2 * c + j] = acc;
    }
}

// flat (c == 1) moments of x, or of (a - b) when b != nullptr (advantage = returns - values in fp32)
__global__ void __launch_bounds__(RMS_THREADS) flat_partials_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                                    const double* __restrict__ pivot, double* __restrict__ partials,
                                                                    int64_t m, int vec4, int64_t slab_rows, int64_t slab_stride) {
    __shared__ double s_w[2][RMS_THREADS / 32];
    const double pv = pivot ? pivot[0] : 0.0;
    double s = 0.0, ss = 0.0;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nvec = vec4 ? (m >> 2) : 0;
    const bool slabs = slab_rows < m;                     // vec4 then implies slab_rows % 4 == 0 and slab_stride % 4 == 0
    for (int64_t i = tid; i < nvec; i += stride) {
        const int64_t si = slabs ? (slab_src_row(i * 4, slab_rows, slab_stride) >> 2) : i;
        float4 t = ldg_stream4(reinterpret_cast<const float4*>(a) + si);
        if (b) { const float4 u = ldg_stream4(reinterpret_cast<const float4*>(b) + si); t.x -= u.x; t.y -= u.y; t.z -= u.z; t.w -= u.w; }
        const double d0 = (double)t.x - pv, d1 = (double)t.y - pv, d2 = (double)t.z - pv, d3 = (double)t.w - pv;
        s += (d0 + d1) + (d2 + d3);
        ss += (d0 * d0 + d1 * d1) + (d2 * d2 + d3 * d3);
    }
    for (int64_t i = nvec * 4 + tid; i < m; i += stride) {
        const int64_t si = slabs ? slab_src_row(i, slab_rows, slab_stride) : i;
        float t = a[si];
        if (b) t -= b[si];
        const double d = (double)t - pv;
        s += d; ss += d * d;
    }
    s = warp_sum(s); ss = warp_sum(ss);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) { s_w[0][wid] = s; s_w[1][wid] = ss; }
    __syncthreads();
    if (threadIdx.x < 2) {
        double acc = 0.0;
        for (int q = 0; q < RMS_THREADS / 32; ++q) acc += s_w[threadIdx.x][q];
        partials[(int64_t)blockIdx.x * 2 + threadIdx.x] = acc;
    }
}

// Deterministic fold of per-block partials: ONE WARP per output column j.  Lane l sums blocks l, l+32, ... with up to 8
// independent loads in flight, then the 32 lane sums are folded by a fixed xor-shuffle tree.  (A single thread walking
// 592..8192 partials serially costs 40..600 us of pure L2 latency -- measured, profiles/r01_kernels.md.)
__device__ __forceinline__ double fold_column(const double* __restrict__ partials, int nblocks, int ncols, int j, int lane) {
    double t = 0.0;
    int b = lane;
    for (; b + 7 * 32 < nblocks; b += 8 * 32) {
        double v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = partials[(int64_t)(b + u * 32) * ncols + j];
#pragma unroll
        for (int u = 0; u < 8; ++u) t += v[u];
    }
    for (; b < nblocks; b += 32) t += partials[(int64_t)b * ncols + j];
    return warp_sum(t);
}

// acc = [m, sums(c), sumsqs(c)]
// With snap_mean != nullptr the OLD running statistics are appended: acc[1+2c ..] = [mean(c), var(c), count] -- the snapshot
// rms_merge_normalize_kernel merges from, so that it never reads running_* while its CTA 0 overwrites them.
__global__ void __launch_bounds__(256) moments_finalize_kernel(const double* __restrict__ partials, int nblocks, int c, int64_t m,
                                                               double* __restrict__ acc, const double* __restrict__ snap_mean = nullptr,
                                                               const double* __restrict__ snap_var = nullptr,
                                                               const double* __restrict__ snap_count = nullptr) {
    pdl_wait();                 // programmatic dependent launch: everything below may read the previous kernel's output
    pdl_launch_dependents();
    // blockIdx.y = batch: its nblocks partial rows, its own accumulator row
    partials += (int64_t)blockIdx.y * nblocks * 2 * c;
    acc += (int64_t)blockIdx.y * (1 + 2 * c);
    const int lane = threadIdx.x & 31;
    const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (snap_mean && blockIdx.x == 0) {
        for (int k = threadIdx.x; k < c; k += blockDim.x) { acc[1 + 2 * c + k] = snap_mean[k]; acc[1 + 3 * c + k] = snap_var[k]; }
        if (threadIdx.x == 0) acc[1 + 4 * c] = snap_count[0];
    }
    if (j == 0 && lane == 0) acc[0] = (double)m;
    if (j >= 2 * c) return;
    const double t = fold_column(partials, nblocks, 2 * c, j, lane);
    if (lane == 0) acc[1 + j] = t;
}

// K4b: merge (reference running_mean_std.py training branch, fp64):
//   batch mean = p + S/B, batch var (unbiased) = (SS - S*S/B)/(B-1)
//   delta = mean_b - mean; tot = count + B; new_mean = mean + delta*B/tot
//   M2 = var*count + var_b*B + delta^2*count*B/tot ; new_var = M2/tot ; count = tot
__global__ void rms_merge_kernel(const double* __restrict__ acc, const double* __restrict__ pivot, double* running_mean,
                                 double* running_var, double* count, int c) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const double B = acc[0];
    const double cnt = count[0];
    const double tot = cnt + B;
    if (j < c && B > 0.0) {
        const double p = pivot ? pivot[j] : 0.0;
        const double S = acc[1 + j], SS = acc[1 + c + j];
        const double mean_b = p + S / B;
        const double var_b = (SS - S * S / B) / (B - 1.0);          // NaN for B == 1, like torch.var
        const double mean = running_mean[j], var = running_var[j];
        const double delta = mean_b - mean;
        running_mean[j] = mean + delta * B / tot;
        running_var[j] = (var * cnt + var_b * B + delta * delta * cnt * B / tot) / tot;
    }
    __syncthreads();
    // count is read by every thread of every block above; a single trailing kernel-ordered write
    // would race across blocks, so the launcher uses ONE block (c <= 1024).
    if (j == 0 && B > 0.0) count[0] = tot;
}

// K4c: a whole SEQUENCE of merges in one launch.  The obs normaliser is updated with the same few minibatches again and again
// (mini_epochs x minibatches per epoch, rl_games calc_gradients) and its batch moments do not depend on the policy, so they are
// computed ONCE per distinct minibatch (acc rows, all with the pivot taken at plan time) and this kernel replays the reference's
// update `order[u]`, u = 0 .. nu-1, writing the statistics AFTER update u to seq[u] = [mean(c), var(c)] -- what the u-th train
// forward normalises with -- and the final state back to running_*.  One thread per column, the updates in order: the same
// arithmetic as nu calls of rms_merge_kernel (only the pivot of the moments differs, at fp64 rounding level).
__global__ void rms_merge_sequence_kernel(const double* __restrict__ acc, const int32_t* __restrict__ order, int nu,
                                          const double* __restrict__ pivot, double* running_mean, double* running_var, double* count,
                                          double* __restrict__ seq, int c) {
    const int j = threadIdx.x;
    double cnt = count[0];
    const double p = (pivot && j < c) ? pivot[j] : 0.0;
    double mean = j < c ? running_mean[j] : 0.0, var = j < c ? running_var[j] : 1.0;
    for (int u = 0; u < nu; ++u) {
        const double* a = acc + (int64_t)order[u] * (1 + 2 * c);
        const double B = a[0];
        if (B > 0.0) {
            const double tot = cnt + B;
            if (j < c) {
                const double S = a[1 + j], SS = a[1 + c + j];
                const double mean_b = p + S / B;
                const double var_b = (SS - S * S / B) / (B - 1.0);          // NaN for B == 1, like torch.var
                const double delta = mean_b - mean;
                const double new_mean = mean + delta * B / tot;
                var = (var * cnt + var_b * B + delta * delta * cnt * B / tot) / tot;
                mean = new_mean;
            }
            cnt = tot;
        }
        if (j < c) { seq[((int64_t)u * 2 + 0) * c + j] = mean; seq[((int64_t)u * 2 + 1) * c + j] = var; }
    }
    __syncthreads();                    // every thread has read count[0]
    if (j < c) { running_mean[j] = mean; running_var[j] = var; }
    if (j == 0) count[0] = cnt;
}

// K5: normalise / un-normalise
template <bool SLABS>
__global__ void __launch_bounds__(256, 8) rms_normalize_kernel(const float* __restrict__ x, const double* __restrict__ running_mean,
                                                            const double* __restrict__ running_var, float eps, int unnorm,
                                                            float* __restrict__ y, int64_t total, int c, int vec4,
                                                            int64_t slab_src_elems, int64_t x_batch_elems = 0,
                                                            int64_t y_batch_elems = 0, int64_t stat_batch = 0) {
    // blockIdx.y = slab: `total` elements of THIS slab, read from x + blockIdx.y * slab_src_elems, written to
    // y + blockIdx.y * total (one slab = the whole array in the contiguous case)
    // blockIdx.z = batch (bezk_rms_normalize_slabs_batched): several minibatches, each with its OWN statistics, in one launch
    if (SLABS) {
        x += (int64_t)blockIdx.z * x_batch_elems + (int64_t)blockIdx.y * slab_src_elems;
        y += (int64_t)blockIdx.z * y_batch_elems + (int64_t)blockIdx.y * total;
        running_mean += (int64_t)blockIdx.z * stat_batch;
        running_var += (int64_t)blockIdx.z * stat_batch;
    }
    extern __shared__ float s_stat[];       // [2][c]: mean.float(), sqrt(var.float() + eps)
    for (int j = threadIdx.x; j < c; j += blockDim.x) {
        s_stat[j] = (float)running_mean[j];
        s_stat[c + j] = sqrtf((float)running_var[j] + eps);
    }
    __syncthreads();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nvec = vec4 ? (total >> 2) : 0;
    for (int64_t i = tid; i < nvec; i += stride) {
        const float4 t = ldg_stream4(reinterpret_cast<const float4*>(x) + i);
        const float in[4] = {t.x, t.y, t.z, t.w};
        float out[4];
        const int col0 = (int)((i * 4) % c);
        int col = col0;
        Mth<true> mq;                              // exact division without a branch per element (bezk_common.cuh)
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float mean = s_stat[col], den = s_stat[c + col];
            out[k] = unnorm ? (den * clamp_nan(in[k], -5.0f, 5.0f) + mean) : clamp_nan(mq.div(in[k] - mean, den), -5.0f, 5.0f);
            col = (col + 1 == c) ? 0 : col + 1;
        }
        if (!unnorm && mq.bad()) {                 // an operand outside the fast sequence's range: plain operator
            col = col0;
            for (int k = 0; k < 4; ++k) {
                out[k] = clamp_nan((in[k] - s_stat[col]) / s_stat[c + col], -5.0f, 5.0f);
                col = (col + 1 == c) ? 0 : col + 1;
            }
        }
        __stcs(reinterpret_cast<float4*>(y) + i, make_float4(out[0], out[1], out[2], out[3]));
    }
    for (int64_t i = nvec * 4 + tid; i < total; i += stride) {
        const int col = (int)(i % c);
        const float mean = s_stat[col], den = s_stat[c + col];
        y[i] = unnorm ? (den * clamp_nan(x[i], -5.0f, 5.0f) + mean) : clamp_nan((x[i] - mean) / den, -5.0f, 5.0f);
    }
}

// K4b + K5 in one launch: every CTA merges acc_ext = [B, S(c), SS(c), old mean(c), old var(c), old count] (the batch moments,
// possibly all-reduced over ranks, and the snapshot of the running statistics moments_finalize_kernel appended) with the
// reference's parallel-variance update -- identical arithmetic in every CTA -- then normalises its share of x with the UPDATED
// statistics; CTA (0,0) writes running_mean / running_var / count back.  Nothing reads running_* here, so there is no race.
template <bool SLABS>
__global__ void __launch_bounds__(256, 8) rms_merge_normalize_kernel(const float* __restrict__ x, const double* __restrict__ acc,
                                                                  double* running_mean, double* running_var, double* count, float eps,
                                                                  float* __restrict__ y, int64_t total, int c, int vec4,
                                                                  int64_t slab_src_elems) {
    pdl_wait();                 // programmatic dependent launch: everything below may read the previous kernel's output
    pdl_launch_dependents();
    if (SLABS) {
        x += (int64_t)blockIdx.y * slab_src_elems;
        y += (int64_t)blockIdx.y * total;
    }
    extern __shared__ float s_stat[];       // [2][c]: mean.float(), sqrt(var.float() + eps)
    const double B = acc[0], cnt = acc[1 + 4 * c], tot = cnt + B;
    const bool writer = (blockIdx.x == 0 && blockIdx.y == 0);
    for (int j = threadIdx.x; j < c; j += blockDim.x) {
        const double S = acc[1 + j], SS = acc[1 + c + j], mean = acc[1 + 2 * c + j], var = acc[1 + 3 * c + j];
        double new_mean = mean, new_var = var;
        if (B > 0.0) {
            const double mean_b = mean + S / B;                         // pivot = the old running mean
            const double var_b = (SS - S * S / B) / (B - 1.0);          // NaN for B == 1, like torch.var
            const double delta = mean_b - mean;
            new_mean = mean + delta * B / tot;
            new_var = (var * cnt + var_b * B + delta * delta * cnt * B / tot) / tot;
        }
        s_stat[j] = (float)new_mean;
        s_stat[c + j] = sqrtf((float)new_var + eps);
        if (writer) { running_mean[j] = new_mean; running_var[j] = new_var; }
    }
    if (writer && threadIdx.x == 0 && B > 0.0) count[0] = tot;
    __syncthreads();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nvec = vec4 ? (total >> 2) : 0;
    for (int64_t i = tid; i < nvec; i += stride) {
        const float4 t = ldg_stream4(reinterpret_cast<const float4*>(x) + i);
        const float in[4] = {t.x, t.y, t.z, t.w};
        float out[4];
        const int col0 = (int)((i * 4) % c);
        int col = col0;
        Mth<true> mq;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            out[k] = clamp_nan(mq.div(in[k] - s_stat[col], s_stat[c + col]), -5.0f, 5.0f);
            col = (col + 1 == c) ? 0 : col + 1;
        }
        if (mq.bad()) {
            col = col0;
            for (int k = 0; k < 4; ++k) {
                out[k] = clamp_nan((in[k] - s_stat[col]) / s_stat[c + col], -5.0f, 5.0f);
                col = (col + 1 == c) ? 0 : col + 1;
            }
        }
        __stcs(reinterpret_cast<float4*>(y) + i, make_float4(out[0], out[1], out[2], out[3]));
    }
    for (int64_t i = nvec * 4 + tid; i < total; i += stride) {
        const int col = (int)(i % c);
        y[i] = clamp_nan((x[i] - s_stat[col]) / s_stat[c + col], -5.0f, 5.0f);
    }
}

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
static inline bool aligned8(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 7u) == 0; }

static inline int stream_blocks(int64_t work_items, int threads, int per_sm) {
    int64_t b = (work_items + threads - 1) / threads;
    if (b < 1) b = 1;
    const int64_t cap = 148LL * per_sm;
    return (int)(b > cap ? cap : b);
}

// per-block partials of the largest grid + room for one (1 + 2c) accumulator and a c-wide pivot (bezk_rms_train_forward's chain)
int64_t rms_scratch_doubles(int c) { const int64_t cc = c > 0 ? c : 1; return (int64_t)RMS_MAX_BLOCKS * 2 * cc + (2 + 4 * cc) + 4; }

cudaError_t launch_rms_moments(const float* x, const double* pivot, double* acc, double* partials, int64_t m, int c,
                               int64_t slab_rows, int64_t slab_stride, cudaStream_t st, const double* snap_var,
                               const double* snap_count) {
    // snap_var != nullptr: acc is the EXTENDED accumulator (2 + 4c doubles) and also receives [pivot (= old mean), var, count]
    const double* snap_mean = snap_var ? pivot : nullptr;
    int nblocks;
    if (slab_rows <= 0 || slab_rows >= m) { slab_rows = m; slab_stride = m; }
    if (m % slab_rows != 0) return cudaErrorInvalidValue;
    const bool slabs = slab_rows < m;
    if (c == 1) {
        const int vec4 = aligned16(x) && (!slabs || (slab_rows % 4 == 0 && slab_stride % 4 == 0));
        nblocks = stream_blocks(vec4 ? m / 4 : m, RMS_THREADS, 4);
        flat_partials_kernel<<<nblocks, RMS_THREADS, 0, st>>>(x, nullptr, pivot, partials, m, vec4, slab_rows, slab_stride);
    } else {
        if (c > RMS_MAX_C) return cudaErrorInvalidValue;
        // TMA path: every tile start (64 rows) and every tile size must be a multiple of 16 bytes
        const bool tma_ok = aligned16(x) && ((RMS_TR * c * 4) % 16 == 0) && (((m % RMS_TR) * c * 4) % 16 == 0) && m >= 4 * RMS_TR &&
                            (!slabs || (slab_rows % RMS_TR == 0 && (slab_stride * c * 4) % 16 == 0)) &&
                            (size_t)RMS_STAGES * RMS_TR * c * sizeof(float) <= 220 * 1024;      // wider rows: the plain-load kernel
        if (tma_ok) {
            const int64_t ntiles = (m + RMS_TR - 1) / RMS_TR;
            size_t smem = (size_t)RMS_STAGES * RMS_TR * c * sizeof(float);
            const size_t red = (size_t)2 * (RMS_THREADS / c) * c * sizeof(double);     // fold buffer aliases the ring
            if (red > smem) smem = red;
            static SmemOptIn opt_plain, opt_slabs;       // opt in to the cap once per device; the launch passes the real size
            if (cudaError_t e2 = opt_plain.ensure(rms_partials_tma_kernel<false>, 220 * 1024)) return e2;
            if (cudaError_t e2 = opt_slabs.ensure(rms_partials_tma_kernel<true>, 220 * 1024)) return e2;
            int per_sm = (int)((220 * 1024) / (smem + 1024));
            if (per_sm > 8) per_sm = 8;
            if (per_sm < 1) per_sm = 1;
            int64_t cap = 148LL * per_sm;
            if (cap > RMS_MAX_BLOCKS) cap = RMS_MAX_BLOCKS;
            nblocks = (int)(ntiles < cap ? ntiles : cap);
            cudaError_t err = slabs ? launch_pdl(learner_pdl(), rms_partials_tma_kernel<true>, dim3((unsigned)nblocks), dim3(RMS_THREADS), smem, st, x, pivot,
                                                partials, m, c, slab_rows, slab_stride, (int64_t)0)
                                    : launch_pdl(learner_pdl(), rms_partials_tma_kernel<false>, dim3((unsigned)nblocks), dim3(RMS_THREADS), smem, st, x, pivot,
                                                partials, m, c, m, m, (int64_t)0);
            if (err != cudaSuccess) return err;
            return launch_pdl(learner_pdl(), moments_finalize_kernel, dim3((unsigned)((2 * c + 7) / 8)), dim3(256), 0, st, partials, nblocks, c, m, acc,
                             snap_mean, snap_var, snap_count);
        }
        const bool v2 = (c % 2 == 0) && aligned8(x);      // rows start at multiples of c floats: even c keeps 8-byte alignment in slab mode too
        const int cg = v2 ? c / 2 : c;
        const int rpi = RMS_THREADS / cg;
        int64_t b = (m + rpi - 1) / rpi;
        b = (b + RMS_UNROLL - 1) / RMS_UNROLL;         // >= RMS_UNROLL row slots per thread where possible
        if (b < 1) b = 1;
        nblocks = (int)(b > RMS_MAX_BLOCKS ? RMS_MAX_BLOCKS : b);
        const size_t smem = (size_t)2 * rpi * c * sizeof(double);
        if (v2) rms_partials_kernel<2><<<nblocks, RMS_THREADS, smem, st>>>(x, pivot, partials, m, c, slab_rows, slab_stride);
        else rms_partials_kernel<1><<<nblocks, RMS_THREADS, smem, st>>>(x, pivot, partials, m, c, slab_rows, slab_stride);
    }
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return err;
    return launch_pdl(learner_pdl(), moments_finalize_kernel, dim3((unsigned)((2 * c + 7) / 8)), dim3(256), 0, st, partials, nblocks, c, m, acc, snap_mean,
                     snap_var, snap_count);
}

// The moments of n_batches equally spaced minibatches in ONE pair of launches (partials + fold, blockIdx.y = batch): batch b is
// the slab view based at x + b * x_batch_rows * c; acc (n_batches, 1 + 2c).  Only the TMA path is batched, and only while every
// batch gets at least one of the RMS_MAX_BLOCKS partial rows; anything else falls back to one launch_rms_moments per batch.
cudaError_t launch_rms_moments_batched(const float* x, const double* pivot, double* acc, double* partials, int64_t m, int c,
                                       int64_t slab_rows, int64_t slab_stride, int64_t x_batch_rows, int n_batches, cudaStream_t st) {
    if (n_batches <= 0) return cudaSuccess;
    if (slab_rows <= 0 || slab_rows >= m) { slab_rows = m; slab_stride = m; }
    if (m % slab_rows != 0) return cudaErrorInvalidValue;
    const bool slabs = slab_rows < m;
    const bool tma_ok = c > 1 && c <= RMS_MAX_C && n_batches <= RMS_MAX_BLOCKS && aligned16(x) && ((RMS_TR * c * 4) % 16 == 0) &&
                        (((m % RMS_TR) * c * 4) % 16 == 0) && m >= 4 * RMS_TR && ((x_batch_rows * c * 4) % 16 == 0) &&
                        (!slabs || (slab_rows % RMS_TR == 0 && (slab_stride * c * 4) % 16 == 0)) &&
                        (size_t)RMS_STAGES * RMS_TR * c * sizeof(float) <= 220 * 1024;
    if (!tma_ok || n_batches == 1) {
        for (int b = 0; b < n_batches; ++b)
            if (cudaError_t e = launch_rms_moments(x + (int64_t)b * x_batch_rows * c, pivot, acc + (int64_t)b * (1 + 2 * c), partials, m, c,
                                                   slab_rows, slab_stride, st, nullptr, nullptr))
                return e;
        return cudaSuccess;
    }
    const int64_t ntiles = (m + RMS_TR - 1) / RMS_TR;
    size_t smem = (size_t)RMS_STAGES * RMS_TR * c * sizeof(float);
    const size_t red = (size_t)2 * (RMS_THREADS / c) * c * sizeof(double);
    if (red > smem) smem = red;
    static SmemOptIn opt_plain, opt_slabs;
    if (cudaError_t e2 = opt_plain.ensure(rms_partials_tma_kernel<false>, 220 * 1024)) return e2;
    if (cudaError_t e2 = opt_slabs.ensure(rms_partials_tma_kernel<true>, 220 * 1024)) return e2;
    int per_sm = (int)((220 * 1024) / (smem + 1024));
    if (per_sm > 8) per_sm = 8;
    if (per_sm < 1) per_sm = 1;
    int64_t cap = 148LL * per_sm;
    if (cap > RMS_MAX_BLOCKS) cap = RMS_MAX_BLOCKS;
    int64_t per_batch = cap / n_batches;                 // the batches share the resident CTAs (and the partials scratch)
    if (per_batch < 1) per_batch = 1;                    // n_batches <= RMS_MAX_BLOCKS above: the partials still fit
    const int nblocks = (int)(ntiles < per_batch ? ntiles : per_batch);
    const dim3 grid((unsigned)nblocks, (unsigned)n_batches);
    cudaError_t err = slabs ? launch_pdl(learner_pdl(), rms_partials_tma_kernel<true>, grid, dim3(RMS_THREADS), smem, st, x, pivot, partials, m, c,
                                        slab_rows, slab_stride, (int64_t)(x_batch_rows * c))
                            : launch_pdl(learner_pdl(), rms_partials_tma_kernel<false>, grid, dim3(RMS_THREADS), smem, st, x, pivot, partials, m, c,
                                        m, m, (int64_t)(x_batch_rows * c));
    if (err != cudaSuccess) return err;
    return launch_pdl(learner_pdl(), moments_finalize_kernel, dim3((unsigned)((2 * c + 7) / 8), (unsigned)n_batches), dim3(256), 0, st,
                      (const double*)partials, nblocks, c, m, acc, (const double*)nullptr, (const double*)nullptr, (const double*)nullptr);
}

cudaError_t launch_rms_merge_normalize(const float* x, const double* acc_ext, double* running_mean, double* running_var, double* count,
                                       float eps, float* y, int64_t m, int c, int64_t slab_rows, int64_t slab_stride, cudaStream_t st) {
    if (m * c == 0) return cudaSuccess;
    if (slab_rows <= 0 || slab_rows >= m) { slab_rows = m; slab_stride = m; }
    if (m % slab_rows != 0) return cudaErrorInvalidValue;
    const int64_t nslabs = m / slab_rows;
    if (nslabs > 65535) return cudaErrorInvalidValue;
    const int64_t total = slab_rows * c;
    const int vec4 = aligned16(x) && aligned16(y) && (nslabs == 1 || (total % 4 == 0 && (slab_stride * c) % 4 == 0));
    int blocks = stream_blocks(vec4 ? total / 4 : total, 256, 8);
    const int per_slab_cap = (int)((148 * 8 + nslabs - 1) / nslabs);
    if (blocks > per_slab_cap) blocks = per_slab_cap;
    if (nslabs > 1)
        return launch_pdl(learner_pdl(), rms_merge_normalize_kernel<true>, dim3((unsigned)blocks, (unsigned)nslabs), dim3(256), 2 * c * sizeof(float), st, x,
                         acc_ext, running_mean, running_var, count, eps, y, total, c, vec4, slab_stride * c);
    return launch_pdl(learner_pdl(), rms_merge_normalize_kernel<false>, dim3((unsigned)blocks), dim3(256), 2 * c * sizeof(float), st, x, acc_ext, running_mean,
                     running_var, count, eps, y, total, c, vec4, (int64_t)0);
}

cudaError_t launch_rms_merge(const double* acc, const double* pivot, double* running_mean, double* running_var,
                             double* count, int c, cudaStream_t st) {
    if (c > 1024) return cudaErrorInvalidValue;
    rms_merge_kernel<<<1, ((c + 31) / 32) * 32, 0, st>>>(acc, pivot, running_mean, running_var, count, c);
    return cudaGetLastError();
}

cudaError_t launch_rms_merge_sequence(const double* acc, const int32_t* order, int nu, const double* pivot, double* running_mean,
                                      double* running_var, double* count, double* seq, int c, cudaStream_t st) {
    if (c > 1024) return cudaErrorInvalidValue;
    if (nu == 0) return cudaSuccess;
    rms_merge_sequence_kernel<<<1, ((c + 31) / 32) * 32, 0, st>>>(acc, order, nu, pivot, running_mean, running_var, count, seq, c);
    return cudaGetLastError();
}

// n_batches minibatches in one launch: batch b is the slab view based at x + b * x_batch_rows * c, normalised with the statistics
// at running_mean / running_var + b * stat_batch into y + b * m * c
cudaError_t launch_rms_normalize_batched(const float* x, const double* running_mean, const double* running_var, float eps, float* y,
                                         int64_t m, int c, int64_t slab_rows, int64_t slab_stride, int64_t x_batch_rows,
                                         int64_t stat_batch, int n_batches, cudaStream_t st) {
    if (m * c == 0 || n_batches == 0) return cudaSuccess;
    if (slab_rows <= 0 || slab_rows > m || m % slab_rows != 0) return cudaErrorInvalidValue;
    const int64_t nslabs = m / slab_rows;
    if (nslabs > 65535 || n_batches > 65535) return cudaErrorInvalidValue;
    const int64_t total = slab_rows * c;
    const int vec4 = aligned16(x) && aligned16(y) && total % 4 == 0 && (slab_stride * c) % 4 == 0 && (x_batch_rows * c) % 4 == 0 &&
                     (m * c) % 4 == 0;
    int blocks = stream_blocks(vec4 ? total / 4 : total, 256, 8);
    const int cap = (int)((148 * 8 + nslabs * n_batches - 1) / (nslabs * n_batches));
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    rms_normalize_kernel<true><<<dim3((unsigned)blocks, (unsigned)nslabs, (unsigned)n_batches), 256, 2 * c * sizeof(float), st>>>(
        x, running_mean, running_var, eps, 0, y, total, c, vec4, slab_stride * c, x_batch_rows * c, m * c, stat_batch);
    return cudaGetLastError();
}

cudaError_t launch_rms_normalize(const float* x, const double* running_mean, const double* running_var, float eps,
                                 int unnorm, float* y, int64_t m, int c, int64_t slab_rows, int64_t slab_stride, cudaStream_t st) {
    if (m * c == 0) return cudaSuccess;
    if (slab_rows <= 0 || slab_rows >= m) { slab_rows = m; slab_stride = m; }
    if (m % slab_rows != 0) return cudaErrorInvalidValue;
    const int64_t nslabs = m / slab_rows;
    if (nslabs > 65535) return cudaErrorInvalidValue;
    const int64_t total = slab_rows * c;                 // elements per slab
    const int vec4 = aligned16(x) && aligned16(y) && (nslabs == 1 || (total % 4 == 0 && (slab_stride * c) % 4 == 0));
    int blocks = stream_blocks(vec4 ? total / 4 : total, 256, 8);
    const int per_slab_cap = (int)((148 * 8 + nslabs - 1) / nslabs);
    if (blocks > per_slab_cap) blocks = per_slab_cap;
    if (nslabs > 1)
        rms_normalize_kernel<true><<<dim3((unsigned)blocks, (unsigned)nslabs), 256, 2 * c * sizeof(float), st>>>(
            x, running_mean, running_var, eps, unnorm, y, total, c, vec4, slab_stride * c);
    else
        rms_normalize_kernel<false><<<blocks, 256, 2 * c * sizeof(float), st>>>(x, running_mean, running_var, eps, unnorm, y, total, c,
                                                                                vec4, 0);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// K7: advantage statistics / normalisation (a2c_common.py prepare_dataset)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) adv_normalize_kernel(const float* __restrict__ returns, const float* __restrict__ values,
                                                            const double* __restrict__ acc, float* __restrict__ adv, int normalize,
                                                            int64_t m, int vec4) {
    float mean = 0.0f, den = 1.0f;
    if (normalize) {
        const double B = acc[0], S = acc[1], SS = acc[2];
        const double mu = S / B;
        const double var = (SS - S * mu) / (B - 1.0);              // unbiased, torch.std default
        mean = (float)mu;
        // a rounding-negative variance is 0; a NaN one (B == 1) stays NaN, like torch.std
        den = (float)sqrt(var < 0.0 ? 0.0 : var) + 1e-8f;
    }
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nvec = vec4 ? (m >> 2) : 0;
    for (int64_t i = tid; i < nvec; i += stride) {
        const float4 r = ldg_stream4(reinterpret_cast<const float4*>(returns) + i);
        const float4 v = ldg_stream4(reinterpret_cast<const float4*>(values) + i);
        float4 o = make_float4(r.x - v.x, r.y - v.y, r.z - v.z, r.w - v.w);
        if (normalize) { o.x = (o.x - mean) / den; o.y = (o.y - mean) / den; o.z = (o.z - mean) / den; o.w = (o.w - mean) / den; }
        __stcs(reinterpret_cast<float4*>(adv) + i, o);
    }
    for (int64_t i = nvec * 4 + tid; i < m; i += stride) {
        float o = returns[i] - values[i];
        if (normalize) o = (o - mean) / den;
        adv[i] = o;
    }
}

cudaError_t launch_adv_moments(const float* returns, const float* values, double* acc, double* partials, int64_t m,
                               cudaStream_t st) {
    const int vec4 = aligned16(returns) && aligned16(values);
    const int nblocks = stream_blocks(vec4 ? m / 4 : m, RMS_THREADS, 4);
    flat_partials_kernel<<<nblocks, RMS_THREADS, 0, st>>>(returns, values, nullptr, partials, m, vec4, m, m);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return err;
    return launch_pdl(learner_pdl(), moments_finalize_kernel, dim3(1), dim3(256), 0, st, (const double*)partials, nblocks, 1, m, acc, (const double*)nullptr,
                     (const double*)nullptr, (const double*)nullptr);
}

cudaError_t launch_adv_normalize(const float* returns, const float* values, const double* acc, float* adv, int normalize,
                                 int64_t m, cudaStream_t st) {
    if (m == 0) return cudaSuccess;
    const int vec4 = aligned16(returns) && aligned16(values) && aligned16(adv);
    const int blocks = stream_blocks(vec4 ? m / 4 : m, 256, 8);
    adv_normalize_kernel<<<blocks, 256, 0, st>>>(returns, values, acc, adv, normalize, m, vec4);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// K8: fused PPO loss forward + backward.  One thread per sample; the four (m,18) row arrays of a
// 128-sample tile arrive as four cp.async.bulk copies (9216 contiguous bytes each) and grad_mu leaves
// as one bulk store.  Per-block partial sums (fp64) of the five loss terms, clip fraction and the 18
// logstd gradients are folded in block order by a finalize kernel.
// ------------------------------------------------------------------------------------------------
constexpr int PPO_TILE = 128;
constexpr int PPO_NSTAT = 7;                    // a, c, b, kl, clipped, (spare), (spare)
constexpr int PPO_PART = PPO_NSTAT + 18;        // doubles per block
constexpr int PPO_FLUSH = 8;                    // tiles between fp32 -> fp64 flushes
constexpr int PPO_MAX_BLOCKS = 148 * 4;         // persistent grid: every CTA walks tiles blockIdx.x, +gridDim.x, ...

// s_tot: the PPO_PART column totals.  Thread 0 forms the loss terms (means), threads 0..17 the logstd gradients.
__device__ __forceinline__ void ppo_form_loss(const double* s_tot, int64_t m, const float* __restrict__ logstd, const BezkPpoCfg& cfg,
                                              double* __restrict__ stats, float* __restrict__ grad_logstd, int tid) {
    const double inv_m = 1.0 / (double)m;
    if (tid == 0) {
        double ent = 0.0;
        for (int k = 0; k < 18; ++k) ent += (double)((0.5f + 0.9189385332046727f) + logstd[k]);   // 0.5*log(2*pi)
        const double a_m = s_tot[0] * inv_m, c_m = s_tot[1] * inv_m, b_m = s_tot[2] * inv_m, kl_m = s_tot[3] * inv_m;
        stats[1] = a_m; stats[2] = c_m; stats[3] = ent; stats[4] = b_m; stats[5] = kl_m; stats[6] = s_tot[4] * inv_m; stats[7] = 0.0;
        stats[0] = a_m + 0.5 * c_m * (double)cfg.critic_coef - ent * (double)cfg.entropy_coef + b_m * (double)cfg.bounds_loss_coef;
    }
    if (grad_logstd && tid < 18)
        grad_logstd[tid] = (float)(s_tot[PPO_NSTAT + tid] * inv_m - (double)cfg.entropy_coef);
}

__global__ void __launch_bounds__(PPO_TILE, 4) ppo_loss_kernel(const PpoArgs a, const __grid_constant__ BezkPpoCfg cfg) {
    __shared__ __align__(128) float s_act[PPO_TILE * 18];
    __shared__ __align__(128) float s_mu[PPO_TILE * 18];
    __shared__ __align__(128) float s_omu[PPO_TILE * 18];
    __shared__ __align__(128) float s_osig[PPO_TILE * 18];
    __shared__ __align__(128) float s_gmu[PPO_TILE * 18];
    __shared__ __align__(8) uint64_t s_bar;
    __shared__ float s_sigma[18], s_logstd[18], s_isig[18], s_ry[18];
    __shared__ double s_red[PPO_TILE / 32][PPO_PART];

    const int tid = threadIdx.x;
    constexpr uint32_t TILE_BYTES = PPO_TILE * 18 * 4;
    const int64_t ntiles = (a.m + PPO_TILE - 1) / PPO_TILE;
    const float inv_m = 1.0f / (float)a.m;

    if (tid == 0) { mbar_init(&s_bar, 1); fence_mbar_init(); }
    pdl_wait();
    pdl_launch_dependents();
    if (tid < 18) { const float ls = a.logstd[tid]; s_logstd[tid] = ls; s_sigma[tid] = expf(ls); }
    __syncthreads();
    // per-column constants.  The FORWARD quantities (neglogp, KL) divide by sigma exactly as the reference does (branch-free IEEE
    // division, Mth); only the hand-derived GRADIENT sweep below multiplies by 1/sigma (it has no reference op order to follow).
    // (the 2 x 18 constants are read from shared memory -- broadcast loads -- instead of living in 36 registers)
    if (tid < 18) { s_isig[tid] = 1.0f / s_sigma[tid]; s_ry[tid] = Mth<true>::rcp_refined(s_sigma[tid]); }
    __syncthreads();
    const float* sig = s_sigma;
    const float* isig = s_isig;
    float lsum = 0.0f;
#pragma unroll
    for (int j = 0; j < 18; ++j) lsum += s_logstd[j];

    // per-thread fp32 running sums, flushed every PPO_FLUSH tiles (a thread adds one sample per tile) through a
    // fixed-order fp64 warp reduction into per-warp fp64 accumulators in shared memory: 25 registers instead of 50,
    // deterministic, and the fp32 partial sums never hold more than PPO_FLUSH terms
    float part[PPO_PART];
#pragma unroll
    for (int k = 0; k < PPO_PART; ++k) part[k] = 0.0f;
    for (int k = tid; k < (PPO_TILE / 32) * PPO_PART; k += PPO_TILE) (&s_red[0][0])[k] = 0.0;
    int since_flush = 0;
    const int lane = tid & 31, wid = tid >> 5;
    auto flush = [&]() {
#pragma unroll
        for (int k = 0; k < PPO_PART; ++k) {
            const double t = warp_sum((double)part[k]);
            if (lane == 0) s_red[wid][k] += t;
            part[k] = 0.0f;
        }
    };
    uint32_t phase = 0;
    bool store_pending = false;

    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t i0 = tile * PPO_TILE;
        const int nv = (int)((a.m - i0) < (int64_t)PPO_TILE ? (a.m - i0) : (int64_t)PPO_TILE);
        const bool full = (nv == PPO_TILE) && a.use_tma;
        const int64_t i = i0 + tid;
        const bool valid = tid < nv;
        // rollout-side tensors (actions, old_*, returns, advantages) may be slabs of time-major storage; the network-side
        // ones (mu, values) and every output are contiguous batch rows.  TMA tiles never straddle a slab (launcher check).
        const int64_t j0 = a.slabs ? slab_src_row(i0, a.slab_rows, a.slab_stride) : i0;
        const int64_t ji = a.slabs ? ((full || !valid) ? j0 + tid : slab_src_row(i, a.slab_rows, a.slab_stride)) : i;

        // per-sample scalars first (five independent loads in flight while thread 0 sets up the bulk copies)
        float val = 0.f, oval = 0.f, ret = 0.f, onlp = 0.f, adv = 0.f;
        if (valid) { val = a.values[i]; oval = a.old_values[ji]; ret = a.returns[ji]; onlp = a.old_neglogp[ji]; adv = a.advantages[ji]; }
        if (tid == 0 && store_pending) bulk_wait_read0();          // s_gmu of the previous tile has been read out
        __syncthreads();                                           // everybody is done with the previous tile's rows
        if (full) {
            if (tid == 0) {
                mbar_arrive_expect_tx(&s_bar, 4 * TILE_BYTES);
                bulk_g2s(s_act, a.actions + j0 * 18, TILE_BYTES, &s_bar);
                bulk_g2s(s_mu, a.mu + i0 * 18, TILE_BYTES, &s_bar);
                bulk_g2s(s_omu, a.old_mu + j0 * 18, TILE_BYTES, &s_bar);
                bulk_g2s(s_osig, a.old_sigma + j0 * 18, TILE_BYTES, &s_bar);
            }
        } else {
            for (int k = tid; k < nv * 18; k += PPO_TILE) {
                const int row = k / 18;
                const int64_t jk = (a.slabs ? slab_src_row(i0 + row, a.slab_rows, a.slab_stride) : (i0 + row)) * 18 + (k - row * 18);
                s_act[k] = a.actions[jk]; s_mu[k] = a.mu[i0 * 18 + k];
                s_omu[k] = a.old_mu[jk]; s_osig[k] = a.old_sigma[jk];
            }
        }
        if (full) { mbar_wait(&s_bar, phase); phase ^= 1u; }
        else __syncthreads();

        if (valid) {
            // ---- neglogp (models.py), bound loss, KL: one sweep over the 18 action dims ----
            float sq = 0.0f, bsum = 0.0f, kl = 0.0f;
            Mth<true> mk;
            // two of the three quotients per action dim divide by sigma_j, a per-column constant: its refined reciprocal is
            // formed once per CTA and the divisors are range-checked once per thread (same bits as mk.div, fewer instructions)
#pragma unroll
            for (int j = 0; j < 18; ++j) mk.check_divisor(sig[j]);
            const float2* act2 = reinterpret_cast<const float2*>(s_act + tid * 18);
            const float2* mu2 = reinterpret_cast<const float2*>(s_mu + tid * 18);
            const float2* omu2 = reinterpret_cast<const float2*>(s_omu + tid * 18);
            const float2* osig2 = reinterpret_cast<const float2*>(s_osig + tid * 18);
#pragma unroll
            for (int h = 0; h < 9; ++h) {
                const float2 A2 = act2[h], M2 = mu2[h], OM2 = omu2[h], OS2 = osig2[h];
                const float av[2] = {A2.x, A2.y}, mv[2] = {M2.x, M2.y}, omv[2] = {OM2.x, OM2.y}, osv[2] = {OS2.x, OS2.y};
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const int j = 2 * h + q;
                    const float zz = mk.div_by(av[q] - mv[q], sig[j], s_ry[j]);   // the reference DIVIDES by sigma (models.py neglogp): exact
                    sq += zz * zz;
                    float hi, lo;
                    if (cfg.bound_form == 0) {          // rl_games 1.1.3 as recalled
                        hi = fminf(mv[q] - cfg.soft_bound, 0.0f); lo = fminf(-mv[q] + cfg.soft_bound, 0.0f);
                    } else {                            // later releases
                        hi = fmaxf(mv[q] - cfg.soft_bound, 0.0f); lo = fminf(mv[q] + cfg.soft_bound, 0.0f);
                    }
                    bsum += lo * lo + hi * hi;
                    const float c1 = logf(mk.div_by(osv[q], sig[j], s_ry[j]) + 1e-5f);   // torch_ext.policy_kl: log(p1_sigma / p0_sigma + 1e-5)
                    const float dm = omv[q] - mv[q];
                    const float c2 = mk.div(sig[j] * sig[j] + dm * dm, 2.0f * (osv[q] * osv[q] + 1e-5f));   // exact, no branch per dim
                    kl += (c1 + c2) + (-0.5f);
                }
            }
            if (mk.bad()) {                    // an operand outside the fast division's range: redo both sums with the plain operator
                kl = 0.0f; sq = 0.0f;
                for (int j = 0; j < 18; ++j) {
                    const float a_ = s_act[tid * 18 + j], m_ = s_mu[tid * 18 + j], om_ = s_omu[tid * 18 + j], os_ = s_osig[tid * 18 + j];
                    const float zz = (a_ - m_) / sig[j];
                    sq += zz * zz;
                    const float c1 = logf(os_ / sig[j] + 1e-5f);
                    const float dm = om_ - m_;
                    const float c2 = (sig[j] * sig[j] + dm * dm) / (2.0f * (os_ * os_ + 1e-5f));
                    kl += (c1 + c2) + (-0.5f);
                }
            }
            const float nlp = (0.5f * sq + (float)(0.5 * 1.8378770664093453 * 18.0)) + lsum;   // log(2*pi) = 1.83787706...
            if (a.neglogp_out) a.neglogp_out[i] = nlp;
            // ---- actor loss (common_losses.actor_loss) ----
            const float ratio = expf(onlp - nlp);
            const float lo_r = 1.0f - cfg.e_clip, hi_r = 1.0f + cfg.e_clip;
            const float s1 = adv * ratio, s2 = adv * clamp_nan(ratio, lo_r, hi_r);
            const float a_loss = max_nan(-s1, -s2);
            const bool inside = (ratio >= lo_r) && (ratio <= hi_r);
            const bool through = inside || (-s1 > -s2);
            const float dnlp = through ? (adv * ratio) : 0.0f;            // d a_loss / d neglogp
            // ---- critic loss (common_losses.critic_loss) ----
            float c_loss, dval;
            const float t1 = (val - ret) * (val - ret);
            if (cfg.clip_value) {
                const float dv = val - oval;
                const float vpc = oval + clamp_nan(dv, -cfg.e_clip, cfg.e_clip);
                const float t2 = (vpc - ret) * (vpc - ret);
                c_loss = max_nan(t1, t2);
                const float g1 = 2.0f * (val - ret);
                const float g2 = (dv >= -cfg.e_clip && dv <= cfg.e_clip) ? 2.0f * (vpc - ret) : 0.0f;
                dval = (t1 > t2) ? g1 : ((t2 > t1) ? g2 : 0.5f * (g1 + g2));
            } else {
                c_loss = t1;
                dval = 2.0f * (val - ret);
            }
            if (a.grad_values) a.grad_values[i] = (0.5f * cfg.critic_coef) * dval * inv_m;
            // ---- gradients wrt mu (row) and running sums for logstd ----
            // second sweep: z and the bound-loss derivative are recomputed from the shared-memory rows (cheaper than
            // keeping 36 values alive across the actor / critic block)
            float2* g2p = reinterpret_cast<float2*>(s_gmu + tid * 18);
#pragma unroll
            for (int h = 0; h < 9; ++h) {
                const int j = 2 * h;
                const float2 A2 = act2[h], M2 = mu2[h];
                const float av[2] = {A2.x, A2.y}, mv[2] = {M2.x, M2.y};
                float gout[2];
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const float zz = (av[q] - mv[q]) * isig[j + q];
                    float dbound;
                    if (cfg.bound_form == 0) dbound = 2.0f * fminf(mv[q] - cfg.soft_bound, 0.0f) + (-2.0f) * fminf(-mv[q] + cfg.soft_bound, 0.0f);
                    else dbound = 2.0f * fmaxf(mv[q] - cfg.soft_bound, 0.0f) + 2.0f * fminf(mv[q] + cfg.soft_bound, 0.0f);
                    gout[q] = (dnlp * (-zz * isig[j + q]) + cfg.bounds_loss_coef * dbound) * inv_m;
                    part[PPO_NSTAT + j + q] += dnlp * (1.0f - zz * zz);
                }
                g2p[h] = make_float2(gout[0], gout[1]);
            }
            part[0] += a_loss; part[1] += c_loss; part[2] += bsum; part[3] += kl;
            part[4] += inside ? 0.0f : 1.0f;
        }
        if (++since_flush == PPO_FLUSH) { flush(); since_flush = 0; }

        // ---- grad_mu tile out ----
        if (a.grad_mu) {
            if (full) {
                fence_proxy_async_smem();
                __syncthreads();
                if (tid == 0) { bulk_s2g(a.grad_mu + i0 * 18, s_gmu, TILE_BYTES); bulk_commit(); store_pending = true; }
            } else {
                __syncthreads();
                for (int k = tid; k < nv * 18; k += PPO_TILE) a.grad_mu[i0 * 18 + k] = s_gmu[k];
            }
        }
    }

    // ---- final flush, then a fixed-order fold over the 4 warps ----
    flush();
    __syncthreads();
    if (tid < PPO_PART) {
        double t = 0.0;
#pragma unroll
        for (int q = 0; q < PPO_TILE / 32; ++q) t += s_red[q][tid];
        a.partials[(int64_t)blockIdx.x * PPO_PART + tid] = t;
    }
    if (tid == 0 && store_pending) bulk_wait_read0();
    if (a.fused_finalize) {
        // single-launch mode (cooperative grid): after a grid-wide barrier CTA 0 folds the partials and forms the loss -- the
        // separate finalize launch costs more than the whole kernel at the reference's minibatch (32 768 samples)
        __threadfence();
        cooperative_groups::this_grid().sync();
        if (blockIdx.x != 0) return;
        double* s_tot = &s_red[0][0];
        // fixed-order fold with every load of a chunk in flight: thread (column j = tid % 32 < 25, row group q = tid / 32) sums CTAs
        // q, q + 4, ... (unrolled by 8: independent loads), then the 4 row groups are added in order
        __shared__ double s_fold[PPO_TILE / 32][32];
        {
            const int j = lane, q = wid;
            double t = 0.0;
            if (j < PPO_PART) {
                int b = q;
                const int nb = (int)gridDim.x, stride = PPO_TILE / 32;
                for (; b + 7 * stride < nb; b += 8 * stride) {
                    double v[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) v[u] = __ldcg(a.partials + (int64_t)(b + u * stride) * PPO_PART + j);
#pragma unroll
                    for (int u = 0; u < 8; ++u) t += v[u];
                }
                for (; b < nb; b += stride) t += __ldcg(a.partials + (int64_t)b * PPO_PART + j);
            }
            s_fold[q][j] = t;
        }
        __syncthreads();
        if (tid < PPO_PART) {
            double t = 0.0;
#pragma unroll
            for (int q = 0; q < PPO_TILE / 32; ++q) t += s_fold[q][tid];
            s_tot[tid] = t;
        }
        __syncthreads();
        ppo_form_loss(s_tot, a.m, a.logstd, cfg, a.stats, a.grad_logstd, tid);
    }
}

// one warp per statistic folds the per-CTA partials (fixed order), thread 0 of warp 0 then forms the loss
__global__ void __launch_bounds__(1024) ppo_finalize_kernel(const double* __restrict__ partials, int nblocks, int64_t m,
                                                            const float* __restrict__ logstd, const __grid_constant__ BezkPpoCfg cfg,
                                                            double* __restrict__ stats, float* __restrict__ grad_logstd) {
    __shared__ double s_tot[PPO_PART];
    pdl_wait();                 // programmatic dependent launch: everything below may read the previous kernel's output
    pdl_launch_dependents();
    const int lane = threadIdx.x & 31, j = threadIdx.x >> 5;
    if (j < PPO_PART) {
        const double t = fold_column(partials, nblocks, PPO_PART, j, lane);
        if (lane == 0) s_tot[j] = t;
    }
    __syncthreads();
    ppo_form_loss(s_tot, m, logstd, cfg, stats, grad_logstd, (int)threadIdx.x);
}


int64_t ppo_scratch_doubles() { return (int64_t)PPO_MAX_BLOCKS * PPO_PART; }

cudaError_t launch_ppo_loss(const PpoArgs& args, const BezkPpoCfg& cfg, double* stats, float* grad_logstd, cudaStream_t st) {
    PpoArgs a = args;
    if (a.m <= 0) return cudaErrorInvalidValue;
    const int64_t ntiles = (a.m + PPO_TILE - 1) / PPO_TILE;
    const int nblocks = (int)(ntiles < PPO_MAX_BLOCKS ? ntiles : PPO_MAX_BLOCKS);
    if (a.slab_rows <= 0 || a.slab_rows >= a.m) { a.slab_rows = a.m; a.slab_stride = a.m; }
    if (a.m % a.slab_rows != 0) return cudaErrorInvalidValue;
    a.slabs = a.slab_rows < a.m;
    a.use_tma = aligned16(a.actions) && aligned16(a.mu) && aligned16(a.old_mu) && aligned16(a.old_sigma) &&
                (a.grad_mu == nullptr || aligned16(a.grad_mu)) &&
                (!a.slabs || (a.slab_rows % PPO_TILE == 0 && (a.slab_stride * 18 * 4) % 16 == 0));
    a.stats = stats; a.grad_logstd = grad_logstd;
    // The grid never exceeds 4 resident CTAs per SM (PPO_MAX_BLOCKS), so it CAN be launched cooperatively with CTA 0 finalizing
    // after a grid barrier (BEZK_PPO_SINGLE_LAUNCH=1).  Measured at the reference's minibatch (32 768): 11.9 us against 10.7 us
    // for the two-kernel form -- a cooperative launch + grid barrier costs more than a second launch -- so two kernels ship.
    static const int single = env_int("BEZK_PPO_SINGLE_LAUNCH", 0);
    if (single) {
        a.fused_finalize = 1;
        cudaLaunchConfig_t lc = {};
        lc.gridDim = dim3((unsigned)nblocks); lc.blockDim = dim3(PPO_TILE); lc.dynamicSmemBytes = 0; lc.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeCooperative;
        attr[0].val.cooperative = 1;
        lc.attrs = attr; lc.numAttrs = 1;
        return cudaLaunchKernelEx(&lc, ppo_loss_kernel, a, cfg);
    }
    a.fused_finalize = 0;
    cudaError_t err = launch_pdl(learner_pdl(), ppo_loss_kernel, dim3((unsigned)nblocks), dim3(PPO_TILE), 0, st, a, cfg);
    if (err != cudaSuccess) return err;
    return launch_pdl(learner_pdl(), ppo_finalize_kernel, dim3(1), dim3(32 * PPO_PART), 0, st, (const double*)a.partials, nblocks, a.m, a.logstd, cfg, stats,
                     grad_logstd);
}

}  // namespace bezk
