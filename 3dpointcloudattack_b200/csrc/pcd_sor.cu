// pcd_sor.cu -- statistical outlier removal (SOR), the standard point-cloud defence, in float64, sm_100a.
//
// attack/SIadv/baselines/defense/drop_points/SOR.py:24-54 builds two [B,N,N] float64 matrices (inner, dist), runs
// topk(k + 1) on the negated distances, and thresholds the mean of the k nearest non-self distances at
// mean + alpha * std over the cloud.  Here the matrix never exists:
//   sor_sweep_kernel     every row keeps its k + 1 smallest distance VALUES in a sorted register list while the CTA
//                        streams the sample's columns through shared memory; the row's mean of entries 1..k is stored.
//   sor_epilogue_kernel  one CTA per sample: two-pass mean and unbiased std in a fixed order, the keep-mask, and a
//                        stable block-scan compaction of the kept indices.
// The arithmetic is the contract of pcd_sor_forward in include/pcdist.h.  Float32 inputs make every coordinate
// product exact in float64, so fma(a, b, c) == (a * b) + c here and the pair distance costs DMUL + 2 DFMA + DADD.
#include <math.h>

#include "pcd_common.cuh"

namespace pcd {

constexpr int kSorThreads = 64;      // sweep CTA; each thread loads one column of every staged tile
constexpr int kSorTile = kSorThreads;
constexpr int kSorEpiThreads = 1024;

struct __align__(32) SorCol {
    double x, y, z, n;
};

__device__ __forceinline__ double sq_norm3_f64(double x, double y, double z) {
    return __dadd_rn(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)), __dmul_rn(z, z));
}

// L: list length (k + 1 <= L), R: rows per thread.  The front L - (k + 1) slots hold -inf and never move, so the
// last k + 1 slots are the k + 1 smallest values seen; every index below is static (no local memory).
template <int L, int R>
__global__ void __launch_bounds__(kSorThreads) sor_sweep_kernel(const float *__restrict__ pc, long long sb, long long sp,
                                                                long long sc, int N, int k, int tiles_per_sample,
                                                                double *__restrict__ value) {
    __shared__ SorCol cols[2][kSorTile];
    const int b = blockIdx.x / tiles_per_sample, row0 = (blockIdx.x - b * tiles_per_sample) * (R * kSorThreads);
    const float *base = pc + (size_t)b * sb;
    const int tid = threadIdx.x;

    // row side: -2 * coordinates (exact) so that the dot product comes out as -2 * dot without a rounding of its own
    double mx[R], my[R], mz[R], nr[R], list[R][L];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const long long i = min(row0 + r * kSorThreads + tid, N - 1);
        const double x = base[i * sp], y = base[i * sp + sc], z = base[i * sp + 2 * sc];
        nr[r] = sq_norm3_f64(x, y, z);
        mx[r] = -2.0 * x;
        my[r] = -2.0 * y;
        mz[r] = -2.0 * z;
#pragma unroll
        for (int s = 0; s < L; ++s) list[r][s] = s < L - 1 - k ? -INFINITY : INFINITY;
    }

    // columns: one per thread per tile, loaded into registers a tile ahead; padding columns have norm +inf, so their
    // values (+inf or NaN) never pass the insertion gate
    const int ntiles = (N + kSorTile - 1) / kSorTile;
    float cx = 0.f, cy = 0.f, cz = 0.f;
    auto load = [&](int t) {
        const long long j = (long long)t * kSorTile + tid;
        if (j < N) {
            cx = base[j * sp];
            cy = base[j * sp + sc];
            cz = base[j * sp + 2 * sc];
        }
    };
    load(0);
    for (int t = 0; t < ntiles; ++t) {
        SorCol c;
        c.x = cx; c.y = cy; c.z = cz;
        c.n = t * kSorTile + tid < N ? sq_norm3_f64(c.x, c.y, c.z) : INFINITY;
        if (t * kSorTile + tid >= N) c.x = c.y = c.z = 0.0;
        cols[t & 1][tid] = c;               // the buffer last read two tiles ago: every thread has passed a barrier since
        __syncthreads();
        if (t + 1 < ntiles) load(t + 1);
        const SorCol *tile = cols[t & 1];
#pragma unroll 2
        for (int jj = 0; jj < kSorTile; ++jj) {
            const SorCol q = tile[jj];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                // xx[j] + (-2 * dot): d minus the row norm, which rounding-monotonicity lets the ranking leave out
                const double e = __dadd_rn(q.n, __fma_rn(mz[r], q.z, __fma_rn(my[r], q.y, __dmul_rn(mx[r], q.x))));
                if (e < list[r][L - 1]) {
#pragma unroll
                    for (int s = L - 1; s > 0; --s) list[r][s] = fmax(list[r][s - 1], fmin(list[r][s], e));
                    list[r][0] = fmin(list[r][0], e);
                }
            }
        }
    }

#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int i = row0 + r * kSorThreads + tid;
        if (i >= N) continue;
        double acc = 0.0;                   // s_1 + ... + s_k, left to right; s_0 (slot L-1-k) is dropped
#pragma unroll
        for (int s = 0; s < L; ++s)
            if (s >= L - k) acc = __dadd_rn(acc, __dadd_rn(list[r][s], nr[r]));
        value[(size_t)b * N + i] = __ddiv_rn(acc, (double)k);
    }
}

__device__ __forceinline__ int warp_inclusive_scan(int v) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += u;
    }
    return v;
}

__global__ void __launch_bounds__(kSorEpiThreads) sor_epilogue_kernel(int N, double alpha, const double *__restrict__ value,
                                                                      double *__restrict__ thr_out, uint8_t *__restrict__ keep,
                                                                      int32_t *__restrict__ kept_idx, int32_t *__restrict__ lengths) {
    __shared__ double shd[kSorEpiThreads / 32];
    __shared__ int shi[kSorEpiThreads / 32];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const double *v = value + (size_t)b * N;
    uint8_t *kp = keep + (size_t)b * N;
    int32_t *out = kept_idx + (size_t)b * N;

    double s = 0.0;
    for (int i = tid; i < N; i += kSorEpiThreads) s = __dadd_rn(s, v[i]);
    const double mean = __ddiv_rn(block_sum<double, kSorEpiThreads>(s, shd), (double)N);
    double q = 0.0;
    for (int i = tid; i < N; i += kSorEpiThreads) {
        const double c = __dadd_rn(v[i], -mean);
        q = __dadd_rn(q, __dmul_rn(c, c));
    }
    const double var = __ddiv_rn(block_sum<double, kSorEpiThreads>(q, shd), (double)(N - 1));   // unbiased (torch.std)
    const double thr = __dadd_rn(mean, __dmul_rn(alpha, __dsqrt_rn(var)));

    // stable compaction, one block-wide chunk at a time: ballot within the warp, scan over the warp counts
    int count = 0;
    for (int i0 = 0; i0 < N; i0 += kSorEpiThreads) {
        const int i = i0 + tid;
        const bool kept = i < N && v[i] <= thr;
        if (i < N) kp[i] = kept ? 1 : 0;
        const unsigned m = __ballot_sync(0xffffffffu, kept);
        if (lane == 0) shi[warp] = __popc(m);
        __syncthreads();
        const int incl = warp_inclusive_scan(lane < kSorEpiThreads / 32 ? shi[lane] : 0);
        const int before = __shfl_sync(0xffffffffu, incl, warp) - shi[warp];      // kept in the warps below this one
        if (kept) out[count + before + __popc(m & ((1u << lane) - 1u))] = i;
        count += __shfl_sync(0xffffffffu, incl, 31);
        __syncthreads();                    // shi is rewritten by the next chunk
    }
    for (int i = count + tid; i < N; i += kSorEpiThreads) out[i] = -1;
    if (tid == 0) {
        thr_out[b] = thr;
        lengths[b] = count;
    }
}

template <int L, int R>
static int launch_sor(const float *pc, int64_t sb, int64_t sp, int64_t sc, int B, int N, int k, double *value, cudaStream_t st) {
    const int tiles = (N + R * kSorThreads - 1) / (R * kSorThreads);
    if ((long long)tiles * B > 2147483647LL) {
        set_error("pcd_sor_forward: B * ceil(N / %d) exceeds the grid limit", R * kSorThreads);
        return PCD_ERR_ARG;
    }
    sor_sweep_kernel<L, R><<<(unsigned)(tiles * B), kSorThreads, 0, st>>>(pc, sb, sp, sc, N, k, tiles, value);
    PCD_CUDA_CHECK(cudaGetLastError());
    return PCD_OK;
}

}  // namespace pcd

using namespace pcd;

extern "C" int pcd_sor_forward(const float *pc, int64_t sb, int64_t sp, int64_t sc, int B, int N, int k, double alpha,
                               double *value, double *threshold, uint8_t *keep, int32_t *kept_idx, int32_t *lengths,
                               void *stream) {
    if (!pc || !value || !threshold || !keep || !kept_idx || !lengths || B <= 0 || k < 1 || k > PCD_SOR_MAX_K || N < k + 1 ||
        !isfinite(alpha)) {
        set_error("pcd_sor_forward: bad argument (need B >= 1, 1 <= k <= %d, N >= k + 1, finite alpha, no NULL pointer)",
                  PCD_SOR_MAX_K);
        return PCD_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int rc = k + 1 <= 4   ? launch_sor<4, 4>(pc, sb, sp, sc, B, N, k, value, st)
                   : k + 1 <= 8 ? launch_sor<8, 4>(pc, sb, sp, sc, B, N, k, value, st)
                                : launch_sor<16, 2>(pc, sb, sp, sc, B, N, k, value, st);
    if (rc != PCD_OK) return rc;
    sor_epilogue_kernel<<<B, kSorEpiThreads, 0, st>>>(N, alpha, value, threshold, keep, kept_idx, lengths);
    PCD_CUDA_CHECK(cudaGetLastError());
    return PCD_OK;
}
