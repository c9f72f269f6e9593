// pcd_sor.cu -- statistical outlier removal (SOR), the standard point-cloud defence, in float64, sm_100a.
//
// attack/SIadv/baselines/defense/drop_points/SOR.py:24-54 builds two [B,N,N] float64 matrices (inner, dist), runs
// topk(k + 1) on the negated distances, and thresholds the mean of the k nearest non-self distances at
// mean + alpha * std over the cloud.  Here the matrix never exists:
//   sor_sweep_kernel     every row keeps its k + 1 smallest distance VALUES in a sorted register list while the CTA
//                        streams the sample's columns through shared memory; the row's mean of entries 1..k is stored.
//   sor_epilogue_kernel  one CTA per sample: two-pass mean and unbiased std in a fixed order, the keep-mask, and a
//                        stable block-scan compaction of the kept indices.
// pcd_sor_forward_len runs the same arithmetic on the first len[b] points of every sample, with the columns of a
// sample optionally split over several CTAs:
//   sor_len_sweep_kernel     as sor_sweep_kernel over one column range; with one range it stores the row's value,
//                            otherwise the range's k + 1 smallest values go to the workspace.
//   sor_merge_kernel         one thread per valid row: merges the ranges' sorted lists into the k + 1 smallest values.
//                            They are the same multiset at any split, so the value has the same bits.
//   sor_len_epilogue_kernel  sor_epilogue_kernel on the valid rows, plus the padding rows and the short samples.
// The arithmetic is the contract of pcd_sor_forward in include/pcdist.h.  Float32 inputs make every coordinate
// product exact in float64, so fma(a, b, c) == (a * b) + c here and the pair distance costs DMUL + 2 DFMA + DADD.
#include <math.h>

#include <algorithm>

#include "pcd_common.cuh"

namespace pcd {

constexpr int kSorThreads = 64;      // sweep CTA; each thread loads one column of every staged tile
constexpr int kSorTile = kSorThreads;
constexpr int kSorEpiThreads = 1024;
constexpr int kSorMergeThreads = 256;
// Column split of pcd_sor_forward_len: while B * row tiles is below about two waves of a 148-SM B200 at eight sweep CTAs
// per SM, a row tile's columns are spread over several CTAs.  A fixed target (no device query) keeps the workspace size
// a function of the shape alone.
constexpr long long kSorTargetCtas = 2 * 148 * 8;
constexpr int kSorMaxSplit = 64;

struct __align__(32) SorCol {
    double x, y, z, n;
};

__device__ __forceinline__ double sq_norm3_f64(double x, double y, double z) {
    return __dadd_rn(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)), __dmul_rn(z, z));
}

__device__ __forceinline__ int sor_len(const int32_t *len, int b, int N) { return len ? min(max(len[b], 0), N) : N; }

// L: list length (k + 1 <= L).  The front L - (k + 1) slots hold -inf and never move, so the last k + 1 slots are the
// k + 1 smallest values seen; every index below is static (no local memory).
template <int L>
__device__ __forceinline__ void sor_list_init(double (&list)[L], int k) {
#pragma unroll
    for (int s = 0; s < L; ++s) list[s] = s < L - 1 - k ? -INFINITY : INFINITY;
}

template <int L>
__device__ __forceinline__ void sor_list_insert(double (&list)[L], double e) {
    if (e < list[L - 1]) {
#pragma unroll
        for (int s = L - 1; s > 0; --s) list[s] = fmax(list[s - 1], fmin(list[s], e));
        list[0] = fmin(list[0], e);
    }
}

// s_1 + ... + s_k, left to right, each plus the row norm; s_0 (slot L-1-k) is dropped
template <int L>
__device__ __forceinline__ double sor_list_value(const double (&list)[L], double nr, int k) {
    double acc = 0.0;
#pragma unroll
    for (int s = 0; s < L; ++s)
        if (s >= L - k) acc = __dadd_rn(acc, __dadd_rn(list[s], nr));
    return __ddiv_rn(acc, (double)k);
}

// R rows per thread, rows row0 + r * kSorThreads + tid of one sample (clamped to n - 1), against the m columns that
// start at cbase.  Leaves each row's norm in nr and its k + 1 smallest e = d - nr in the last k + 1 slots of list.
template <int L, int R>
__device__ __forceinline__ void sor_sweep_rows(const float *base, long long sp, long long sc, int n, int row0,
                                               const float *cbase, int m, int k, SorCol (&cols)[2][kSorTile],
                                               double (&nr)[R], double (&list)[R][L]) {
    const int tid = threadIdx.x;

    // row side: -2 * coordinates (exact) so that the dot product comes out as -2 * dot without a rounding of its own
    double mx[R], my[R], mz[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const long long i = min(row0 + r * kSorThreads + tid, n - 1);
        const double x = base[i * sp], y = base[i * sp + sc], z = base[i * sp + 2 * sc];
        nr[r] = sq_norm3_f64(x, y, z);
        mx[r] = -2.0 * x;
        my[r] = -2.0 * y;
        mz[r] = -2.0 * z;
        sor_list_init<L>(list[r], k);
    }

    // columns: one per thread per tile, loaded into registers a tile ahead; padding columns have norm +inf, so their
    // values (+inf or NaN) never pass the insertion gate
    const int ntiles = (m + kSorTile - 1) / kSorTile;
    float cx = 0.f, cy = 0.f, cz = 0.f;
    auto load = [&](int t) {
        const long long j = (long long)t * kSorTile + tid;
        if (j < m) {
            cx = cbase[j * sp];
            cy = cbase[j * sp + sc];
            cz = cbase[j * sp + 2 * sc];
        }
    };
    load(0);
    for (int t = 0; t < ntiles; ++t) {
        SorCol c;
        c.x = cx; c.y = cy; c.z = cz;
        c.n = t * kSorTile + tid < m ? sq_norm3_f64(c.x, c.y, c.z) : INFINITY;
        if (t * kSorTile + tid >= m) c.x = c.y = c.z = 0.0;
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
                sor_list_insert<L>(list[r], e);
            }
        }
    }
}

// L: list length (k + 1 <= L), R: rows per thread.  The front L - (k + 1) slots hold -inf and never move, so the
// last k + 1 slots are the k + 1 smallest values seen; every index below is static (no local memory).
// sor_sweep_rows above is this loop for a column range; pcd_sor_forward keeps its own copy here because routing it
// through the helper changes this kernel's register allocation and SASS.
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

// blockIdx covers (sample, column range, row tile).  PART = false (split == 1): the value of every valid row.  PART: the
// range's k + 1 smallest e of every valid row, slot-major: part[((c * B + b) * (k + 1) + s) * N + i].
// The explicit minimum of one CTA per SM lets ptxas keep every variant in registers (113 to 155, no spills); with the
// bare thread count it holds some variants to 128 registers and spills.
template <int L, int R, bool PART>
__global__ void __launch_bounds__(kSorThreads, 1) sor_len_sweep_kernel(const float *__restrict__ pc, long long sb, long long sp,
                                                                    long long sc, int B, int N, int k,
                                                                    const int32_t *__restrict__ len, int tiles_per_sample,
                                                                    int split, double *__restrict__ value,
                                                                    double *__restrict__ part) {
    __shared__ SorCol cols[2][kSorTile];
    const int g = blockIdx.x / tiles_per_sample, row0 = (blockIdx.x - g * tiles_per_sample) * (R * kSorThreads);
    const int b = g / split, c = g - b * split;
    const int n = sor_len(len, b, N);
    if (n < k + 1 || row0 >= n) return;     // the epilogue fills short samples; rows past n take no work

    // this CTA's column range: whole tiles, the valid columns spread evenly over the split
    const long long per_split = ((n + kSorTile - 1) / kSorTile + split - 1) / split * (long long)kSorTile;
    const int c0 = (int)min((long long)c * per_split, (long long)n), c1 = (int)min(c0 + per_split, (long long)n);

    const float *base = pc + (size_t)b * sb;
    double nr[R], list[R][L];
    sor_sweep_rows<L, R>(base, sp, sc, n, row0, base + c0 * sp, c1 - c0, k, cols, nr, list);
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int i = row0 + r * kSorThreads + threadIdx.x;
        if (i >= n) continue;
        if (!PART) {
            value[(size_t)b * N + i] = sor_list_value<L>(list[r], nr[r], k);
        } else {
            // list slot s >= L - 1 - k goes to entry s - (L - 1 - k)
            double *out = part + (((size_t)c * B + b) * (size_t)(k + 1) - (L - 1 - k)) * N + i;
#pragma unroll
            for (int s = 0; s < L; ++s)
                if (s >= L - 1 - k) out[(size_t)s * N] = list[r][s];
        }
    }
}

// One thread per valid row: the k + 1 smallest of the split ranges' sorted lists, then the value as the sweep forms it.
template <int L>
__global__ void __launch_bounds__(kSorMergeThreads) sor_merge_kernel(const float *__restrict__ pc, long long sb, long long sp,
                                                                     long long sc, int B, int N, int k,
                                                                     const int32_t *__restrict__ len, int row_blocks,
                                                                     int split, const double *__restrict__ part,
                                                                     double *__restrict__ value) {
    const int b = blockIdx.x / row_blocks, i = (blockIdx.x - b * row_blocks) * kSorMergeThreads + threadIdx.x;
    const int n = sor_len(len, b, N);
    if (n < k + 1 || i >= n) return;
    const float *p = pc + (size_t)b * sb + i * sp;
    const double nr = sq_norm3_f64(p[0], p[sc], p[2 * sc]);
    double list[L];
    sor_list_init<L>(list, k);
    const size_t stride = (size_t)B * (k + 1) * N;       // from one range to the next
    const double *src = part + (size_t)b * (k + 1) * N + i;
#pragma unroll 4
    for (int c = 0; c < split; ++c) {
        double e[L];
#pragma unroll
        for (int s = 0; s < L; ++s) e[s] = s <= k ? src[c * stride + (size_t)s * N] : INFINITY;
#pragma unroll
        for (int s = 0; s < L; ++s) sor_list_insert<L>(list, e[s]);
    }
    value[(size_t)b * N + i] = sor_list_value<L>(list, nr, k);
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

// The statistics of the first n rows of sample b (row stride N), the keep-mask of those rows, and the compaction of
// the kept indices into kept_idx[b, :], padded with -1 to N.
__device__ __forceinline__ void sor_epilogue_rows(int b, int n, int N, double alpha, const double *__restrict__ value,
                                                  double *__restrict__ thr_out, uint8_t *__restrict__ keep,
                                                  int32_t *__restrict__ kept_idx, int32_t *__restrict__ lengths,
                                                  double (&shd)[kSorEpiThreads / 32], int (&shi)[kSorEpiThreads / 32]) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const double *v = value + (size_t)b * N;
    uint8_t *kp = keep + (size_t)b * N;
    int32_t *out = kept_idx + (size_t)b * N;

    double s = 0.0;
    for (int i = tid; i < n; i += kSorEpiThreads) s = __dadd_rn(s, v[i]);
    const double mean = __ddiv_rn(block_sum<double, kSorEpiThreads>(s, shd), (double)n);
    double q = 0.0;
    for (int i = tid; i < n; i += kSorEpiThreads) {
        const double c = __dadd_rn(v[i], -mean);
        q = __dadd_rn(q, __dmul_rn(c, c));
    }
    const double var = __ddiv_rn(block_sum<double, kSorEpiThreads>(q, shd), (double)(n - 1));   // unbiased (torch.std)
    const double thr = __dadd_rn(mean, __dmul_rn(alpha, __dsqrt_rn(var)));

    // stable compaction, one block-wide chunk at a time: ballot within the warp, scan over the warp counts
    int count = 0;
    for (int i0 = 0; i0 < n; i0 += kSorEpiThreads) {
        const int i = i0 + tid;
        const bool kept = i < n && v[i] <= thr;
        if (i < n) kp[i] = kept ? 1 : 0;
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

__global__ void __launch_bounds__(kSorEpiThreads) sor_epilogue_kernel(int N, double alpha, const double *__restrict__ value,
                                                                      double *__restrict__ thr_out, uint8_t *__restrict__ keep,
                                                                      int32_t *__restrict__ kept_idx, int32_t *__restrict__ lengths) {
    __shared__ double shd[kSorEpiThreads / 32];
    __shared__ int shi[kSorEpiThreads / 32];
    sor_epilogue_rows(blockIdx.x, N, N, alpha, value, thr_out, keep, kept_idx, lengths, shd, shi);
}

__global__ void __launch_bounds__(kSorEpiThreads) sor_len_epilogue_kernel(int N, int k, const int32_t *__restrict__ len,
                                                                          double alpha, double *__restrict__ value,
                                                                          double *__restrict__ thr_out,
                                                                          uint8_t *__restrict__ keep,
                                                                          int32_t *__restrict__ kept_idx,
                                                                          int32_t *__restrict__ lengths) {
    __shared__ double shd[kSorEpiThreads / 32];
    __shared__ int shi[kSorEpiThreads / 32];
    const int b = blockIdx.x, n = sor_len(len, b, N);
    double *v = value + (size_t)b * N;
    uint8_t *kp = keep + (size_t)b * N;
    // rows past n, and every row of a sample without a statistic (n < k + 1: value <= NaN is false, nothing is kept)
    const int first_pad = n < k + 1 ? 0 : n;
    for (int i = first_pad + threadIdx.x; i < N; i += kSorEpiThreads) {
        v[i] = NAN;
        kp[i] = 0;
    }
    if (n < k + 1) {
        int32_t *out = kept_idx + (size_t)b * N;
        for (int i = threadIdx.x; i < N; i += kSorEpiThreads) out[i] = -1;
        if (threadIdx.x == 0) {
            thr_out[b] = NAN;
            lengths[b] = 0;
        }
        return;
    }
    sor_epilogue_rows(b, n, N, alpha, value, thr_out, keep, kept_idx, lengths, shd, shi);
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

// rows per sweep CTA for k: the (L, R) ladder of the dispatch below
static int sor_rows_per_cta(int k) { return (k + 1 <= 8 ? 4 : 2) * kSorThreads; }

static int sor_split(int B, int N, int k, int col_split) {
    if (col_split > 0) return col_split;
    const long long ctas = (long long)B * ((N + sor_rows_per_cta(k) - 1) / sor_rows_per_cta(k));
    if (ctas >= kSorTargetCtas) return 1;
    const long long want = (kSorTargetCtas + ctas - 1) / ctas;
    const long long col_tiles = (N + kSorTile - 1) / kSorTile;      // at least one tile per range
    return (int)std::min<long long>(std::min<long long>(want, col_tiles), kSorMaxSplit);
}

// one range writes the values directly: no workspace
static size_t sor_workspace(int B, int N, int k, int split) {
    return split > 1 ? (size_t)split * (size_t)B * (size_t)(k + 1) * (size_t)N * sizeof(double) : 0;
}

template <int L, int R>
static int launch_sor_len(const float *pc, int64_t sb, int64_t sp, int64_t sc, int B, int N, int k, const int32_t *len,
                          int split, double *value, double *part, cudaStream_t st) {
    const int tiles = (N + R * kSorThreads - 1) / (R * kSorThreads);
    const long long grid = (long long)B * split * tiles;
    if (grid > 2147483647LL) {
        set_error("pcd_sor_forward_len: B * col_split * ceil(N / %d) (%lld) exceeds the grid limit", R * kSorThreads, grid);
        return PCD_ERR_ARG;
    }
    if (split == 1)
        sor_len_sweep_kernel<L, R, false><<<(unsigned)grid, kSorThreads, 0, st>>>(pc, sb, sp, sc, B, N, k, len, tiles, 1, value, part);
    else
        sor_len_sweep_kernel<L, R, true><<<(unsigned)grid, kSorThreads, 0, st>>>(pc, sb, sp, sc, B, N, k, len, tiles, split, value, part);
    PCD_CUDA_CHECK(cudaGetLastError());
    if (split > 1) {
        const int row_blocks = (N + kSorMergeThreads - 1) / kSorMergeThreads;      // B * row_blocks <= grid above
        sor_merge_kernel<L><<<(unsigned)(B * row_blocks), kSorMergeThreads, 0, st>>>(pc, sb, sp, sc, B, N, k, len, row_blocks,
                                                                                    split, part, value);
        PCD_CUDA_CHECK(cudaGetLastError());
    }
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

extern "C" size_t pcd_sor_workspace_bytes(int B, int N, int k, int col_split) {
    if (B <= 0 || N <= 0 || k < 1 || k > PCD_SOR_MAX_K || col_split < 0) return 0;
    return sor_workspace(B, N, k, sor_split(B, N, k, col_split));
}

extern "C" int pcd_sor_forward_len(const float *pc, int64_t sb, int64_t sp, int64_t sc, int B, int N, int k, double alpha,
                                   const int32_t *len, int col_split, double *value, double *threshold, uint8_t *keep,
                                   int32_t *kept_idx, int32_t *lengths, void *workspace, size_t workspace_bytes,
                                   void *stream) {
    if (!pc || !value || !threshold || !keep || !kept_idx || !lengths || B <= 0 || N <= 0 || k < 1 || k > PCD_SOR_MAX_K ||
        !isfinite(alpha) || col_split < 0) {
        set_error("pcd_sor_forward_len: bad argument (need B, N >= 1, 1 <= k <= %d, finite alpha, col_split >= 0, "
                  "no NULL pointer)", PCD_SOR_MAX_K);
        return PCD_ERR_ARG;
    }
    const int split = sor_split(B, N, k, col_split);
    const size_t need = sor_workspace(B, N, k, split);
    if (need && (!workspace || workspace_bytes < need)) {
        set_error("pcd_sor_forward_len: workspace of %zu bytes, %zu needed", workspace_bytes, need);
        return PCD_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    double *part = (double *)workspace;
    const int rc = k + 1 <= 4   ? launch_sor_len<4, 4>(pc, sb, sp, sc, B, N, k, len, split, value, part, st)
                   : k + 1 <= 8 ? launch_sor_len<8, 4>(pc, sb, sp, sc, B, N, k, len, split, value, part, st)
                                : launch_sor_len<16, 2>(pc, sb, sp, sc, B, N, k, len, split, value, part, st);
    if (rc != PCD_OK) return rc;
    sor_len_epilogue_kernel<<<B, kSorEpiThreads, 0, st>>>(N, k, len, alpha, value, threshold, keep, kept_idx, lengths);
    PCD_CUDA_CHECK(cudaGetLastError());
    return PCD_OK;
}
