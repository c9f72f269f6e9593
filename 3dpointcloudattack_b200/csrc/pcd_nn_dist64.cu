// pcd_nn_dist64.cu -- exact float64 nearest-neighbour distances between the clouds of a batch, both directions, with the
// per-sample Chamfer / Hausdorff reductions, for clouds of unequal valid sizes, sm_100a.
//
// utils/dis_utils_numpy.py:13-38 builds the full N x M float64 matrix with scipy's distance_matrix, one cloud at a time
// on the host.  Here the matrix never exists:
//   nnd64_sweep_kernel     R rows per thread keep a running (min, arg) of s over one range of the other cloud's valid
//                          columns, which stream through shared memory as double-buffered float64 tiles.  blockIdx covers
//                          (sample, column range, direction, row tile); each CTA writes its partial pairs to the workspace.
//   nnd64_epilogue_kernel  one CTA per (sample, direction): merges the partials of the column ranges, writes the per-point
//                          outputs and reduces them in a fixed order.
// The arithmetic is the contract of pcd_nn_dist64_forward in include/pcdist.h.
#include <math.h>

#include <algorithm>

#include "pcd_common.cuh"

namespace pcd {

constexpr int kNndThreads = 128;
constexpr int kNndRows = 4;                          // rows per thread
constexpr int kNndRowTile = kNndRows * kNndThreads;
constexpr int kNndColTile = kNndThreads;             // each thread stages one column of every tile
constexpr int kNndEpiThreads = 512;
// Column split: while B * row tiles (both directions) is below about two waves of a 148-SM B200 at four CTAs per SM,
// a row tile's columns are spread over several CTAs.  A fixed target (no device query) keeps the workspace size a
// function of the shape alone.
constexpr long long kNndTargetCtas = 2 * 148 * 4;
constexpr int kNndMaxSplit = 64;

struct __align__(32) NndCol {
    double x, y, z, pad;
};

struct NndArgs {
    const float *p[2];                  // cloud 0 = a, cloud 1 = b
    long long sb[2], sp[2], sc[2];
    const int32_t *len[2];
    int n[2];                           // N, M
    int tiles[2];                       // row tiles of direction 0 (rows of a) and 1 (rows of b)
    int B, split;
    double *part_val;                   // [split][B][N + M]: a rows first, then b rows
    int32_t *part_arg;
};

__device__ __forceinline__ int nnd_len(const int32_t *len, int b, int n) { return len ? min(max(len[b], 0), n) : n; }

// s = ((dx*dx) + (dy*dy)) + (dz*dz), dx = column - row: no contraction into FMA
__device__ __forceinline__ double nnd_pair(double rx, double ry, double rz, const NndCol &q) {
    const double dx = __dsub_rn(q.x, rx), dy = __dsub_rn(q.y, ry), dz = __dsub_rn(q.z, rz);
    return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}

// (v, i) comes before (w, j) for numpy's argmin: a NaN first, else the smaller value, equal values and NaN pairs by the
// lower index.  An empty pair (index < 0) comes after everything.  A total order, so the merge is associative and
// commutative.
__device__ __forceinline__ bool nnd_min_before(double v, int i, double w, int j) {
    if (i < 0 || j < 0) return j < 0 && i >= 0;
    const bool vn = isnan(v), wn = isnan(w);
    if (vn != wn) return vn;
    if (!vn && v != w) return v < w;
    return i < j;
}
// the same for argmax: a NaN first, else the larger value, then the lower index
__device__ __forceinline__ bool nnd_max_before(double v, int i, double w, int j) {
    if (i < 0 || j < 0) return j < 0 && i >= 0;
    const bool vn = isnan(v), wn = isnan(w);
    if (vn != wn) return vn;
    if (!vn && v != w) return v > w;
    return i < j;
}

// One staged tile, columns ascending.  FINITE: the CTA's rows and this tile's columns are all finite, so s is finite and
// a strict < keeps the first of equal minima.  Otherwise the first column always enters, a NaN sticks, and the first NaN
// replaces a number.
template <bool FINITE>
__device__ __forceinline__ void nnd_tile(const NndCol *__restrict__ tile, int nj, int j0, const double (&rx)[kNndRows],
                                         const double (&ry)[kNndRows], const double (&rz)[kNndRows],
                                         double (&cur)[kNndRows], int (&arg)[kNndRows]) {
#pragma unroll 4
    for (int jj = 0; jj < nj; ++jj) {
        const NndCol q = tile[jj];
#pragma unroll
        for (int r = 0; r < kNndRows; ++r) {
            const double s = nnd_pair(rx[r], ry[r], rz[r], q);
            const bool take = FINITE ? s < cur[r] : arg[r] < 0 || (!isnan(cur[r]) && (s < cur[r] || isnan(s)));
            if (take) {
                cur[r] = s;
                arg[r] = j0 + jj;
            }
        }
    }
}

__global__ void __launch_bounds__(kNndThreads) nnd64_sweep_kernel(const NndArgs p) {
    __shared__ NndCol cols[2][kNndColTile];
    const int per = p.tiles[0] + p.tiles[1];
    const int g = blockIdx.x / per, t = blockIdx.x - g * per;
    const int b = g / p.split, c = g - b * p.split;
    const int dir = t < p.tiles[0] ? 0 : 1, row0 = (dir ? t - p.tiles[0] : t) * kNndRowTile;
    // every p.x[dir] is a select: a dynamic index into the parameter struct would copy it to local memory
    const int rlen = dir ? nnd_len(p.len[1], b, p.n[1]) : nnd_len(p.len[0], b, p.n[0]);
    if (row0 >= rlen) return;           // rows past the length take no partial
    const int tid = threadIdx.x;

    // this CTA's column range: whole tiles, the valid columns spread evenly over the split
    const int clen = dir ? nnd_len(p.len[0], b, p.n[0]) : nnd_len(p.len[1], b, p.n[1]);
    const long long per_split = ((clen + kNndColTile - 1) / kNndColTile + p.split - 1) / p.split * (long long)kNndColTile;
    const int c0 = (int)min((long long)c * per_split, (long long)clen), c1 = (int)min(c0 + per_split, (long long)clen);

    const float *rp = dir ? p.p[1] + (size_t)b * p.sb[1] : p.p[0] + (size_t)b * p.sb[0];
    const long long rsp = dir ? p.sp[1] : p.sp[0], rsc = dir ? p.sc[1] : p.sc[0];
    double rx[kNndRows], ry[kNndRows], rz[kNndRows], cur[kNndRows];
    int arg[kNndRows];
    bool nonfinite = false;
#pragma unroll
    for (int r = 0; r < kNndRows; ++r) {
        const long long i = min(row0 + r * kNndThreads + tid, rlen - 1);
        rx[r] = rp[i * rsp];
        ry[r] = rp[i * rsp + rsc];
        rz[r] = rp[i * rsp + 2 * rsc];
        nonfinite |= !(isfinite(rx[r]) && isfinite(ry[r]) && isfinite(rz[r]));
        cur[r] = INFINITY;
        arg[r] = -1;
    }
    const bool rows_nonfinite = __syncthreads_or(nonfinite);

    const float *cp = dir ? p.p[0] + (size_t)b * p.sb[0] : p.p[1] + (size_t)b * p.sb[1];
    const long long csp = dir ? p.sp[0] : p.sp[1], csc = dir ? p.sc[0] : p.sc[1];
    const int ntiles = (c1 - c0 + kNndColTile - 1) / kNndColTile;
    float fx = 0.f, fy = 0.f, fz = 0.f;
    auto load = [&](int k) {
        const long long j = c0 + (long long)k * kNndColTile + tid;
        if (j < c1) {
            fx = cp[j * csp];
            fy = cp[j * csp + csc];
            fz = cp[j * csp + 2 * csc];
        }
    };
    load(0);
    for (int k = 0; k < ntiles; ++k) {
        const int j0 = c0 + k * kNndColTile, nj = min(kNndColTile, c1 - j0);
        const bool bad = tid < nj && !(isfinite(fx) && isfinite(fy) && isfinite(fz));
        NndCol q;
        q.x = fx; q.y = fy; q.z = fz; q.pad = 0.0;
        cols[k & 1][tid] = q;           // the buffer last read two tiles ago: every thread has passed a barrier since
        const bool finite = !__syncthreads_or(bad) && !rows_nonfinite;
        if (k + 1 < ntiles) load(k + 1);
        if (finite)
            nnd_tile<true>(cols[k & 1], nj, j0, rx, ry, rz, cur, arg);
        else
            nnd_tile<false>(cols[k & 1], nj, j0, rx, ry, rz, cur, arg);
    }

    const size_t base = ((size_t)c * p.B + b) * ((size_t)p.n[0] + p.n[1]) + (dir ? p.n[0] : 0);
#pragma unroll
    for (int r = 0; r < kNndRows; ++r) {
        const int i = row0 + r * kNndThreads + tid;
        if (i < rlen) {
            p.part_val[base + i] = cur[r];
            p.part_arg[base + i] = arg[r];
        }
    }
}

__global__ void __launch_bounds__(kNndEpiThreads) nnd64_epilogue_kernel(const NndArgs p, double *__restrict__ a_min,
                                                                        int32_t *__restrict__ a_arg, double *__restrict__ b_min,
                                                                        int32_t *__restrict__ b_arg, double *__restrict__ stats,
                                                                        int32_t *__restrict__ argmax) {
    constexpr int W = kNndEpiThreads / 32;
    __shared__ double shd[W];
    __shared__ int shi[W];
    const int b = blockIdx.x >> 1, dir = blockIdx.x & 1, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n = dir ? p.n[1] : p.n[0], rlen = nnd_len(dir ? p.len[1] : p.len[0], b, n);
    double *vmin = (dir ? b_min : a_min) + (size_t)b * n;
    int32_t *varg = (dir ? b_arg : a_arg) + (size_t)b * n;
    const size_t pstride = (size_t)p.B * ((size_t)p.n[0] + p.n[1]);
    const size_t pbase = (size_t)b * ((size_t)p.n[0] + p.n[1]) + (dir ? p.n[0] : 0);

    double sum = 0.0, sum_sqrt = 0.0, mx = NAN;
    int mi = -1;
    for (int i = tid; i < n; i += kNndEpiThreads) {
        double v = NAN;
        int a = -1;
        if (i < rlen) {
            for (int c = 0; c < p.split; ++c) {
                const double w = p.part_val[c * pstride + pbase + i];
                const int j = p.part_arg[c * pstride + pbase + i];
                if (nnd_min_before(w, j, v, a)) {
                    v = w;
                    a = j;
                }
            }
            if (a < 0) v = NAN;         // the other side has length 0
            sum = __dadd_rn(sum, v);
            sum_sqrt = __dadd_rn(sum_sqrt, __dsqrt_rn(v));
            if (nnd_max_before(v, i, mx, mi)) {
                mx = v;
                mi = i;
            }
        }
        vmin[i] = v;
        varg[i] = a;
    }
    sum = block_sum<double, kNndEpiThreads>(sum, shd);
    sum_sqrt = block_sum<double, kNndEpiThreads>(sum_sqrt, shd);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double w = __shfl_xor_sync(0xffffffffu, mx, o);
        const int j = __shfl_xor_sync(0xffffffffu, mi, o);
        if (nnd_max_before(w, j, mx, mi)) {
            mx = w;
            mi = j;
        }
    }
    __syncthreads();                    // shd is still read by block_sum's last step
    if (lane == 0) {
        shd[warp] = mx;
        shi[warp] = mi;
    }
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < W; ++w)
            if (nnd_max_before(shd[w], shi[w], mx, mi)) {
                mx = shd[w];
                mi = shi[w];
            }
        double *st = stats + ((size_t)dir * p.B + b) * 4;
        const bool empty = rlen == 0;
        st[0] = empty ? NAN : __ddiv_rn(sum, (double)rlen);
        st[1] = empty ? NAN : __ddiv_rn(sum_sqrt, (double)rlen);
        st[2] = mx;                     // NaN and -1 when empty
        st[3] = __dsqrt_rn(mx);
        argmax[(size_t)dir * p.B + b] = mi;
    }
}

static int nnd_row_tiles(int n) { return (n + kNndRowTile - 1) / kNndRowTile; }

static int nnd_split(int B, int N, int M, int col_split) {
    if (col_split > 0) return col_split;
    const long long ctas = (long long)B * (nnd_row_tiles(N) + nnd_row_tiles(M));
    if (ctas >= kNndTargetCtas) return 1;
    const long long want = (kNndTargetCtas + ctas - 1) / ctas;
    const long long col_tiles = ((N > M ? N : M) + kNndColTile - 1) / kNndColTile;      // at least one tile per range
    return (int)std::min<long long>(std::min<long long>(want, col_tiles), kNndMaxSplit);
}

static size_t nnd_workspace(int B, int N, int M, int split) {
    return (size_t)split * (size_t)B * ((size_t)N + (size_t)M) * (sizeof(double) + sizeof(int32_t));
}

}  // namespace pcd

using namespace pcd;

extern "C" size_t pcd_nn_dist64_workspace_bytes(int B, int N, int M, int col_split) {
    if (B <= 0 || N <= 0 || M <= 0 || col_split < 0) return 0;
    return nnd_workspace(B, N, M, nnd_split(B, N, M, col_split));
}

extern "C" int pcd_nn_dist64_forward(const float *a, int64_t sab, int64_t sap, int64_t sac, const float *b, int64_t sbb,
                                     int64_t sbp, int64_t sbc, int B, int N, int M, const int32_t *a_len,
                                     const int32_t *b_len, int col_split, double *a_min, int32_t *a_arg, double *b_min,
                                     int32_t *b_arg, double *stats, int32_t *argmax, void *workspace,
                                     size_t workspace_bytes, void *stream) {
    if (!a || !b || !a_min || !a_arg || !b_min || !b_arg || !stats || !argmax || B <= 0 || N <= 0 || M <= 0 ||
        col_split < 0) {
        set_error("pcd_nn_dist64_forward: bad argument (need B, N, M >= 1, col_split >= 0, no NULL pointer)");
        return PCD_ERR_ARG;
    }
    NndArgs p;
    p.split = nnd_split(B, N, M, col_split);
    p.tiles[0] = nnd_row_tiles(N);
    p.tiles[1] = nnd_row_tiles(M);
    const long long grid = (long long)B * p.split * (p.tiles[0] + p.tiles[1]);
    if (grid > 2147483647LL || 2LL * B > 2147483647LL) {
        set_error("pcd_nn_dist64_forward: B * col_split * row tiles (%lld) exceeds the grid limit", grid);
        return PCD_ERR_ARG;
    }
    const size_t need = nnd_workspace(B, N, M, p.split);
    if (!workspace || workspace_bytes < need) {
        set_error("pcd_nn_dist64_forward: workspace of %zu bytes, %zu needed", workspace_bytes, need);
        return PCD_ERR_WORKSPACE;
    }
    p.p[0] = a; p.sb[0] = sab; p.sp[0] = sap; p.sc[0] = sac; p.len[0] = a_len; p.n[0] = N;
    p.p[1] = b; p.sb[1] = sbb; p.sp[1] = sbp; p.sc[1] = sbc; p.len[1] = b_len; p.n[1] = M;
    p.B = B;
    p.part_val = (double *)workspace;
    p.part_arg = (int32_t *)(p.part_val + (size_t)p.split * B * ((size_t)N + M));
    cudaStream_t st = (cudaStream_t)stream;
    nnd64_sweep_kernel<<<(unsigned)grid, kNndThreads, 0, st>>>(p);
    PCD_CUDA_CHECK(cudaGetLastError());
    nnd64_epilogue_kernel<<<(unsigned)(2 * B), kNndEpiThreads, 0, st>>>(p, a_min, a_arg, b_min, b_arg, stats, argmax);
    PCD_CUDA_CHECK(cudaGetLastError());
    return PCD_OK;
}
