// pcd_siadv.cu -- the tangent-plane step of the SI-Adv shape-invariant attack as ONE launch, sm_100a.
//
// SI-Adv's PointCloudAttack.shape_invariant_ifgm (attack/SIadv/SIadv_attack.py: get_spin_axis_matrix,
// get_transformed_point_cloud, get_original_point_cloud) builds a 3x3 spin-axis frame per point from its normal, moves
// the point along the part of the gradient that lies in its tangent plane, normalised over the whole sample, maps it
// back and clips the perturbation: about 40 small torch ops per iteration.  Here one thread owns P consecutive points and
// keeps them in registers across the two sample-wide reductions (the gradient norm, then the per-axis perturbation
// norms of the clip), so every input is read once and pc is written once.
//
// A sample is reduced over an aligned power-of-two tree of its points (pcd_si_step in include/pcdist.h).  The summands
// are squares, so padding the block with +0 leaves every node's bits unchanged: a CTA reduces its points in registers,
// then over lanes by an xor butterfly of increasing stride, then over warps; the S CTAs of a cluster that share the sample
// (S = 1 when the batch alone fills the GPU) read each other's totals through distributed shared memory and finish the
// tree in rank order.  A sample's bits therefore depend on its inputs and N only.
// Every operation is rounded on its own (the file is compiled with --fmad=false and uses the _rn intrinsics).
#include <cooperative_groups.h>

#include <cmath>

#include "pcd_common.cuh"

namespace cg = cooperative_groups;

namespace pcd {

constexpr int kSiMaxThreads = 256;
constexpr int kSiMaxSplit = 16;

struct SiCloud {
    const float *p;
    long long sb, sp, sc;
    __device__ __forceinline__ float at(int b, int i, int c) const { return p[b * sb + i * sp + c * sc]; }
};

// u = the spin-axis rows of normal (x, y, z) (get_spin_axis_matrix)
__device__ __forceinline__ void spin_axis(float x, float y, float z, float u[3][3]) {
    const float zz = __fmul_rn(z, z);
    if (fabsf(__fsub_rn(zz, 1.f)) < 1e-4f) {
        const float r = 0.70710677f, s2 = 1.41421354f;              // fp32(1/sqrt(2)), fp32(sqrt(2))
        const float w = __fdiv_rn(z, s2);
        u[0][0] = r;   u[0][1] = -r;  u[0][2] = 0.f;
        u[1][0] = w;   u[1][1] = w;   u[1][2] = 0.f;
        u[2][0] = 0.f; u[2][1] = 0.f; u[2][2] = z;
    } else {
        const float den = __fsqrt_rn(__fsub_rn(1.f, zz));
        u[0][0] = __fdiv_rn(y, den);                 u[0][1] = __fdiv_rn(-x, den);               u[0][2] = 0.f;
        u[1][0] = __fdiv_rn(__fmul_rn(x, z), den);   u[1][1] = __fdiv_rn(__fmul_rn(y, z), den);  u[1][2] = -den;
        u[2][0] = x;                                 u[2][1] = y;                                u[2][2] = z;
    }
}
__device__ __forceinline__ float dot3(float a0, float a1, float a2, float b0, float b1, float b2) {
    return __fadd_rn(__fadd_rn(__fmul_rn(a0, b0), __fmul_rn(a1, b1)), __fmul_rn(a2, b2));
}

// Pairwise tree over a thread's P values, in point order
template <int P>
__device__ __forceinline__ float tree_local(const float (&v)[P]) {
    float t[P];
#pragma unroll
    for (int k = 0; k < P; ++k) t[k] = v[k];
#pragma unroll
    for (int w = 1; w < P; w *= 2) {
#pragma unroll
        for (int k = 0; k < P; k += 2 * w) t[k] = __fadd_rn(t[k], t[k + w]);
    }
    return t[0];
}
// The lanes' values in lane order (lane l holds the l-th aligned block of the warp): the butterfly pairs lane l with l ^ 1
// first, so every lane ends with the tree total (addition is commutative, so both partners round alike).
__device__ __forceinline__ float tree_warp(float v) {
#pragma unroll
    for (int o = 1; o < 32; o *= 2) v = __fadd_rn(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
// Pairwise tree over n (a power of two, <= kSiMaxSplit) values read by get(i), in index order
template <typename Get>
__device__ __forceinline__ float tree_n(int n, Get get) {
    float t[kSiMaxSplit];
#pragma unroll
    for (int k = 0; k < kSiMaxSplit; ++k) t[k] = k < n ? get(k) : 0.f;
#pragma unroll
    for (int w = 1; w < kSiMaxSplit; w *= 2) {
#pragma unroll
        for (int k = 0; k < kSiMaxSplit; k += 2 * w) t[k] = __fadd_rn(t[k], t[k + w]);
    }
    return t[0];
}

// Sample-wide sums of NV values per thread: the CTA's tree total lands in cta_tot[0..NV), then the cluster's tree over the
// S CTA totals is returned in every thread.  warp_sh: NV x 8 floats.
template <int NV>
__device__ __forceinline__ void sample_sum(const float (&v)[NV], float (&out)[NV], float *warp_sh, float *cta_tot, int S) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, W = blockDim.x >> 5;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        const float w = tree_warp(v[j]);
        if (lane == 0) warp_sh[j * 8 + warp] = w;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
        for (int j = 0; j < NV; ++j) cta_tot[j] = tree_n(W, [&](int k) { return warp_sh[j * 8 + k]; });
    }
    if (S == 1) {
        __syncthreads();
#pragma unroll
        for (int j = 0; j < NV; ++j) out[j] = cta_tot[j];
        return;
    }
    cg::cluster_group cluster = cg::this_cluster();
    cluster.sync();                                   // every CTA's total is written and visible cluster-wide
#pragma unroll
    for (int j = 0; j < NV; ++j) out[j] = tree_n(S, [&](int r) { return *cluster.map_shared_rank(cta_tot + j, r); });
}

// One sample per S consecutive CTAs (a cluster of S when S > 1); CTA rank r holds points [r * T * P, (r + 1) * T * P),
// thread t of it P consecutive ones.  Points at or past N are padding: they read nothing and add +0.
template <int P>
__global__ void __launch_bounds__(kSiMaxThreads)
si_step_kernel(float *__restrict__ pc, long long sb, long long sp, long long sc, SiCloud ori, SiCloud nrm, SiCloud grd,
               int N, int S, float a, float eps, float *__restrict__ gnorm) {
    __shared__ float warp_sh[3 * 8];
    __shared__ float tot1[1], tot2[3];
    const int b = blockIdx.x / S, rank = blockIdx.x - b * S;
    const int i0 = (rank * blockDim.x + threadIdx.x) * P;
    const SiCloud pcr{pc, sb, sp, sc};

    float n[P][3], c[P], pp[P][3], g0[P], g1[P], sq[P];
#pragma unroll
    for (int k = 0; k < P; ++k) {
        const int i = i0 + k;
        sq[k] = 0.f;
        if (i >= N) continue;
        float p[3], g[3], u[3][3];
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            p[r] = pcr.at(b, i, r);
            n[k][r] = nrm.at(b, i, r);
            g[r] = grd.at(b, i, r);
        }
        c[k] = dot3(p[0], p[1], p[2], n[k][0], n[k][1], n[k][2]);
        float q[3];
#pragma unroll
        for (int r = 0; r < 3; ++r) q[r] = __fadd_rn(p[r], __fmul_rn(c[k], n[k][r]));
        spin_axis(n[k][0], n[k][1], n[k][2], u);
#pragma unroll
        for (int r = 0; r < 3; ++r) pp[k][r] = dot3(u[r][0], u[r][1], u[r][2], q[0], q[1], q[2]);
        g0[k] = dot3(u[0][0], u[0][1], u[0][2], g[0], g[1], g[2]);
        g1[k] = dot3(u[1][0], u[1][1], u[1][2], g[0], g[1], g[2]);
        sq[k] = __fadd_rn(__fmul_rn(g0[k], g0[k]), __fmul_rn(g1[k], g1[k]));
    }
    float s1[1] = {tree_local(sq)}, r1[1];
    sample_sum<1>(s1, r1, warp_sh, tot1, S);
    const float norm = __fsqrt_rn(r1[0]);
    const float den = __fadd_rn(norm, 1e-9f);

    float d[P][3], o[P][3], sx[P], sy[P], sz[P];
#pragma unroll
    for (int k = 0; k < P; ++k) {
        const int i = i0 + k;
        sx[k] = sy[k] = sz[k] = 0.f;
        if (i >= N) continue;
        float u[3][3];
        spin_axis(n[k][0], n[k][1], n[k][2], u);
        const float q0 = __fsub_rn(pp[k][0], __fdiv_rn(__fmul_rn(a, g0[k]), den));
        const float q1 = __fsub_rn(pp[k][1], __fdiv_rn(__fmul_rn(a, g1[k]), den));
        const float q2 = __fsub_rn(pp[k][2], __fdiv_rn(__fmul_rn(a, 0.f), den));
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const float pn = __fsub_rn(dot3(u[0][r], u[1][r], u[2][r], q0, q1, q2), __fmul_rn(c[k], n[k][r]));
            o[k][r] = ori.at(b, i, r);
            d[k][r] = __fsub_rn(pn, o[k][r]);
        }
        sx[k] = __fmul_rn(d[k][0], d[k][0]);
        sy[k] = __fmul_rn(d[k][1], d[k][1]);
        sz[k] = __fmul_rn(d[k][2], d[k][2]);
    }
    float s2[3] = {tree_local(sx), tree_local(sy), tree_local(sz)}, r2[3];
    sample_sum<3>(s2, r2, warp_sh, tot2, S);
    float scale[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const float s = __fdiv_rn(eps, __fadd_rn(__fsqrt_rn(r2[r]), 1e-9f));
        scale[r] = s > 1.f ? 1.f : s;                // NaN stays NaN
    }
#pragma unroll
    for (int k = 0; k < P; ++k) {
        const int i = i0 + k;
        if (i >= N) continue;
#pragma unroll
        for (int r = 0; r < 3; ++r) pc[b * sb + i * sp + r * sc] = __fadd_rn(o[k][r], __fmul_rn(d[k][r], scale[r]));
    }
    if (gnorm && rank == 0 && threadIdx.x == 0) gnorm[b] = norm;
    if (S > 1) cg::this_cluster().sync();            // no CTA leaves while another still reads its totals
}

// Largest cluster size the device schedules for the step (8 is portable; 16 needs the non-portable attribute on every
// instantiation), once per device.  The P = 8 form asks for the most registers, so its answer holds for the others.
static int max_split() {
    static PerDeviceInt cache = {};
    const int dev = current_device();
    if (dev < 0) return 8;
    if (cache.v[dev]) return cache.v[dev];
    int best = 8;
    if (cudaFuncSetAttribute(si_step_kernel<1>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess &&
        cudaFuncSetAttribute(si_step_kernel<2>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess &&
        cudaFuncSetAttribute(si_step_kernel<4>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess &&
        cudaFuncSetAttribute(si_step_kernel<8>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(kSiMaxSplit);
        cfg.blockDim = dim3(kSiMaxThreads);
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = kSiMaxSplit;
        attr[0].val.clusterDim.y = attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        int clusters = 0;
        if (cudaOccupancyMaxActiveClusters(&clusters, si_step_kernel<8>, &cfg) == cudaSuccess && clusters > 0)
            best = kSiMaxSplit;
    }
    cudaGetLastError();                              // a refused query is an answer, not a pending error
    cache.v[dev] = best;
    return best;
}

template <int P>
static int launch_si(int B, int S, int T, float *pc, long long sb, long long sp, long long sc, SiCloud ori, SiCloud nrm,
                     SiCloud grd, int N, float a, float eps, float *gnorm, cudaStream_t st) {
    const auto kernel = si_step_kernel<P>;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)((long long)B * S));
    cfg.blockDim = dim3(T);
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = S;
    attr[0].val.clusterDim.y = attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = S > 1 ? 1 : 0;
    PCD_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kernel, pc, sb, sp, sc, ori, nrm, grd, N, S, a, eps, gnorm));
    return PCD_OK;
}

// ------------------------------------------------------------------------------------------------------------------------
// SI-Adv's query-based attack (shape_invariant_query_attack; pcd_si_sensitivity and pcd_si_query_round in include/pcdist.h).
// The frames, the tangent-plane move and the clip are the step kernel's, with the same rounding.

// Per point: the surrogate's gradient in the frame, its tangent length s and unit direction (one thread per point)
__global__ void __launch_bounds__(256)
si_sensitivity_kernel(SiCloud grd, SiCloud nrm, int B, int N, float *__restrict__ s, float *__restrict__ dir) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= (long long)B * N) return;
    const int b = (int)(k / N), i = (int)(k - (long long)b * N);
    float g[3], u[3][3];
#pragma unroll
    for (int r = 0; r < 3; ++r) g[r] = grd.at(b, i, r);
    spin_axis(nrm.at(b, i, 0), nrm.at(b, i, 1), nrm.at(b, i, 2), u);
    const float gx = dot3(u[0][0], u[0][1], u[0][2], g[0], g[1], g[2]);
    const float gy = dot3(u[1][0], u[1][1], u[1][2], g[0], g[1], g[2]);
    float v = __fsqrt_rn(__fadd_rn(__fmul_rn(gx, gx), __fmul_rn(gy, gy))), dx = 0.f, dy = 0.f;
    if (isnan(v)) {
        v = -1.f;                                     // ranks last and moves nothing
    } else {
        const float den = __fadd_rn(v, 1e-16f);
        dx = __fdiv_rn(gx, den);
        dy = __fdiv_rn(gy, den);
    }
    s[k] = v;
    dir[2 * k] = dx;
    dir[2 * k + 1] = dy;
}

struct SiCloudOut {
    float *p;
    long long sb, sp, sc;
    __device__ __forceinline__ float &at(int b, int i, int c) const { return p[b * sb + i * sp + c * sc]; }
};

constexpr int kSqThreads = 256;
constexpr int kSqMaxBlocks = PCD_SI_MAX_N / 32;      // 32-point block totals per axis
enum : int { kSqIdle = 0, kSqStep = 1, kSqTake = 2, kSqDone = 4 };

// Point i of the next trial before the clip: src's point, and for the chosen one the step's transform, a move of
// sigma * a * (dx, dy) in the tangent plane and the explicit inverse transform
__device__ __forceinline__ void sq_point(const SiCloudOut &src, const SiCloud &nrm, int b, int i, int moved, float sa,
                                         float dx, float dy, float (&p)[3]) {
#pragma unroll
    for (int r = 0; r < 3; ++r) p[r] = src.at(b, i, r);
    if (i != moved) return;
    float n[3], u[3][3], t[3], q[3], pp[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) n[r] = nrm.at(b, i, r);
    const float c = dot3(p[0], p[1], p[2], n[0], n[1], n[2]);
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        t[r] = __fmul_rn(c, n[r]);
        q[r] = __fadd_rn(p[r], t[r]);
    }
    spin_axis(n[0], n[1], n[2], u);
#pragma unroll
    for (int r = 0; r < 3; ++r) pp[r] = dot3(u[r][0], u[r][1], u[r][2], q[0], q[1], q[2]);
    pp[0] = __fadd_rn(pp[0], __fmul_rn(sa, dx));
    pp[1] = __fadd_rn(pp[1], __fmul_rn(sa, dy));
#pragma unroll
    for (int r = 0; r < 3; ++r) p[r] = __fsub_rn(dot3(u[0][r], u[1][r], u[2][r], pp[0], pp[1], pp[2]), t[r]);
}

// One CTA per sample.  Warp 0 scores the logits row and lane 0 makes the decision; then the CTA writes the next trial.
// Thread t owns points t, t + T, ...: a warp's 32 consecutive points are summed by the lane butterfly, the 32-point
// block totals by an in-place aligned tree in shared memory, so the clip's norms follow the fixed tree of pcd_si_step.
__global__ void __launch_bounds__(kSqThreads)
si_query_round_kernel(const float *__restrict__ logits, long long l_sb, long long l_sc, int C,
                      const long long *__restrict__ target, SiCloud ori, SiCloud nrm, const int *__restrict__ order,
                      const float *__restrict__ dir, SiCloudOut cloud, SiCloudOut trial, int *__restrict__ state,
                      float *__restrict__ best, int N, float a, float eps, int max_query, int targeted,
                      int *__restrict__ active) {
    __shared__ int dec[3];                            // mode, moved point, sigma of the next trial
    __shared__ float tot[3][kSqMaxBlocks];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, T = blockDim.x;
    if (tid < 32) {
        int *st = state + 4 * (long long)b;
        int mode = kSqIdle, moved = -1, sigma = st[0];
        if (st[3] == 0) {
            const long long y = target[b];
            const bool y_ok = y >= 0 && y < C;
            const float *row = logits + b * l_sb;
            bool nan = false;
            float other = -10000.f, top = -INFINITY;  // other: the max of (1 - onehot) * logits - onehot * 10000
            int arg = 0x7fffffff;
            for (int j = lane; j < C; j += 32) {
                const float v = row[j * l_sc];
                nan |= isnan(v);
                if (j != y) other = fmaxf(other, v);
                if (v > top) top = v, arg = j;
            }
#pragma unroll
            for (int o = 1; o < 32; o *= 2) {         // max and first arg-max are exact: any combining order agrees
                nan |= __shfl_xor_sync(0xffffffffu, (int)nan, o) != 0;
                other = fmaxf(other, __shfl_xor_sync(0xffffffffu, other, o));
                const float tv = __shfl_xor_sync(0xffffffffu, top, o);
                const int ta = __shfl_xor_sync(0xffffffffu, arg, o);
                if (tv > top || (tv == top && ta < arg)) top = tv, arg = ta;
            }
            if (lane == 0) {
                const float real = y_ok ? row[y * l_sc] : 0.f;
                const float margin = targeted ? __fsub_rn(other, real) : __fsub_rn(real, other);
                const bool valid = y_ok && !nan && isfinite(margin);
                const bool success = valid && (targeted ? arg == y : arg != y);
                int cur = st[1], q = st[2] + 1, status = 0;
                bool take = false;
                if (q == 1) {                         // round 0: the trial is the cloud itself
                    best[b] = margin;
                    if (success) status = 1, take = true;
                } else if (success) {
                    status = 1, take = true;
                } else if (valid && margin < best[b]) {
                    best[b] = margin;
                    take = true, cur += 1, sigma = -1;
                } else if (sigma == -1) {
                    sigma = 1;
                } else {
                    cur += 1, sigma = -1;
                }
                if (status == 0 && q >= max_query) status = 2;
                st[0] = sigma, st[1] = cur, st[2] = q, st[3] = status;
                if (status != 0 && active) atomicSub(active, 1);
                mode = (take ? kSqTake : 0) | (status != 0 ? kSqDone : kSqStep);
                if (status == 0) {
                    moved = order[(long long)b * N + (int)((unsigned)cur % (unsigned)N)];
                    if (moved < 0 || moved >= N) moved = -1;
                }
                dec[0] = mode, dec[1] = moved, dec[2] = sigma;
            }
        } else if (lane == 0) {
            dec[0] = kSqIdle;
        }
    }
    __syncthreads();
    const int mode = dec[0], moved = dec[1];
    if (mode == kSqIdle) return;
    const SiCloudOut src = (mode & kSqTake) ? trial : cloud;
    if (mode & kSqDone) {                             // the sample ends here: its trial and its cloud become equal
        const SiCloudOut dst = (mode & kSqTake) ? cloud : trial;
        for (int i = tid; i < N; i += T) {
#pragma unroll
            for (int r = 0; r < 3; ++r) dst.at(b, i, r) = src.at(b, i, r);
        }
        return;
    }
    float dx = 0.f, dy = 0.f;
    if (moved >= 0) {
        dx = dir[2 * ((long long)b * N + moved)];
        dy = dir[2 * ((long long)b * N + moved) + 1];
    }
    const float sa = __fmul_rn((float)dec[2], a);
    const int nb = (N + 31) / 32, W = T / 32, warp = tid >> 5;
    int nbp = 1;
    while (nbp < nb) nbp *= 2;
    for (int m = warp; m < nb; m += W) {
        const int i = m * 32 + lane;
        float sq[3] = {0.f, 0.f, 0.f};
        if (i < N) {
            float p[3];
            sq_point(src, nrm, b, i, moved, sa, dx, dy, p);
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                const float d = __fsub_rn(p[r], ori.at(b, i, r));
                sq[r] = __fmul_rn(d, d);
            }
        }
#pragma unroll
        for (int r = 0; r < 3; ++r) sq[r] = tree_warp(sq[r]);
        if (lane == 0) {
#pragma unroll
            for (int r = 0; r < 3; ++r) tot[r][m] = sq[r];
        }
    }
    for (int m = nb + tid; m < nbp; m += T) tot[0][m] = tot[1][m] = tot[2][m] = 0.f;
    __syncthreads();
    for (int w = 1; w < nbp; w *= 2) {
        for (int m = tid * 2 * w; m < nbp; m += T * 2 * w) {
#pragma unroll
            for (int r = 0; r < 3; ++r) tot[r][m] = __fadd_rn(tot[r][m], tot[r][m + w]);
        }
        __syncthreads();
    }
    float scale[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const float s = __fdiv_rn(eps, __fadd_rn(__fsqrt_rn(tot[r][0]), 1e-9f));
        scale[r] = s > 1.f ? 1.f : s;                // NaN stays NaN
    }
    // the same points as above, in the same threads: a thread reads src before it writes trial or cloud there
    for (int i = tid; i < N; i += T) {
        float p[3];
        sq_point(src, nrm, b, i, moved, sa, dx, dy, p);
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const float o = ori.at(b, i, r);
            if (mode & kSqTake) cloud.at(b, i, r) = src.at(b, i, r);
            trial.at(b, i, r) = __fadd_rn(o, __fmul_rn(__fsub_rn(p[r], o), scale[r]));
        }
    }
}

}  // namespace pcd

using namespace pcd;

extern "C" int pcd_si_step(float *pc, int64_t sb, int64_t sp, int64_t sc, const float *ori, int64_t o_sb, int64_t o_sp,
                           int64_t o_sc, const float *normal, int64_t n_sb, int64_t n_sp, int64_t n_sc, const float *grad,
                           int64_t g_sb, int64_t g_sp, int64_t g_sc, int B, int N, double step_size, double step_scale,
                           float eps, int split, float *gnorm, void *stream) {
    if (B < 0 || N < 1 || !(eps >= 0.f) || split < 0 || split > kSiMaxSplit || (split & (split - 1)) ||
        (B > 0 && (!pc || !ori || !normal || !grad))) {
        set_error("pcd_si_step: bad argument (need B >= 0, N >= 1, eps >= 0, split 0 or a power of two <= %d, no NULL "
                  "cloud) B=%d N=%d eps=%g split=%d",
                  kSiMaxSplit, B, N, (double)eps, split);
        return PCD_ERR_ARG;
    }
    if (N > PCD_SI_MAX_N) {
        set_error("pcd_si_step: N = %d exceeds %d points per sample", N, PCD_SI_MAX_N);
        return PCD_ERR_UNSUPPORTED;
    }
    int Np = 1;
    while (Np < N) Np *= 2;
    const int smin = Np > 2048 ? Np / 2048 : 1;    // at most 2048 points (256 threads x 8) per CTA
    if (split && split < smin) {
        set_error("pcd_si_step: split %d leaves more than 2048 points per CTA at N = %d", split, N);
        return PCD_ERR_ARG;
    }
    if (B == 0) return PCD_OK;
    int S = split;
    if (!S) {                                        // split samples over more CTAs while the batch does not fill the GPU
        S = smin;
        const long long sms = num_sms();
        while (S < kSiMaxSplit && (long long)B * S < sms && Np / (2 * S) >= 256) S *= 2;
        if (S > 8 && S > max_split()) S = 8;
    } else if (S > 8 && S > max_split()) {
        set_error("pcd_si_step: split %d is not schedulable on this device", S);
        return PCD_ERR_UNSUPPORTED;
    }
    const int chunk = Np / S > 32 ? Np / S : 32;   // points per CTA; padding to a whole warp adds +0 only
    const int P = chunk > kSiMaxThreads ? chunk / kSiMaxThreads : 1, T = chunk / P;
    const float a = (float)(step_size * step_scale);
    const SiCloud o{ori, o_sb, o_sp, o_sc}, n{normal, n_sb, n_sp, n_sc}, g{grad, g_sb, g_sp, g_sc};
    cudaStream_t st = (cudaStream_t)stream;
    switch (P) {
    case 1: return launch_si<1>(B, S, T, pc, sb, sp, sc, o, n, g, N, a, eps, gnorm, st);
    case 2: return launch_si<2>(B, S, T, pc, sb, sp, sc, o, n, g, N, a, eps, gnorm, st);
    case 4: return launch_si<4>(B, S, T, pc, sb, sp, sc, o, n, g, N, a, eps, gnorm, st);
    default: return launch_si<8>(B, S, T, pc, sb, sp, sc, o, n, g, N, a, eps, gnorm, st);
    }
}

extern "C" int pcd_si_sensitivity(const float *grad, int64_t g_sb, int64_t g_sp, int64_t g_sc, const float *normal,
                                  int64_t n_sb, int64_t n_sp, int64_t n_sc, int B, int N, float *s, float *dir,
                                  void *stream) {
    if (B < 0 || N < 1 || (B > 0 && (!grad || !normal || !s || !dir))) {
        set_error("pcd_si_sensitivity: bad argument (need B >= 0, N >= 1, no NULL pointer) B=%d N=%d", B, N);
        return PCD_ERR_ARG;
    }
    if (B == 0) return PCD_OK;
    const long long total = (long long)B * N;
    si_sensitivity_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        SiCloud{grad, g_sb, g_sp, g_sc}, SiCloud{normal, n_sb, n_sp, n_sc}, B, N, s, dir);
    PCD_CUDA_CHECK(cudaGetLastError());
    return PCD_OK;
}

extern "C" int pcd_si_query_round(const float *logits, int64_t l_sb, int64_t l_sc, int C, const int64_t *target,
                                  const float *ori, int64_t o_sb, int64_t o_sp, int64_t o_sc, const float *normal,
                                  int64_t n_sb, int64_t n_sp, int64_t n_sc, const int32_t *order, const float *dir,
                                  float *cloud, int64_t c_sb, int64_t c_sp, int64_t c_sc, float *trial, int64_t t_sb,
                                  int64_t t_sp, int64_t t_sc, int32_t *state, float *best, int B, int N,
                                  float step_size, float eps, int max_query, int targeted, int32_t *active,
                                  void *stream) {
    if (B < 0 || N < 1 || C < 2 || !std::isfinite(step_size) || !(eps >= 0.f) || max_query < 1 ||
        (targeted != 0 && targeted != 1) ||
        (B > 0 && (!logits || !target || !ori || !normal || !order || !dir || !cloud || !trial || !state || !best ||
                   cloud == trial))) {
        set_error("pcd_si_query_round: bad argument (need B >= 0, N >= 1, C >= 2, finite step_size, eps >= 0, "
                  "max_query >= 1, targeted 0 or 1, no NULL pointer but active, cloud != trial) B=%d N=%d C=%d "
                  "step_size=%g eps=%g max_query=%d targeted=%d",
                  B, N, C, (double)step_size, (double)eps, max_query, targeted);
        return PCD_ERR_ARG;
    }
    if (N > PCD_SI_MAX_N) {
        set_error("pcd_si_query_round: N = %d exceeds %d points per sample", N, PCD_SI_MAX_N);
        return PCD_ERR_UNSUPPORTED;
    }
    if (B == 0) return PCD_OK;
    int T = 32;                                      // one warp per 32 points, at most kSqThreads threads
    while (T < kSqThreads && T < N) T *= 2;
    si_query_round_kernel<<<(unsigned)B, T, 0, (cudaStream_t)stream>>>(
        logits, l_sb, l_sc, C, (const long long *)target, SiCloud{ori, o_sb, o_sp, o_sc},
        SiCloud{normal, n_sb, n_sp, n_sc}, order, dir, SiCloudOut{cloud, c_sb, c_sp, c_sc},
        SiCloudOut{trial, t_sb, t_sp, t_sc}, state, best, N, step_size, eps, max_query, targeted, active);
    PCD_CUDA_CHECK(cudaGetLastError());
    return PCD_OK;
}
