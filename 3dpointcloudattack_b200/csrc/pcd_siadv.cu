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
