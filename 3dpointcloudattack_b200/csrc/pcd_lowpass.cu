// pcd_lowpass.cu -- the low-frequency projection of AOF (attack on frequency) as ONE launch, sm_100a.
//
// AOF (attack/AOF/TAOF_attack.py) splits a cloud into the part spanned by the Kl eigenvectors of the smallest eigenvalues
// of its graph Laplacian and the rest.  With those eigenvectors as the rows of V [Kl,N], low(x) = V^T (V x) per sample
// and per channel; in torch that is two skinny bmm's forward and two backward.  Here one launch does both products:
//   phase 1  c[k] = sum_n V[k,n] * x[n]:  one warp owns a row; lane l sums n = l (mod 32) in ascending order, then an
//            xor butterfly with offsets 16, 8, 4, 2, 1 (every lane ends with the same total);
//   phase 2  y[n] = sum_k V[k,n] * c[k], k ascending.
// A sample is one cluster of S CTAs.  A CTA owns whole rows in phase 1 and a range of points in phase 2, and reads the
// other CTAs' coefficients through distributed shared memory.  Neither sum's order depends on S, the chunking or B, so a
// sample's bits depend only on its inputs.  x is streamed through shared memory in chunks of whole warps of points, so a
// chunk boundary never changes which lane sums a point.  Every operation is rounded on its own (--fmad=false, _rn).
#include <cooperative_groups.h>

#include "pcd_common.cuh"

namespace cg = cooperative_groups;

namespace pcd {

cudaError_t opt_in_smem_fn(const void *kernel, size_t bytes, bool max_carveout);     // pcd_host.cu

constexpr int kLpThreads = 256, kLpWarps = kLpThreads / 32;
constexpr int kLpRows = 2;                 // rows a warp sums at once in phase 1
constexpr int kLpUnroll = 8;               // steps of a lane in phase 1 whose loads are in flight together
constexpr int kLpPts = 2;                  // points a thread sums at once in phase 2
constexpr int kLpDepth = 16;               // rows of phase 2 whose loads are in flight together
constexpr int kLpMaxSplit = 16;
constexpr int kLpMaxChunk = 4096;          // points of x staged in shared memory at once
constexpr int kLpSmemMax = 227 * 1024;     // the opt-in limit of sm_100 per CTA

struct LpIn {
    const float *p;
    long long sb, sp, sc;
    __device__ __forceinline__ float at(int b, int i, int c) const { return p[b * sb + i * sp + c * sc]; }
};
struct LpOut {
    float *p;
    long long sb, sp, sc;
    __device__ __forceinline__ float &at(int b, int i, int c) const { return p[b * sb + i * sp + c * sc]; }
};

// Shared memory: own[rows][3], this CTA's coefficients; buf[3 * chunk], x channel-major in phase 1, then up to chunk
// coefficients [k][3] at a time in phase 2.
__global__ void __launch_bounds__(kLpThreads)
low_pass_kernel(const float *__restrict__ basis, long long b_sb, int Kl, LpIn x, LpOut y, int N, int S, int rows,
                int chunk) {
    extern __shared__ float sh[];
    float *own = sh, *buf = sh + 3 * rows;
    const int b = blockIdx.x / S, rank = blockIdx.x - b * S;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float *V = basis + b * b_sb;

    // phase 1: rows [r0, r1) of this CTA, kLpRows per warp and pass
    const int r0 = rank * rows, r1 = min(Kl, r0 + rows);
    const int npass = r1 > r0 ? (r1 - r0 + kLpWarps * kLpRows - 1) / (kLpWarps * kLpRows) : 0;
    const int nchunks = (N + chunk - 1) / chunk;
    for (int pass = 0; pass < npass; ++pass) {
        const int k0 = r0 + (pass * kLpWarps + warp) * kLpRows;
        float acc[kLpRows][3];
#pragma unroll
        for (int j = 0; j < kLpRows; ++j) acc[j][0] = acc[j][1] = acc[j][2] = 0.f;
        for (int ch = 0; ch < nchunks; ++ch) {
            const int n0 = ch * chunk, cn = min(chunk, N - n0);
            if (nchunks > 1 || pass == 0) {
                __syncthreads();                     // every warp is done with the previous chunk
                for (int i = tid; i < cn; i += kLpThreads) {
#pragma unroll
                    for (int c = 0; c < 3; ++c) buf[c * chunk + i] = x.at(b, n0 + i, c);
                }
                __syncthreads();
            }
            // kLpUnroll steps of the lane at once: all their loads are issued before the first add
            for (int i0 = lane; i0 < cn; i0 += 32 * kLpUnroll) {
                float v[kLpUnroll][kLpRows], xv[kLpUnroll][3];
#pragma unroll
                for (int u = 0; u < kLpUnroll; ++u) {
                    const int i = i0 + 32 * u;
                    const bool in = i < cn;
#pragma unroll
                    for (int c = 0; c < 3; ++c) xv[u][c] = in ? buf[c * chunk + i] : 0.f;
#pragma unroll
                    for (int j = 0; j < kLpRows; ++j) v[u][j] = in && k0 + j < r1 ? V[(long long)(k0 + j) * N + n0 + i] : 0.f;
                }
#pragma unroll
                for (int u = 0; u < kLpUnroll; ++u) {
                    if (i0 + 32 * u >= cn) break;
#pragma unroll
                    for (int j = 0; j < kLpRows; ++j) {
                        if (k0 + j >= r1) break;
#pragma unroll
                        for (int c = 0; c < 3; ++c) acc[j][c] = __fadd_rn(acc[j][c], __fmul_rn(v[u][j], xv[u][c]));
                    }
                }
            }
        }
#pragma unroll
        for (int j = 0; j < kLpRows; ++j) {
            if (k0 + j >= r1) break;                 // warp-uniform
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                float s = acc[j][c];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) s = __fadd_rn(s, __shfl_xor_sync(0xffffffffu, s, o));
                if (lane == 0) own[(k0 + j - r0) * 3 + c] = s;
            }
        }
    }
    if (S > 1)
        cg::this_cluster().sync();                   // every CTA's coefficients are written and visible cluster-wide
    else
        __syncthreads();

    // phase 2: points [p0, p1) of this CTA, kLpPts per thread and pass
    const int per = ((N + S - 1) / S + 31) / 32 * 32;
    const int p0 = min(N, rank * per), p1 = min(N, p0 + per);
    const int kchunks = (Kl + chunk - 1) / chunk;
    for (int q0 = p0; q0 < p1; q0 += kLpThreads * kLpPts) {
        float acc[kLpPts][3];
#pragma unroll
        for (int j = 0; j < kLpPts; ++j) acc[j][0] = acc[j][1] = acc[j][2] = 0.f;
        for (int kc = 0; kc < kchunks; ++kc) {
            const int k0 = kc * chunk, kn = min(chunk, Kl - k0);
            if (kchunks > 1 || q0 == p0) {
                __syncthreads();                     // every thread is done with the previous coefficients
                for (int k = tid; k < kn; k += kLpThreads) {
                    const int owner = (k0 + k) / rows;
                    const float *src = own + (k0 + k - owner * rows) * 3;
                    if (S > 1) src = cg::this_cluster().map_shared_rank(src, owner);
#pragma unroll
                    for (int c = 0; c < 3; ++c) buf[k * 3 + c] = src[c];
                }
                __syncthreads();
            }
            // kLpDepth rows at once: all their loads are issued before the first add
            for (int k = 0; k < kn; k += kLpDepth) {
                float v[kLpDepth][kLpPts];
#pragma unroll
                for (int u = 0; u < kLpDepth; ++u) {
#pragma unroll
                    for (int j = 0; j < kLpPts; ++j) {
                        const int n = q0 + j * kLpThreads + tid;
                        v[u][j] = k + u < kn && n < p1 ? V[(long long)(k0 + k + u) * N + n] : 0.f;
                    }
                }
#pragma unroll
                for (int u = 0; u < kLpDepth; ++u) {
                    if (k + u >= kn) break;
                    const float c0 = buf[(k + u) * 3], c1 = buf[(k + u) * 3 + 1], c2 = buf[(k + u) * 3 + 2];
#pragma unroll
                    for (int j = 0; j < kLpPts; ++j) {
                        acc[j][0] = __fadd_rn(acc[j][0], __fmul_rn(v[u][j], c0));
                        acc[j][1] = __fadd_rn(acc[j][1], __fmul_rn(v[u][j], c1));
                        acc[j][2] = __fadd_rn(acc[j][2], __fmul_rn(v[u][j], c2));
                    }
                }
            }
        }
#pragma unroll
        for (int j = 0; j < kLpPts; ++j) {
            const int n = q0 + j * kLpThreads + tid;
            if (n < p1) {
#pragma unroll
                for (int c = 0; c < 3; ++c) y.at(b, n, c) = acc[j][c];
            }
        }
    }
    if (S > 1) cg::this_cluster().sync();            // no CTA leaves while another still reads its coefficients
}

// Shared memory of a launch, and the chunk of points (a multiple of 32) that fits beside the CTA's coefficients
static void lp_geometry(int N, int rows, int *chunk, size_t *smem) {
    int ch = (N + 31) / 32 * 32;
    if (ch > kLpMaxChunk) ch = kLpMaxChunk;
    const int fit = (kLpSmemMax / 4 - 3 * rows) / 3 / 32 * 32;
    if (ch > fit) ch = fit;
    *chunk = ch;
    *smem = (size_t)(3 * rows + 3 * ch) * sizeof(float);
}

// Largest cluster size the device schedules for this kernel (8 is portable; 16 needs the non-portable attribute), once
// per device, asked with the most shared memory a 16-CTA launch uses.
static int lp_max_split() {
    static PerDeviceInt cache = {};
    const int dev = current_device();
    if (dev < 0) return 8;
    if (cache.v[dev]) return cache.v[dev];
    int best = 8, chunk = 0;
    size_t smem = 0;
    lp_geometry(PCD_LP_MAX_N, PCD_LP_MAX_N / kLpMaxSplit, &chunk, &smem);
    if (cudaFuncSetAttribute(low_pass_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess &&
        opt_in_smem_fn((const void *)low_pass_kernel, smem, false) == cudaSuccess) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(kLpMaxSplit);
        cfg.blockDim = dim3(kLpThreads);
        cfg.dynamicSmemBytes = smem;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = kLpMaxSplit;
        attr[0].val.clusterDim.y = attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        int clusters = 0;
        if (cudaOccupancyMaxActiveClusters(&clusters, low_pass_kernel, &cfg) == cudaSuccess && clusters > 0)
            best = kLpMaxSplit;
    }
    cudaGetLastError();                              // a refused query is an answer, not a pending error
    cache.v[dev] = best;
    return best;
}

}  // namespace pcd

using namespace pcd;

extern "C" int pcd_low_pass(const float *basis, int64_t b_sb, int Kl, const float *x, int64_t x_sb, int64_t x_sp,
                            int64_t x_sc, int B, int N, float *y, int64_t y_sb, int64_t y_sp, int64_t y_sc, int split,
                            void *stream) {
    if (B < 0 || N < 1 || Kl < 1 || Kl > N || b_sb < 0 || split < 0 || split > kLpMaxSplit || (split & (split - 1)) ||
        (B > 0 && (!basis || !x || !y))) {
        set_error("pcd_low_pass: bad argument (need B >= 0, N >= 1, 1 <= Kl <= N, b_sb >= 0, split 0 or a power of two "
                  "<= %d, no NULL pointer) B=%d N=%d Kl=%d b_sb=%lld split=%d",
                  kLpMaxSplit, B, N, Kl, (long long)b_sb, split);
        return PCD_ERR_ARG;
    }
    if (N > PCD_LP_MAX_N) {
        set_error("pcd_low_pass: N = %d exceeds %d points per sample", N, PCD_LP_MAX_N);
        return PCD_ERR_UNSUPPORTED;
    }
    if (B == 0) return PCD_OK;
    int S = split;
    if (!S) {                                        // split samples over more CTAs while the batch does not fill the GPU
        S = 1;
        const long long sms = num_sms();
        while (S < kLpMaxSplit && (long long)B * S < sms && (Kl + 2 * S - 1) / (2 * S) >= 4 && N / (2 * S) >= 64)
            S *= 2;
        if (S > 8 && S > lp_max_split()) S = 8;
    } else if (S > 8 && S > lp_max_split()) {
        set_error("pcd_low_pass: split %d is not schedulable on this device", S);
        return PCD_ERR_UNSUPPORTED;
    }
    const int rows = (Kl + S - 1) / S;
    int chunk = 0;
    size_t smem = 0;
    lp_geometry(N, rows, &chunk, &smem);
    PCD_CUDA_CHECK(opt_in_smem_fn((const void *)low_pass_kernel, smem, false));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)((long long)B * S));
    cfg.blockDim = dim3(kLpThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = S;
    attr[0].val.clusterDim.y = attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = S > 1 ? 1 : 0;
    PCD_CUDA_CHECK(cudaLaunchKernelEx(&cfg, low_pass_kernel, basis, (long long)b_sb, Kl, LpIn{x, x_sb, x_sp, x_sc},
                                      LpOut{y, y_sb, y_sp, y_sc}, N, S, rows, chunk));
    return PCD_OK;
}
