// pcd_knnloss.cu -- fused epilogue of the k-NN outlier / smoothing loss, sm_100a.
//
// attack/CW/CW_utils/dist_utils.py:143-153 (KNNDist) and attack/GeoA3/loss_utils.py:148-157
// (kNN_smoothing_loss) turn the [B,N,k+1] distances of the self k-NN select into a per-sample loss with
// nine torch launches (slice, mean, mean, std, mul-add, compare, cast, mul, mean) and as many autograd
// nodes:  value_i = mean_j d_ij (self column dropped),  thr = mean_i value + alpha * std_i value (unbiased),
// loss = mean_i value_i [value_i > thr].  Here: ONE kernel forward (one CTA per sample, three passes over
// the sample's values, which stay in L2 / shared memory; fixed reduction order) and ONE kernel backward
// (the mask and the 1/(N k) factors folded into the scatter through the k-NN indices; only the outlier
// points, ~10 %, do any work).  The comparison is non-differentiable in both reference variants (a
// .float() of a boolean), so they share this backward.
#include "pcd_common.cuh"

namespace pcd {

constexpr int kLossThreads = 1024;

__global__ void __launch_bounds__(kLossThreads) knn_outlier_fwd_kernel(const float *__restrict__ dists, int N, int K1, int first, float alpha,
                                                                       float *__restrict__ value, float *__restrict__ mask,
                                                                       float *__restrict__ loss, float *__restrict__ thr_out,
                                                                       float *__restrict__ zero, size_t nzero_per_sample) {
    __shared__ float sh[kLossThreads / 32];
    const int b = blockIdx.x;
    if (zero)                                     // this sample's slice of the backward's gradient buffer
        for (size_t i = threadIdx.x; i < nzero_per_sample; i += kLossThreads) zero[(size_t)b * nzero_per_sample + i] = 0.f;
    const float *d = dists + (size_t)b * N * K1;
    float *val = value + (size_t)b * N, *msk = mask + (size_t)b * N;
    const float k = (float)(K1 - first);
    float s = 0.f;
    for (int i = threadIdx.x; i < N; i += kLossThreads) {
        float a = 0.f;
        for (int j = first; j < K1; ++j) a = __fadd_rn(a, d[(size_t)i * K1 + j]);
        a = __fdiv_rn(a, k);
        val[i] = a;
        s += a;
    }
    const float mean = block_sum<float, kLossThreads>(s, sh) / (float)N;
    float q = 0.f;
    for (int i = threadIdx.x; i < N; i += kLossThreads) {
        const float c = val[i] - mean;           // written by this very thread
        q += c * c;
    }
    const float var = block_sum<float, kLossThreads>(q, sh) / (float)(N - 1);      // unbiased, torch.std default (NaN for N == 1, as torch)
    const float thr = mean + alpha * sqrtf(var);
    float l = 0.f;
    for (int i = threadIdx.x; i < N; i += kLossThreads) {
        const float v = val[i];
        const float m = v > thr ? 1.f : 0.f;
        msk[i] = m;
        l += v * m;
    }
    const float tot = block_sum<float, kLossThreads>(l, sh);
    if (threadIdx.x == 0) {
        loss[b] = tot / (float)N;
        if (thr_out) thr_out[b] = thr;
    }
}

// grad of sum_b g[b] loss[b] w.r.t. the cloud: d loss_b / d d_ij = mask_i / (N k) for the kept columns,
// d d_ij / d p_i = 2 (p_i - p_j), d d_ij / d p_j = -2 (p_i - p_j)   (self k-NN: both land in the same buffer)
__global__ void __launch_bounds__(256) knn_outlier_bwd_kernel(const float *__restrict__ pc, long long sb, long long sp, long long sc,
                                                              const int32_t *__restrict__ idx, const float *__restrict__ mask,
                                                              const float *__restrict__ g, long long g_stride, int B, int N, int K1,
                                                              int first, float *__restrict__ grad) {
    const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (t >= (long long)B * N) return;
    if (mask[t] == 0.f) return;
    const int b = (int)(t / N), i = (int)(t - (long long)b * N);
    const float g2 = 2.f * g[b * g_stride] / ((float)N * (float)(K1 - first));
    if (g2 == 0.f) return;
    const float *base = pc + (size_t)b * sb;
    const float px = base[i * sp], py = base[i * sp + sc], pz = base[i * sp + 2 * sc];
    float ox = 0.f, oy = 0.f, oz = 0.f;
    for (int j = first; j < K1; ++j) {
        const int qi = min(max(idx[(size_t)t * K1 + j], 0), N - 1);
        const float tx = g2 * (px - base[qi * sp]), ty = g2 * (py - base[qi * sp + sc]), tz = g2 * (pz - base[qi * sp + 2 * sc]);
        ox += tx; oy += ty; oz += tz;
        float *gq = grad + ((size_t)b * N + qi) * 3;
        atomicAdd(gq, -tx); atomicAdd(gq + 1, -ty); atomicAdd(gq + 2, -tz);
    }
    float *gp = grad + (size_t)t * 3;
    atomicAdd(gp, ox); atomicAdd(gp + 1, oy); atomicAdd(gp + 2, oz);
}

}  // namespace pcd

using namespace pcd;

extern "C" int pcd_knn_outlier_forward(const float *dists, int B, int N, int K1, int skip_first, float alpha, float *value, float *mask,
                                       float *loss, float *threshold, float *zero_grad, void *stream) {
    if (!dists || !value || !mask || !loss || B <= 0 || N <= 0 || K1 <= 0 || (skip_first ? 1 : 0) >= K1 || B > 2147483647 / 1) {
        set_error("pcd_knn_outlier_forward: bad argument");
        return PCD_ERR_ARG;
    }
    knn_outlier_fwd_kernel<<<B, kLossThreads, 0, (cudaStream_t)stream>>>(dists, N, K1, skip_first ? 1 : 0, alpha, value, mask, loss, threshold,
                                                                         zero_grad, (size_t)N * 3);
    PCD_CUDA_CHECK(cudaGetLastError());
    return PCD_OK;
}

extern "C" int pcd_knn_outlier_backward(const float *pc, int64_t sb, int64_t sp, int64_t sc, const int32_t *idx, const float *mask,
                                        const float *g_loss, int64_t g_stride, int B, int N, int K1, int skip_first, float *grad_pc,
                                        int grad_prezeroed, void *stream) {
    if (!pc || !idx || !mask || !g_loss || !grad_pc || B <= 0 || N <= 0 || K1 <= 0 || (skip_first ? 1 : 0) >= K1) {
        set_error("pcd_knn_outlier_backward: bad argument");
        return PCD_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const long long total = (long long)B * N;
    if (!grad_prezeroed) PCD_CUDA_CHECK(cudaMemsetAsync(grad_pc, 0, (size_t)total * 3 * sizeof(float), st));
    knn_outlier_bwd_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(pc, sb, sp, sc, idx, mask, g_loss, g_stride, B, N, K1,
                                                                            skip_first ? 1 : 0, grad_pc);
    PCD_CUDA_CHECK(cudaGetLastError());
    return PCD_OK;
}
