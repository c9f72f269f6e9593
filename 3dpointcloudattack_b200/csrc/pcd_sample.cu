// pcd_sample.cu -- uniform point draws without replacement (the resampling of the SOR and SRS defences), sm_100a.
//
// The reference draws with np.random.choice on the host, one sample at a time.  Here every draw is a pure function of
// (seed, global sample id, draw counter, n, npoint), so the device path needs no host round trip and a captured graph
// draws afresh on every replay:
//   sample_points_kernel  one CTA per sample: a Philox4x32-10 key per valid point (the point index in its low 14 bits,
//                         so the keys are distinct), a CUB block radix sort of the keys in opt-in shared memory, and the
//                         first points in key order -- a uniformly random permutation -- written out.
// Every CTA reads the device-side draw counter and the last CTA to have read it advances it, so one call is one launch.
// The contract is pcd_sample_points in include/pcdist.h; the CPU oracle restates it in numpy.
#include <cub/block/block_radix_sort.cuh>

#include "pcd_common.cuh"

namespace pcd {

constexpr int kSampleKeyBits = 14;                 // the point index; N <= 2^14
constexpr unsigned long long kSampleIndexMask = (1ull << kSampleKeyBits) - 1;

// Philox4x32-10 (Salmon et al., SC'11; the constants of Random123 and curand)
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}

// THREADS x ITEMS >= N keys per CTA, blocked: thread t holds points t * ITEMS .. t * ITEMS + ITEMS - 1.  RADIX_BITS: the
// digit width of the sort; below 4 the outer scan is not memoised either (register pressure, see the dispatch).
template <int THREADS, int ITEMS, int RADIX_BITS>
using SampleSort = cub::BlockRadixSort<unsigned long long, THREADS, ITEMS, cub::NullType, RADIX_BITS, (RADIX_BITS >= 4)>;

template <int THREADS, int ITEMS, int RADIX_BITS>
__global__ void __launch_bounds__(THREADS) sample_points_kernel(int N, int npoint, const int32_t *__restrict__ len,
                                                                const int32_t *__restrict__ table, long long table_stride,
                                                                uint2 seed, long long first_sample, long long *counter,
                                                                long long *__restrict__ out_idx) {
    using Sort = SampleSort<THREADS, ITEMS, RADIX_BITS>;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ unsigned long long draw;
    const int b = blockIdx.x, tid = threadIdx.x;

    // The draw counter: every CTA reads it, then arrives on counter[1]; the last to arrive (atomicInc wraps the arrival
    // count back to 0 for the next call) advances it.  The fence orders each CTA's read before its arrival, so no CTA
    // can read the advanced value.
    if (tid == 0) {
        draw = *(volatile unsigned long long *)counter;
        __threadfence();
        if (atomicInc((unsigned *)(counter + 1), gridDim.x - 1) == gridDim.x - 1) {
            *(volatile unsigned long long *)counter = draw + 1;
        }
    }
    __syncthreads();

    const int n = len ? min(max(len[b], 0), N) : N;
    long long *out = out_idx + (size_t)b * npoint;
    const int32_t *tab = table ? table + (size_t)b * table_stride : nullptr;
    auto map = [&](int i) -> long long { return tab ? (long long)tab[i] : (long long)i; };

    if (n == 0) {                                 // nothing to draw from
        for (int j = tid; j < npoint; j += THREADS) out[j] = -1;
        return;
    }
    // n < npoint: the whole cloud npoint / n times, then npoint % n points in key order; n == npoint: the cloud as is
    const int whole = n < npoint ? npoint / n * n : (n == npoint ? n : 0);
    for (int j = tid; j < whole; j += THREADS) out[j] = map(j % n);
    const int take = n > npoint ? npoint : npoint - whole;
    if (take == 0) return;                        // CTA-uniform

    const unsigned long long g = (unsigned long long)(first_sample + b);
    const uint32_t c_lo = (uint32_t)draw, c_hi = (uint32_t)(draw >> 32);
    unsigned long long keys[ITEMS];
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const int i = tid * ITEMS + k;
        if (i < n) {
            const uint4 w = philox4x32_10(make_uint4((uint32_t)i, (uint32_t)g, c_lo, c_hi), seed);
            const unsigned long long r = ((unsigned long long)w.x << 32) | w.y;
            keys[k] = (r & ~kSampleIndexMask) | (unsigned long long)i;
        } else {
            keys[k] = ~0ull;                      // after every valid key: equal random bits resolve by blocked position
        }
    }
    // The index bits need no pass: the sort is stable and the input is in ascending index order, so keys with equal
    // random bits come out by index, as the full 64-bit order puts them.
    Sort(*reinterpret_cast<typename Sort::TempStorage *>(smem_raw)).Sort(keys, kSampleKeyBits, 64);
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const int j = tid * ITEMS + k;            // rank in key order
        if (j < take) out[(n > npoint ? 0 : whole) + j] = map((int)(keys[k] & kSampleIndexMask));
    }
}

template <int THREADS, int ITEMS, int RADIX_BITS>
static cudaError_t launch_sample(int B, int N, int npoint, const int32_t *len, const int32_t *table, long long table_stride,
                                 uint2 seed, long long first_sample, long long *counter, long long *out, cudaStream_t st) {
    const auto kernel = sample_points_kernel<THREADS, ITEMS, RADIX_BITS>;
    const size_t smem = sizeof(typename SampleSort<THREADS, ITEMS, RADIX_BITS>::TempStorage);
    const cudaError_t e = opt_in_smem(kernel, smem);
    if (e != cudaSuccess) return e;
    return launch_kernel(kernel, dim3((unsigned)B), dim3(THREADS), smem, st, false, N, npoint, len, table, table_stride,
                         seed, first_sample, counter, out);
}

}  // namespace pcd

using namespace pcd;

extern "C" int pcd_sample_points(int B, int N, int npoint, const int32_t *len, const int32_t *table, int64_t table_stride,
                                 uint64_t seed, int64_t first_sample, int64_t *counter, int64_t *out_idx, void *stream) {
    if (B < 1 || N < 1 || npoint < 1 || !counter || !out_idx || first_sample < 0 || (table && table_stride < N)) {
        set_error("pcd_sample_points: bad argument (need B, N, npoint >= 1, first_sample >= 0, table_stride >= N with a "
                  "table, no NULL counter or out_idx)");
        return PCD_ERR_ARG;
    }
    if (N > PCD_SAMPLE_MAX_N) {
        set_error("pcd_sample_points: N = %d exceeds %d points per sample", N, PCD_SAMPLE_MAX_N);
        return PCD_ERR_UNSUPPORTED;
    }
    const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    cudaStream_t st = (cudaStream_t)stream;
    long long *ctr = (long long *)counter, *out = (long long *)out_idx;
    // size classes: the sort's shared memory grows with THREADS x ITEMS, so small clouds do not reserve 128 KB.  With 32
    // 64-bit keys per thread, 4-bit digits spill at the 128 registers that 512 threads allow (and 1024 x 16 at 64); 2-bit
    // digits without the memoised scan fit, at 25 passes instead of 13.
    const cudaError_t e =
        N <= 1024   ? launch_sample<128, 8, 4>(B, N, npoint, len, table, table_stride, key, first_sample, ctr, out, st)
        : N <= 4096 ? launch_sample<256, 16, 4>(B, N, npoint, len, table, table_stride, key, first_sample, ctr, out, st)
                    : launch_sample<512, 32, 2>(B, N, npoint, len, table, table_stride, key, first_sample, ctr, out, st);
    PCD_CUDA_CHECK(e);
    return PCD_OK;
}
