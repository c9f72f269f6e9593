// pcd_nn1.cu -- NN-1 sweep (Chamfer / Hausdorff / knn_points K=1) for sm_100a.
//
// Pipeline of pcd_nn1_forward (3 launches on the caller's stream, chained by programmatic
// dependent launch, no host sync):
//   1. nn1_arm     resets the (value,tag) keys and the per-sample completion counters.  Dense
//                  clouds ([B,N,3] or [B,3,N], 16-byte aligned, N % 4 == 0) are NOT packed: the
//                  sweep streams the caller's tensors.  Other inputs (arbitrary strides, the
//                  swapped-norm surrogate of knn_points) go through nn1_prep, which packs both
//                  clouds into the sweep layout first.
//   2. nn1_sweep   THE hot kernel: every (row i, col j) distance exactly once; row minima and
//                  column minima are both taken from the same tile sweep.  Packed fp32x2
//                  math (FMUL2/FFMA2/FADD2), FMNMX3 running minima, CREDUX warp minima,
//                  column tiles streamed by 1-D TMA bulk copies behind an mbarrier (raw xyz is
//                  turned into pair records + norms in shared memory, one tile ahead), stream-K
//                  partition of (sample, row tile, col tile) units over a persistent grid.
//                  Emits per point a 64-bit key = (ordered min value, tag of the 32-wide /
//                  R-wide chunk that produced it) with atomicMin.  Its prologue and first tile
//                  overlap nn1_arm (griddepcontrol.wait sits in front of the first key flush).
//   3. nn1_fixup   four lanes per point re-evaluate its winning chunk (bit-identical
//                  arithmetic) for the lowest index with d == min; the last block of a sample
//                  reduces the sample's minima (scaled sum / max / first argmax, fixed order);
//                  optionally zero-fills the gradient buffers of the coming backward.
//
// Reference semantics served: utils/dis_utils_torch.py:8-28, attack/CW/CW_utils/distance.py:15-70,
// attack/GeoA3/knn_utils.py:10-55 (K=1); see include/pcdist.h.
#include <type_traits>

#include "pcd_common.cuh"

namespace pcd {

// ---------------------------------------------------------------------------------- layout
constexpr int kSweepWarps = 4;
constexpr int kSweepThreads = kSweepWarps * 32;
constexpr int kColChunk = 32;     // columns per row-direction tag
constexpr int kMaxColTile = 256;  // columns per TMA stage
constexpr int kRowPadUnit = 2048; // rows are padded to a multiple of 128*R, R <= 16
constexpr int kFixupThreads = 256;
constexpr int kFixupCtasPerSm = 2;                // 128 registers per thread: twelve 16-byte loads in flight per lane
constexpr int kFixupMaxWarps = 16384;             // upper bound of the persistent fix-up grid (any device)

constexpr int kPruneMaxPoints = 16384;            // bucketing capacity per cloud (nn1_bucket_kernel sorts in shared memory)
constexpr int kPruneMinPoints = 4096;             // smaller clouds or batches: the bucketing pass costs more than the pruning
constexpr int kPruneMinBatch = 16;                // saves; set when it took ~30 us on a B200, ~17 us now (DESIGN.md section 4.0)

struct Nn1Layout {
    int Npad, Mpad;
    size_t rowkey, colkey, counters, partials, rowpk, rowpp, colpk;
    size_t queue, brec, bbox, bperm, total;
    size_t nkeys;
    int partial_slots;     // fix-up partials per sample (one per 32-point unit)
    int bslots;            // pruned path: sorted slots per (sample, side) = 32 * chunks of the larger cloud
};
static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
// keys + counters first (all the dense-input path touches), the packed records of the strided
// path behind them, then the bucketed clouds of the pruned path
static Nn1Layout nn1_layout(int B, int N, int M) {
    Nn1Layout L;
    L.Npad = (int)align_up((size_t)N, kRowPadUnit);
    L.Mpad = (int)align_up((size_t)M, kMaxColTile);
    size_t off = 0;
    L.rowkey = off; off += (size_t)B * L.Npad * 8;
    L.colkey = off; off += (size_t)B * L.Mpad * 8;
    L.nkeys = (size_t)B * L.Npad + (size_t)B * L.Mpad;
    L.counters = off; off = align_up(off + (size_t)B * 4, 256);      // [B] completion counters
    L.partial_slots = (N + 31) / 32 + (M + 31) / 32;          // one partial per unit of 32 points: rows first, then columns
    L.partials = off; off = align_up(off + (size_t)B * L.partial_slots * 16, 256);       // (sum, max, bits of argmax, -)
    L.rowpk = off; off = align_up(off + (size_t)B * L.Npad * 16, 256);
    L.rowpp = off; off = align_up(off + (size_t)B * L.Npad * 16, 256);   // the same records in sweep (slot) order
    L.colpk = off; off = align_up(off + (size_t)B * L.Mpad * 16 + 64, 256);   // +64: the sweep prefetches one record past a tile
    L.bslots = (int)align_up((size_t)(N > M ? N : M), 32);
    const size_t nb = (size_t)B * 2 * L.bslots;                          // [B][side][slot]
    L.queue = off; off = align_up(off + 4, 256);                         // work-queue cursor of the pruned sweep
    L.brec = off; off = align_up(off + nb * 16, 256);                    // pair records in Morton order
    L.bbox = off; off = align_up(off + nb / 32 * 32, 256);               // per chunk: (lo xyz, max norm), (hi xyz, never-prune)
    L.bperm = off; off = align_up(off + nb * 4, 256);                    // sorted slot -> original index
    L.total = off;
    return L;
}

// ------------------------------------------------------------------------------ arm / prep
// Row key slots.  Lane l of a sweep warp owns the R consecutive rows i = blk*32R + l*R + r; the
// key of row i lives at slot blk*32R + r*32 + l, so that the warp's atomicMin flushes are
// coalesced (one 256-B run per r instead of 32 scattered lines: the scattered flush cost 1.8 us
// per row tile, 8 us of 131 at BASELINE config 2).
__host__ __device__ __forceinline__ int row_slot(int i, int R) {      // R is 2, 4, 8 or 16: shifts, no divisions
    const int rs = R == 16 ? 4 : (R == 8 ? 3 : (R == 4 ? 2 : 1));
    const int w = i & ((32 << rs) - 1);
    return (i - w) + ((w & (R - 1)) << 5) + (w >> rs);
}

// keys = ~0 ("no minimum yet"), completion counters = 0.  First kernel of the chain: its
// dependents (the sweep) may start right away, they wait in front of their first key flush.
__global__ void __launch_bounds__(256) nn1_arm_kernel(ulonglong2 *__restrict__ keys2, size_t npairs,
                                                      int *__restrict__ counters, int ncounters) {
    pdl_launch_dependents();
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const ulonglong2 ones = make_ulonglong2(~0ull, ~0ull);
    for (size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x; t < npairs; t += stride) keys2[t] = ones;
    for (size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x; t < (size_t)ncounters; t += stride) counters[t] = 0;
}

// Strided / swapped-norm inputs only:
// rowpk[b][i] = float4(-2x, -2y, -2z, nrow)           (AoS, one LDG.128 per query)
// colpk[b][j/2] = {x0,x1,y0,y1,z0,z1,n0,n1}           (pair records: two LDS.128 feed 2 columns
//                                                      as ready-made fp32x2 operands)
// Padded points are inert: coordinates 0, norm +inf  => every distance through them is +inf.
__global__ void nn1_prep_kernel(const float *__restrict__ rows, int64_t r_sb, int64_t r_sp, int64_t r_sc,
                                const float *__restrict__ cols, int64_t c_sb, int64_t c_sp, int64_t c_sc,
                                int B, int N, int M, int Npad, int Mpad, int R, int norm_kind, int swap_norms,
                                float4 *__restrict__ rowpk, float4 *__restrict__ rowpp, float *__restrict__ colpk,
                                unsigned long long *__restrict__ rowkey, unsigned long long *__restrict__ colkey,
                                int *__restrict__ counters) {
    pdl_launch_dependents();
    const long long per_b = (long long)Npad + Mpad;
    const long long total = per_b * B;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const int b = (int)(t / per_b);
        const int p = (int)(t - (long long)b * per_b);
        if (p == 0) counters[b] = 0;
        if (p < Npad) {
            const int i = p;
            float x = 0.f, y = 0.f, z = 0.f, n = __int_as_float(0x7f800000);
            if (i < N) {
                const float *s = rows + b * r_sb + i * r_sp;
                x = s[0]; y = s[r_sc]; z = s[2 * r_sc];
                if (swap_norms) {
                    const float *o = cols + b * c_sb + i * c_sp;
                    n = sq_norm3(norm_kind, o[0], o[c_sc], o[2 * c_sc]);
                } else {
                    n = sq_norm3(norm_kind, x, y, z);
                }
            }
            const float4 rec = make_float4(-2.f * x, -2.f * y, -2.f * z, n);
            rowpk[(size_t)b * Npad + i] = rec;
            rowpp[(size_t)b * Npad + row_slot(i, R)] = rec;
            rowkey[(size_t)b * Npad + i] = ~0ull;
        } else {
            const int j = p - Npad;
            float x = 0.f, y = 0.f, z = 0.f, n = __int_as_float(0x7f800000);
            if (j < M) {
                const float *s = cols + b * c_sb + j * c_sp;
                x = s[0]; y = s[c_sc]; z = s[2 * c_sc];
                if (swap_norms) {
                    const float *o = rows + b * r_sb + j * r_sp;
                    n = sq_norm3(norm_kind, o[0], o[r_sc], o[2 * r_sc]);
                } else {
                    n = sq_norm3(norm_kind, x, y, z);
                }
            }
            float *rec = colpk + ((size_t)b * Mpad + (j & ~1)) * 4 + (j & 1);
            rec[0] = x; rec[2] = y; rec[4] = z; rec[6] = n;
            colkey[(size_t)b * Mpad + j] = ~0ull;
        }
    }
}

// ------------------------------------------------------------------- pruned path: bucketing
// Dense clouds of kPruneMinPoints to kPruneMaxPoints points in batches of kPruneMinBatch or more (no tiling override) take
// the pruned chain
//   nn1_bucket  -> nn1_pruned_sweep -> nn1_fixup (pruned keys)
// instead of arm -> sweep -> fix-up.  A nearest-neighbour search needs only the few chunk pairs
// whose boxes are close; see DESIGN.md section 4.1 for the bound and the rounding margin.
//
// nn1_bucket: one CTA per (sample, side).  Both clouds of a sample are quantised on ONE grid (the
// joint box of their finite points, 32 cells per axis), each side is sorted by the 15-bit Morton
// code of its cell (stable, so equal codes keep index order), and the sorted cloud is cut into
// chunks of 32.  Written per (sample, side):
//   brec [slot]  pair records {x0,x1,y0,y1},{z0,z1,n0,n1} in sorted order; slots past the cloud
//                are inert (0, 0, 0, +inf), as in the packed sweep
//   bperm[slot]  original index of the point in that slot
//   bbox [chunk] (lo xyz, largest norm), (hi xyz, never-prune flag) over the chunk's points
// Non-finite points get a code past every finite one, so they share the last chunks, whose
// never-prune flag makes every comparison against them keep the pair.
//
// The pass is latency bound (a few hundred KB per CTA), so it is built from as few dependent
// steps as possible: 16-byte loads of 4 points at a time, codes packed with the point index into one
// 32-bit word (code << 14 | index, so only the word moves through the sort), two 8-bit LSD radix
// passes in shared memory with four barriers each, and one gather of the sorted points from L1 / L2
// with every load in flight before the first store.
constexpr int kBucketThreads = 1024;
constexpr int kBucketWarps = kBucketThreads / 32;
constexpr int kMortonBits = 5;                    // cells per axis = 2^5: finer grids make no better chunks
                                                  // (DESIGN.md section 4.0) and cost radix-sort passes
constexpr uint32_t kNonFiniteCode = 1u << (3 * kMortonBits);
constexpr int kBucketIndexBits = 14;              // kPruneMaxPoints = 2^14
constexpr int kBucketDigits = 256;
constexpr int kBucketCntStride = kBucketDigits + 1;   // per-warp digit counters; +1: the scan's transposed reads hit 32 banks
static_assert(kPruneMaxPoints <= (1 << kBucketIndexBits), "the sort word holds the point index in its low bits");

#ifdef PCD_SWEEP_TRACE
// development build only (tools/trace_sweep.py, tools/nn1_prune_bench.py --count): per-CTA timestamps of the sweep or of
// the bucketing pass (whichever chain runs)
__device__ unsigned long long *g_sweep_trace = nullptr;
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
// phase k of the bucketing pass ends (0 = start, 1 loads + joint box, 2 codes, 3 / 4 sort passes, 5 gather + stores), in
// the CTA's 8 words of the trace buffer (tools/nn1_prune_bench.py --count reads them)
#define PCD_BUCKET_STAMP(k)                                                                         \
    do {                                                                                            \
        if (g_sweep_trace && threadIdx.x == 0) g_sweep_trace[blockIdx.x * 8 + (k)] = globaltimer_ns(); \
    } while (0)
#else
#define PCD_BUCKET_STAMP(k) do { } while (0)
#endif

__device__ __forceinline__ uint32_t spread3(uint32_t v) {     // bit k of v -> bit 3k
    v &= 0x3ffu;
    v = (v ^ (v << 16)) & 0xff0000ffu;
    v = (v ^ (v << 8)) & 0x0300f00fu;
    v = (v ^ (v << 4)) & 0x030c30c3u;
    v = (v ^ (v << 2)) & 0x09249249u;
    return v;
}

struct BucketArgs {
    const float *rows; long long r_sb, r_sp, r_sc;
    const float *cols; long long c_sb, c_sp, c_sc;
    int N, M, norm_kind, bslots;
    float4 *brec; float4 *bbox; int *bperm;
    int *counters; int *queue;
};

// One dense cloud of the pruned chain: point-major [n,3] (sc == 1) or channel-major [3,n] rows, 16-byte aligned, n % 4 == 0
// (dense_layout), so 4 consecutive points are three 16-byte loads either way.
struct BucketCloud {
    const float *__restrict__ p;
    long long sc;
    __device__ __forceinline__ void quad(int g, float x[4], float y[4], float z[4]) const {
        if (sc == 1) {
            const float4 *q = reinterpret_cast<const float4 *>(p) + 3 * g;
            const float4 a = __ldg(q), b = __ldg(q + 1), c = __ldg(q + 2);
            x[0] = a.x; y[0] = a.y; z[0] = a.z; x[1] = a.w; y[1] = b.x; z[1] = b.y;
            x[2] = b.z; y[2] = b.w; z[2] = c.x; x[3] = c.y; y[3] = c.z; z[3] = c.w;
        } else {
            const float4 a = __ldg(reinterpret_cast<const float4 *>(p) + g);
            const float4 b = __ldg(reinterpret_cast<const float4 *>(p + sc) + g);
            const float4 c = __ldg(reinterpret_cast<const float4 *>(p + 2 * sc) + g);
            x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; y[0] = b.x; y[1] = b.y; y[2] = b.z; y[3] = b.w;
            z[0] = c.x; z[1] = c.y; z[2] = c.z; z[3] = c.w;
        }
    }
    __device__ __forceinline__ void point(int i, float &x, float &y, float &z) const {
        const float *q = p + (sc == 1 ? 3LL * i : (long long)i);
        x = __ldg(q); y = __ldg(q + sc); z = __ldg(q + 2 * sc);
    }
};

__device__ __forceinline__ bool finite3(float x, float y, float z) { return isfinite(x) && isfinite(y) && isfinite(z); }

// One stable LSD pass over the 8-bit digit at `shift` of n sort words, src -> dst (shared memory).  Warp w ranks the items
// [w*S, w*S + S), S = 32 * steps, in index order: eight ballots group the lanes of one step by digit (a fixed cost, where
// __match_any_sync serialises over the distinct digits), the highest lane of each group advances the warp's own counter of
// that digit.  A block scan over (digit, warp) turns the counters into
// output offsets.  4 barriers.
template <int ITEMS>
__device__ __forceinline__ void bucket_sort_pass(const uint32_t *src, uint32_t *dst, int *cnt, int *wsum, int n, int steps,
                                                 int shift, int tid) {
    const int lane = tid & 31, warp = tid >> 5, S = 32 * steps;
    int *row = cnt + warp * kBucketCntStride;
#pragma unroll
    for (int d = lane; d < kBucketDigits; d += 32) row[d] = 0;
    __syncwarp();
    int local[ITEMS];
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        if (k < steps) {
            const int i = warp * S + 32 * k + lane;
            const bool v = i < n;
            const int d = v ? (int)((src[i] >> shift) & (kBucketDigits - 1)) : 0;
            unsigned peers = __ballot_sync(0xffffffffu, v);     // the valid lanes with digit d: one ballot per digit bit
#pragma unroll
            for (int bit = 0; bit < 8; ++bit) {
                const unsigned m = __ballot_sync(0xffffffffu, (d >> bit) & 1);
                peers &= (d >> bit) & 1 ? m : ~m;
            }
            const int leader = 31 - __clz(peers);
            int old = 0;
            if (v && lane == leader) { old = row[d]; row[d] = old + __popc(peers); }
            local[k] = __shfl_sync(0xffffffffu, old, leader) + __popc(peers & ((1u << lane) - 1));
            __syncwarp();
        }
    }
    __syncthreads();
    // thread (digit d, quarter q) scans the counters of warps 8q .. 8q+7 for digit d; the warp holds digits 8*warp .. +7
    const int d = tid >> 2, q = tid & 3;
    int sum = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) sum += cnt[(8 * q + j) * kBucketCntStride + d];
    int incl = sum;                                           // over the quarters of digit d
#pragma unroll
    for (int o = 1; o < 4; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (q >= o) incl += t;
    }
    const int total = __shfl_sync(0xffffffffu, incl, lane | 3);
    int dig = total;                                          // over the digits of this warp, up to d
#pragma unroll
    for (int o = 4; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, dig, o);
        if (lane >= o) dig += t;
    }
    if (lane == 31) wsum[warp] = dig;
    __syncthreads();
    int below = lane < warp ? wsum[lane] : 0;                 // digits of the warps before this one
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) below += __shfl_xor_sync(0xffffffffu, below, o);
    int run = below + dig - total + incl - sum;               // only this thread writes the counters it read
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        int *c = cnt + (8 * q + j) * kBucketCntStride + d;
        const int v = *c;
        *c = run;
        run += v;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        if (k < steps) {
            const int i = warp * S + 32 * k + lane;
            if (i < n) {
                const uint32_t w = src[i];
                dst[row[(w >> shift) & (kBucketDigits - 1)] + local[k]] = w;
            }
        }
    }
    __syncthreads();
}

// Clouds of up to 4096 points keep their coordinates in shared memory (48 KB) for the gather; larger ones (192 KB would not
// fit beside the sort) gather from L1 / L2.
template <int ITEMS>
__host__ __device__ constexpr bool bucket_stages_points() { return ITEMS <= 4; }
// dynamic shared memory: two word buffers of kBucketThreads * ITEMS, the per-warp digit counters, then x, y, z if staged
template <int ITEMS>
constexpr size_t bucket_smem_bytes() {
    return ((2 + (bucket_stages_points<ITEMS>() ? 3 : 0)) * (size_t)kBucketThreads * ITEMS +
            (size_t)kBucketWarps * kBucketCntStride) * sizeof(uint32_t);
}

template <int ITEMS>
__global__ void __launch_bounds__(kBucketThreads, 1) nn1_bucket_kernel(BucketArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint32_t *wa = reinterpret_cast<uint32_t *>(smem_raw), *wb = wa + kBucketThreads * ITEMS;
    int *cnt = reinterpret_cast<int *>(wb + kBucketThreads * ITEMS);
    constexpr bool kStaged = bucket_stages_points<ITEMS>();
    float *sx = reinterpret_cast<float *>(cnt + kBucketWarps * kBucketCntStride), *sy = sx + kBucketThreads * ITEMS,
          *sz = sy + kBucketThreads * ITEMS;     // used only if kStaged
    __shared__ float red[6][kBucketWarps];
    __shared__ int wsum[kBucketWarps];
    PCD_BUCKET_STAMP(0);
    pdl_launch_dependents();     // the pruned sweep may become resident; it waits for our completion
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.x >> 1, side = blockIdx.x & 1;
    if (tid == 0) {
        if (side == 0) a.counters[b] = 0;
        if (blockIdx.x == 0) *a.queue = 0;
    }
    const float pinf = __int_as_float(0x7f800000);
    // built where it is used, from the parameter bank: kept live across the phases, the pointers spill
    auto cloud = [&](int s) {
        return s ? BucketCloud{a.cols + b * a.c_sb, a.c_sc} : BucketCloud{a.rows + b * a.r_sb, a.r_sc};
    };
    const int n = side ? a.M : a.N;

    // joint box of the sample's finite points: both CTAs of the sample compute the same one
    float lo[3] = {pinf, pinf, pinf}, hi[3] = {-pinf, -pinf, -pinf};
    auto widen = [&](const BucketCloud &c, int g) {
        float x[4], y[4], z[4];
        c.quad(g, x, y, z);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            if (finite3(x[e], y[e], z[e])) {
                lo[0] = fminf(lo[0], x[e]); lo[1] = fminf(lo[1], y[e]); lo[2] = fminf(lo[2], z[e]);
                hi[0] = fmaxf(hi[0], x[e]); hi[1] = fmaxf(hi[1], y[e]); hi[2] = fmaxf(hi[2], z[e]);
            }
        }
    };
    const int gr = a.N >> 2, gt = gr + (a.M >> 2);             // 4-point groups of the rows, then of the columns
#pragma unroll 2
    for (int g = tid; g < gt; g += kBucketThreads) widen(cloud(g >= gr), g < gr ? g : g - gr);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[c] = fminf(lo[c], __shfl_xor_sync(0xffffffffu, lo[c], o));
            hi[c] = fmaxf(hi[c], __shfl_xor_sync(0xffffffffu, hi[c], o));
        }
        if (lane == 0) { red[c][warp] = lo[c]; red[3 + c][warp] = hi[c]; }
    }
    __syncthreads();
    float cell[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        lo[c] = red[c][lane]; hi[c] = red[3 + c][lane];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[c] = fminf(lo[c], __shfl_xor_sync(0xffffffffu, lo[c], o));
            hi[c] = fmaxf(hi[c], __shfl_xor_sync(0xffffffffu, hi[c], o));
        }
        cell[c] = hi[c] > lo[c] ? (float)(1 << kMortonBits) / (hi[c] - lo[c]) : 0.f;
    }
    PCD_BUCKET_STAMP(1);

    // sort words in index order (the own cloud is read again: L1 / L2 hits); non-finite points sort last, in index order
    static_assert((kBucketWarps * kBucketCntStride) % 4 == 0, "the staged coordinates are stored as float4");
#pragma unroll
    for (int j = 0; j < ITEMS / 4; ++j) {
        const int g = tid + j * kBucketThreads;
        if (4 * g < n) {
            float x[4], y[4], z[4];
            cloud(side).quad(g, x, y, z);
            uint32_t w[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                uint32_t code = kNonFiniteCode;
                if (finite3(x[e], y[e], z[e])) {
                    const float p[3] = {x[e], y[e], z[e]};
                    code = 0;
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        const float qc = fminf(fmaxf((p[c] - lo[c]) * cell[c], 0.f), (float)((1 << kMortonBits) - 1));
                        code |= spread3((uint32_t)qc) << c;
                    }
                }
                w[e] = code << kBucketIndexBits | (uint32_t)(4 * g + e);
            }
            reinterpret_cast<uint4 *>(wa)[g] = make_uint4(w[0], w[1], w[2], w[3]);
            if (kStaged) {
                reinterpret_cast<float4 *>(sx)[g] = make_float4(x[0], x[1], x[2], x[3]);
                reinterpret_cast<float4 *>(sy)[g] = make_float4(y[0], y[1], y[2], y[3]);
                reinterpret_cast<float4 *>(sz)[g] = make_float4(z[0], z[1], z[2], z[3]);
            }
        }
    }
    __syncthreads();
    PCD_BUCKET_STAMP(2);
    const int steps = (n + kBucketThreads - 1) / kBucketThreads;
    bucket_sort_pass<ITEMS>(wa, wb, cnt, wsum, n, steps, kBucketIndexBits, tid);
    PCD_BUCKET_STAMP(3);
    bucket_sort_pass<ITEMS>(wb, wa, cnt, wsum, n, steps, kBucketIndexBits + 8, tid);
    PCD_BUCKET_STAMP(4);

    // wa holds the sorted words.  Thread tid writes the slot pairs (2t, 2t+1), t = tid + j * kBucketThreads: one 32-byte
    // pair record and one 8-byte permutation entry; the 16 consecutive lanes that hold one chunk reduce its box.  The points
    // come from shared memory if staged, else from L1 / L2.
    const BucketCloud own = cloud(side);
    const size_t base = (size_t)(b * 2 + side) * a.bslots;
    const int nslots = (n + 31) & ~31;
    constexpr int kBatch = ITEMS / 2 < 4 ? ITEMS / 2 : 4;     // slot pairs per thread with their loads in flight together
#pragma unroll
    for (int j0 = 0; j0 < ITEMS / 2; j0 += kBatch) {
        float px[kBatch][2], py[kBatch][2], pz[kBatch][2];
        int idx[kBatch][2];
#pragma unroll
        for (int j = 0; j < kBatch; ++j) {
            const int s = 2 * (tid + (j0 + j) * kBucketThreads);
            px[j][0] = px[j][1] = py[j][0] = py[j][1] = pz[j][0] = pz[j][1] = 0.f;
            if (s < n) {                                      // n is even: both slots hold points
                const uint2 w = reinterpret_cast<const uint2 *>(wa)[s >> 1];
                idx[j][0] = (int)(w.x & ((1u << kBucketIndexBits) - 1));
                idx[j][1] = (int)(w.y & ((1u << kBucketIndexBits) - 1));
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    if (kStaged) {
                        px[j][e] = sx[idx[j][e]]; py[j][e] = sy[idx[j][e]]; pz[j][e] = sz[idx[j][e]];
                    } else {
                        own.point(idx[j][e], px[j][e], py[j][e], pz[j][e]);
                    }
                }
            }
        }
#pragma unroll
        for (int j = 0; j < kBatch; ++j) {
            const int s = 2 * (tid + (j0 + j) * kBucketThreads);
            float blo[3] = {pinf, pinf, pinf}, bhi[3] = {-pinf, -pinf, -pinf}, bn = -pinf, nn[2] = {pinf, pinf};
            int bad = 0;
            if (s < n) {
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    nn[e] = sq_norm3(a.norm_kind, px[j][e], py[j][e], pz[j][e]);
                    if (finite3(px[j][e], py[j][e], pz[j][e])) {
                        blo[0] = fminf(blo[0], px[j][e]); blo[1] = fminf(blo[1], py[j][e]); blo[2] = fminf(blo[2], pz[j][e]);
                        bhi[0] = fmaxf(bhi[0], px[j][e]); bhi[1] = fmaxf(bhi[1], py[j][e]); bhi[2] = fmaxf(bhi[2], pz[j][e]);
                        bn = fmaxf(bn, nn[e]);
                    } else {
                        bad = 1;
                    }
                }
                reinterpret_cast<int2 *>(a.bperm + base)[s >> 1] = make_int2(idx[j][0], idx[j][1]);
            }
            if (s < nslots) {
                float4 *rec = a.brec + base + s;                 // slots s, s+1 = the two float4 of one pair record
                rec[0] = make_float4(px[j][0], px[j][1], py[j][0], py[j][1]);
                rec[1] = make_float4(pz[j][0], pz[j][1], nn[0], nn[1]);
            }
#pragma unroll
            for (int o = 1; o < 16; o <<= 1) {
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    blo[c] = fminf(blo[c], __shfl_xor_sync(0xffffffffu, blo[c], o));
                    bhi[c] = fmaxf(bhi[c], __shfl_xor_sync(0xffffffffu, bhi[c], o));
                }
                bn = fmaxf(bn, __shfl_xor_sync(0xffffffffu, bn, o));
                bad |= __shfl_xor_sync(0xffffffffu, bad, o);
            }
            const int chunk = s >> 5;
            if ((lane & 15) == 0 && chunk * 32 < n) {
                float4 *bx = a.bbox + 2 * (base / 32 + chunk);
                bx[0] = make_float4(blo[0], blo[1], blo[2], bn);
                bx[1] = make_float4(bhi[0], bhi[1], bhi[2], bad ? 1.f : 0.f);
            }
        }
    }
#ifdef PCD_SWEEP_TRACE
    __syncthreads();
    PCD_BUCKET_STAMP(5);
#endif
}

// ---------------------------------------------------------------- pruned path: the sweep
// Persistent grid, one warp per work item = (sample, side, chunk A of 32 sorted points), items
// taken from a queue in (sample, side, chunk) order.  Lane l owns point p_l of A and takes its exact
// minimum over the other side:
//   seed    evaluate the other side's chunks of the same relative Morton rank (+-1); every lane's
//           running minimum best_l is then a computed pair value, and U = the largest of them over A
//   filter  two stages over every other chunk C, in index order:
//           box     a ballot over the chunk boxes, 32 at a time, keeps C unless  fl(LB(A, C) - E(A, C)) > U
//           point   for each C the box stage keeps, lane l needs C unless  fl(LB(p_l, C) - E(p_l, C)) > best_l,
//                   with best_l as it stands when C is queued; the warp evaluates C if any lane needs it
//           Either way every pair value of a chunk a lane skips exceeds that lane's minimum, so it can
//           neither be the minimum nor tie it.  A NaN anywhere keeps the chunk.
//   LB      squared per-axis gap of the two boxes (or of the point and the box), scaled down past its
//           own rounding (lower bound)
//   E       kPruneMarginRel * (largest norm of A, or the norm of p_l, + largest norm of C) + kPruneMarginAbs,
//           a bound on |computed pair value - exact squared distance| for all three forms and both norm
//           kinds (DESIGN.md section 4.0)
//   arg-min once per distinct winning chunk of the item's lanes (neighbouring points share a few):
//           the chunk is re-evaluated and its lanes take the lowest ORIGINAL index with d == minimum.
//           A lane whose minimum two chunks reached (an exact tie) takes it over every chunk it did not
//           skip, re-derived with the final minima, in a second pass of the item.
// Candidate records are requested two chunks ahead of their evaluation, the next 32 boxes one ballot
// ahead, and the next winning chunk's records while the current one is compared.
// Pair values use the sweep's instruction sequence (pair_dist_fixed_x2), so they are the sweep's
// values bit for bit.  Key per point (at its original index) = (minimum, original arg-min): the
// fix-up only transforms, stores and reduces.
constexpr int kPruneThreads = 256;
constexpr float kPruneLbScale = 1.0f - 0x1p-20f;
constexpr float kPruneMarginRel = 40.0f * 0x1p-24f;
constexpr float kPruneMarginAbs = 0x1p-100f;

struct PruneArgs {
    const float4 *brec, *bbox;
    const int *bperm;
    int *queue;
    unsigned long long *rowkey, *colkey;
    int B, N, M, Npad, Mpad, bslots;
};

// 16-byte global -> shared copy that bypasses the registers (LDGSTS); completion is tracked per commit group
__device__ __forceinline__ void cp_async16(void *dst, const void *src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async4(void *dst, const void *src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

#ifdef PCD_SWEEP_TRACE
// development build only (tools/nn1_prune_bench.py --count): items, evaluated chunks, arg-min re-scans, tie passes
__device__ unsigned long long *g_prune_count = nullptr;
#endif

// one item; SIDE 0 = a chunk of rows against the columns, 1 = a chunk of columns against the rows
template <int FORM, int SIDE>
__device__ __forceinline__ void pruned_item(const PruneArgs &a, int b, int c, float4 *ring, float4 *sbuf, int *jbuf, int lane) {
    const float pinf = __int_as_float(0x7f800000);
    const int n_own = SIDE ? a.M : a.N;
    const int ncs = ((SIDE ? a.M : a.N) + 31) >> 5, nco = ((SIDE ? a.N : a.M) + 31) >> 5;
    const size_t own = (size_t)(b * 2 + SIDE) * a.bslots, opp = (size_t)(b * 2 + (SIDE ^ 1)) * a.bslots;
    const int slot = c * 32 + lane;
    const bool valid = slot < n_own;
    const float *orec = reinterpret_cast<const float *>(a.brec) + (own + (slot & ~1)) * 4 + (slot & 1);
    const float m2x = -2.f * __ldg(orec), m2y = -2.f * __ldg(orec + 2), m2z = -2.f * __ldg(orec + 4), pn = __ldg(orec + 6);
    const float4 *crec = a.brec + opp;
    const int cs = (int)((long long)c * nco / ncs);
    const float4 *cbox = a.bbox + 2 * (opp / 32);
    // boxes of chunks base + lane; lanes past the cloud get an empty box (never read by the filter)
    auto load_boxes = [&](int base, float4 &lo, float4 &hi) {
        const int cb = base + lane;
        lo = cb < nco ? __ldg(cbox + 2 * cb) : make_float4(0.f, 0.f, 0.f, 0.f);
        hi = cb < nco ? __ldg(cbox + 2 * cb + 1) : make_float4(0.f, 0.f, 0.f, 0.f);
    };
    float4 nlo, nhi;
    load_boxes(0, nlo, nhi);          // in flight during the seeds
#ifdef PCD_SWEEP_TRACE
    unsigned long long n_eval = 0, n_scan = 0, n_tie = 0;
#endif

    float best = pinf;
    uint32_t tag = 0;
    bool tie = false;
    auto evaluate = [&](int cc, const float4 *s) {
        __syncwarp();                 // the copies of every lane into the slot are visible
        float m = pinf;
#pragma unroll 8                      // fully unrolled, the loop spills at the 3-CTA register budget
        for (int k = 0; k < 16; ++k) {
            const float4 A = s[2 * k], Bv = s[2 * k + 1];
            const f32x2 d = pair_dist_fixed_x2<FORM>(SIDE == 0, m2x, m2y, m2z, pn, pack2(A.x, A.y), pack2(A.z, A.w),
                                                     pack2(Bv.x, Bv.y), pack2(Bv.z, Bv.w));
            float lo, hi;
            unpack2(d, lo, hi);
            m = min3(m, lo, hi);
        }
        if (m < best) { best = m; tag = (uint32_t)cc; tie = false; }
        else if (m == best && m < pinf) tie = true;
#ifdef PCD_SWEEP_TRACE
        ++n_eval;
#endif
    };
    // queue chunk cc (-1: none): its records are copied into ring slot rs now, and the chunk queued two pushes
    // before it (slot rs + 1 of 3) is evaluated.  The copies bypass the registers, so the depth costs none.
    int q0 = -1, q1 = -1, rs = 0;
    auto push = [&](int cc) {
        __syncwarp();                 // every lane is done with the chunk evaluated at the last push, the old tenant of slot rs
        if (cc >= 0) cp_async16(ring + rs * 32 + lane, crec + (size_t)cc * 32 + lane);
        cp_async_commit();
        const int ev = rs == 2 ? 0 : rs + 1;
        if (q0 >= 0) {
            cp_async_wait<2>();
            evaluate(q0, ring + ev * 32);
        }
        q0 = q1; q1 = cc; rs = ev;
    };
    auto drain = [&]() {
#pragma unroll 1
        for (int k = 0; k < 2; ++k) push(-1);
    };
    // the seeds cs, cs - 1, cs + 1 (those inside the other cloud)
    auto seeds = [&](auto &&fn) {
#pragma unroll 1
        for (int k = 0; k < 3; ++k) {
            const int cc = cs + (k == 0 ? 0 : (k == 1 ? -1 : 1));
            if (cc >= 0 && cc < nco) fn(cc);
        }
    };
    seeds(push);
    drain();
    // box stage, once per item: lane g ends with the ballots of chunks 32g .. 32g + 31 (kmask: kept, fmask: kept
    // whatever the point stage says), so nothing of it stays live while chunks are evaluated
    uint32_t kmask = 0, fmask = 0;
    {
        const float4 *obox = a.bbox + 2 * (own / 32 + c);
        const float4 alo = __ldg(obox), ahi = __ldg(obox + 1);
        const bool keep_all = ahi.w != 0.f;
        const float U = ordered_to_f32(__reduce_max_sync(0xffffffffu, valid ? f32_to_ordered(best) : 0u));
        for (int base = 0; base < nco; base += 32) {
            const float4 clo = nlo, chi = nhi;
            if (base + 32 < nco) load_boxes(base + 32, nlo, nhi);
            const int cb = base + lane;
            bool keep = false;
            if (cb < nco && (cb < cs - 1 || cb > cs + 1)) {
                const float gx = fmaxf(fmaxf(clo.x - ahi.x, alo.x - chi.x), 0.f);
                const float gy = fmaxf(fmaxf(clo.y - ahi.y, alo.y - chi.y), 0.f);
                const float gz = fmaxf(fmaxf(clo.z - ahi.z, alo.z - chi.z), 0.f);
                const float lb = (gx * gx + gy * gy + gz * gz) * kPruneLbScale;
                const float e = kPruneMarginRel * (alo.w + clo.w) + kPruneMarginAbs;
                keep = keep_all || chi.w != 0.f || !(lb - e > U);
            }
            const uint32_t k = __ballot_sync(0xffffffffu, keep), f = __ballot_sync(0xffffffffu, keep && (keep_all || chi.w != 0.f));
            if (lane == base >> 5) { kmask = k; fmask = f; }
        }
    }
    // point stage: every chunk of the box stage that some lane with `need` set does not skip, in index order
    auto kept = [&](auto &&fn, bool need) {
        for (int base = 0; base < nco; base += 32) {
            const uint32_t force = __shfl_sync(0xffffffffu, fmask, base >> 5);
            for (uint32_t msk = __shfl_sync(0xffffffffu, kmask, base >> 5); msk; msk &= msk - 1) {
                const int k = __ffs(msk) - 1;
                const float4 blo = __ldg(cbox + 2 * (base + k)), bhi = __ldg(cbox + 2 * (base + k) + 1);     // L1 hits
                const float px = -0.5f * m2x, py = -0.5f * m2y, pz = -0.5f * m2z;     // exact
                const float gx = fmaxf(fmaxf(blo.x - px, px - bhi.x), 0.f);
                const float gy = fmaxf(fmaxf(blo.y - py, py - bhi.y), 0.f);
                const float gz = fmaxf(fmaxf(blo.z - pz, pz - bhi.z), 0.f);
                const float lb = (gx * gx + gy * gy + gz * gz) * kPruneLbScale;
                const float e = kPruneMarginRel * (pn + blo.w) + kPruneMarginAbs;
                if (((force >> k) & 1u) || __any_sync(0xffffffffu, need && !(lb - e > best))) fn(base + k);
            }
        }
    };
    kept(push, valid);
    drain();

    // arg-min: the lowest original index with d == minimum among the candidates in stage buffer sb, for the lanes that ask
    int arg = 0x7fffffff;
    auto compare = [&](int sb, bool want) {
        __syncwarp();                 // the copies of every lane into the buffer are visible
        if (want) {
            const float4 *s = sbuf + sb * 32;
            const int *js = jbuf + sb * 32;
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                const float4 A = s[2 * k], Bv = s[2 * k + 1];
                const f32x2 d = pair_dist_fixed_x2<FORM>(SIDE == 0, m2x, m2y, m2z, pn, pack2(A.x, A.y), pack2(A.z, A.w),
                                                         pack2(Bv.x, Bv.y), pack2(Bv.z, Bv.w));
                float lo, hi;
                unpack2(d, lo, hi);
                if (lo == best) arg = min(arg, js[2 * k]);
                if (hi == best) arg = min(arg, js[2 * k + 1]);
            }
        }
    };
    // records and original indices of chunk cc (-1: none) into stage buffer sb, one commit group; slots past the cloud
    // are inert: never matched.  Every lane must be done with the buffer's last compare (a __syncwarp in between).
    auto stage_scan = [&](int cc, int sb) {
        if (cc >= 0) {
            cp_async16(sbuf + sb * 32 + lane, crec + (size_t)cc * 32 + lane);
            cp_async4(jbuf + sb * 32 + lane, a.bperm + opp + (size_t)cc * 32 + lane);
        }
        cp_async_commit();
    };
    // a lane whose minimum one chunk reached: that chunk, one pass per distinct winning chunk (neighbours share a few);
    // the next one is copied into the other buffer while the current one is compared
    bool pending = valid && best < pinf && !tie;
    uint32_t pm = __ballot_sync(0xffffffffu, pending);
    int cc = pm ? __shfl_sync(0xffffffffu, (int)tag, __ffs(pm) - 1) : -1;
    int sb = 0;
    stage_scan(cc, sb);
    while (cc >= 0) {
        const bool mine = pending && tag == (uint32_t)cc;
        if (mine) pending = false;
        pm = __ballot_sync(0xffffffffu, pending);
        const int nc = pm ? __shfl_sync(0xffffffffu, (int)tag, __ffs(pm) - 1) : -1;
        __syncwarp();                 // every lane is done with the last compare, which read buffer sb ^ 1
        stage_scan(nc, sb ^ 1);
        cp_async_wait<1>();
        compare(sb, mine);
        cc = nc; sb ^= 1;
#ifdef PCD_SWEEP_TRACE
        ++n_scan;
#endif
    }
    // a lane whose minimum two chunks reached (an exact tie, rare): every chunk it does not skip at its final minimum,
    // once more (a superset of the chunks that can hold a pair equal to it)
    const bool tied = valid && best < pinf && tie;
    if (__any_sync(0xffffffffu, tied)) {
        auto all = [&](int cc2) {
            __syncwarp();
            stage_scan(cc2, sb);
            cp_async_wait<0>();
            compare(sb, tied);
            sb ^= 1;
        };
        seeds(all);
        kept(all, tied);
#ifdef PCD_SWEEP_TRACE
        ++n_tie;
#endif
    }
#ifdef PCD_SWEEP_TRACE
    if (g_prune_count && lane == 0) {
        atomicAdd(g_prune_count, 1ull);
        atomicAdd(g_prune_count + 1, n_eval);
        atomicAdd(g_prune_count + 2, n_scan);
        atomicAdd(g_prune_count + 3, n_tie);
    }
#endif

    if (valid) {
        const int p = __ldg(a.bperm + own + slot);
        const uint32_t t = (uint32_t)arg;
        // the sweep's conventions: a row always publishes its minimum, a column only a finite one
        if (SIDE == 0) a.rowkey[(size_t)b * a.Npad + p] = make_key(best, t);
        else a.colkey[(size_t)b * a.Mpad + p] = best < pinf ? make_key(best, t) : ~0ull;
    }
}

template <int FORM>
__global__ void __launch_bounds__(kPruneThreads, 3) nn1_pruned_sweep_kernel(PruneArgs a) {
    __shared__ __align__(16) float4 ring[kPruneThreads / 32][3 * 32];      // candidate records in flight and under evaluation
    __shared__ __align__(16) float4 stage[kPruneThreads / 32][2 * 32];     // the arg-min passes' records and indices
    __shared__ int jstage[kPruneThreads / 32][2 * 32];
    pdl_launch_dependents();
    pdl_wait();                   // records, boxes, permutation and the queue cursor come from nn1_bucket
    for (;;) {
        // recomputed per item from the special and constant-bank registers: nothing stays live across an item
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        const int ncr = (a.N + 31) >> 5, per_b = ncr + ((a.M + 31) >> 5);
        int item = 0;
        if (lane == 0) item = atomicAdd(a.queue, 1);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= a.B * per_b) break;
        const int b = item / per_b, r = item - b * per_b;
        if (r < ncr) pruned_item<FORM, 0>(a, b, r, ring[warp], stage[warp], jstage[warp], lane);
        else pruned_item<FORM, 1>(a, b, r - ncr, ring[warp], stage[warp], jstage[warp], lane);
    }
}

// ----------------------------------------------------------------------------------- sweep
// Lane l of warp w of the CTA working on row tile qt owns the R consecutive rows
//     i = qt*QT + w*32R + l*R + r,  r < R
// Row direction: running minimum per row over 32-column chunks, tag = chunk index.
// Column direction: per column the lane folds its R rows (FMNMX3), CREDUX gives the warp
// minimum, FSETP+VOTE the ballot of the lanes that hold it; (value, ballot) goes to shared
// memory and the per-tile flush turns the lowest set lane into the tag
//     tag = (qt*4 + w)*32 + lane      ->  the R rows of that lane.
//
// Operand sources (SweepSrc): RAW = the caller's dense tensors.  Column tiles arrive as raw xyz
// (point-major: one 3 KB bulk copy, channel-major: three 1 KB copies) and are turned into pair
// records + norms in shared memory one tile AHEAD of the math, in front of the barrier that
// ends a tile anyway (25 instructions per thread and tile); the CTA's row tile arrives by one
// bulk copy per tile change and is pulled into registers from shared memory.  PACKED = the
// records nn1_prep wrote (strided inputs, swapped norms).
struct SweepSrc {
    const float *rows; long long r_sb, r_sc;   // RAW: batch stride, channel stride (channel-major) in floats
    const float *cols; long long c_sb, c_sc;
    int row_cm, col_cm;                         // 1 = channel-major [B,3,N], 0 = point-major [B,N,3]
    int norm_kind;
    const float4 *rowpp, *colpk;                // PACKED
};

template <int R>
struct SweepSmem {
    float4 tile[2][kMaxColTile + 2];                 // column pair-records (TMA destination / converted) + prefetch pad
    uint2 colpart[2][kSweepWarps][kMaxColTile];      // per-warp (column minimum, lane ballot)
    float craw[2][kMaxColTile * 3];                  // RAW: column xyz as it lies in the caller's tensor
    float rraw[kSweepWarps * 32 * R * 3];            // RAW: xyz of the CTA's row tile
    uint64_t full[2];                                // mbarriers: tile[s] / craw[s] has landed
    uint64_t rfull;                                  // mbarrier: rraw has landed
};
template <int R>
struct SweepSmemPacked {
    float4 tile[2][kMaxColTile + 2];
    uint2 colpart[2][kSweepWarps][kMaxColTile];
    uint64_t full[2];
};

constexpr int kQuad = 4;   // columns per scheduling unit (two packed steps)

template <int FORM, int R, bool RAW>
__global__ void __launch_bounds__(kSweepThreads, (R >= 16) ? 2 : ((R >= 8) ? 4 : ((R >= 4) ? 5 : 6)))
nn1_sweep_kernel(SweepSrc src, unsigned long long *__restrict__ rowkey, unsigned long long *__restrict__ colkey,
                 int N, int Npad, int Mpad, int qpt /* quads per TMA tile */, int nqt, int nq /* quads per row tile */,
                 int units) {
    constexpr int QW = 32 * R;            // rows per warp
    constexpr int QT = kSweepWarps * QW;  // rows per CTA tile
    constexpr int kQuadsPerChunk = kColChunk / kQuad;
    using Smem = typename std::conditional<RAW, SweepSmem<R>, SweepSmemPacked<R>>::type;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Smem &sm = *reinterpret_cast<Smem *>(smem_raw);

    pdl_launch_dependents();   // the fix-up may be scheduled as soon as SM resources free up; it waits for our completion
    if (!RAW) pdl_wait();      // PACKED: every operand is written by nn1_prep, the kernel in front of us

    // Stream-K at 4-column granularity: the (sample, row tile, column quad) space is cut into
    // gridDim.x equal contiguous ranges, so every CTA sweeps the same number of pairs (+-1 quad).
    // Ranges may start or end inside a 32-column chunk: a row tag only says "the minimum is in
    // this chunk", and the fix-up re-scans the whole chunk, so partial chunks stay exact.
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#ifdef PCD_SWEEP_TRACE
    unsigned long long *trace = g_sweep_trace;
    if (trace && tid == 0) {
        unsigned int smid;
        asm volatile("mov.u32 %0, %smid;" : "=r"(smid));
        trace[blockIdx.x * 8 + 0] = globaltimer_ns();
        trace[blockIdx.x * 8 + 3] = smid;
    }
#endif
    const int u0 = (int)((long long)units * blockIdx.x / gridDim.x);
    const int u1 = (int)((long long)units * (blockIdx.x + 1) / gridDim.x);
    if (u0 >= u1) return;

    // a segment = the quads [u, u+n) that share one row tile and one qpt-aligned column tile
    auto seg_len = [&](int u) -> int {
        const int q = u % nq;
        int e = (q / qpt + 1) * qpt;
        if (e > nq) e = nq;
        const int n = e - q;
        return n < u1 - u ? n : u1 - u;
    };
    int pu = u0;   // producer cursor (thread 0)
    auto issue = [&](int buf) {
        if (pu >= u1) return;
        const int bq = pu / nq, q = pu - bq * nq, b = bq / nqt;
        const int n = seg_len(pu);
        if constexpr (RAW) {
            const uint32_t ncols = (uint32_t)n * kQuad;
            mbar_expect_tx(&sm.full[buf], ncols * 12u);
            if (src.col_cm) {
                const float *g = src.cols + (size_t)b * src.c_sb + (size_t)q * kQuad;
#pragma unroll
                for (int c = 0; c < 3; ++c)
                    tma_load_1d(sm.craw[buf] + c * kMaxColTile, g + (size_t)c * src.c_sc, ncols * 4u, &sm.full[buf]);
            } else {
                tma_load_1d(sm.craw[buf], src.cols + (size_t)b * src.c_sb + (size_t)q * kQuad * 3, ncols * 12u, &sm.full[buf]);
            }
        } else {
            const uint32_t bytes = (uint32_t)n * kQuad * 16u;
            mbar_expect_tx(&sm.full[buf], bytes);
            tma_load_1d(sm.tile[buf], src.colpk + (size_t)b * Mpad + (size_t)q * kQuad, bytes, &sm.full[buf]);
        }
        pu += n;
    };
    // RAW: bulk copy of the valid rows of row tile bq into rraw
    auto issue_rows = [&](int bq) {
        if constexpr (RAW) {
            const int b = bq / nqt, qt = bq - b * nqt;
            int nv = N - qt * QT;
            if (nv > QT) nv = QT;
            mbar_expect_tx(&sm.rfull, (uint32_t)nv * 12u);
            if (src.row_cm) {
                const float *g = src.rows + (size_t)b * src.r_sb + (size_t)qt * QT;
#pragma unroll
                for (int c = 0; c < 3; ++c)
                    tma_load_1d(sm.rraw + c * QT, g + (size_t)c * src.r_sc, (uint32_t)nv * 4u, &sm.rfull);
            } else {
                tma_load_1d(sm.rraw, src.rows + (size_t)b * src.r_sb + (size_t)qt * QT * 3, (uint32_t)nv * 12u, &sm.rfull);
            }
        }
    };
    // RAW: craw[s] (ncols raw columns) -> pair records {x0,x1,y0,y1},{z0,z1,n0,n1} in tile[d]
    auto convert = [&](int s, int d, int ncols) {
        if constexpr (RAW) {
            const int p = tid;                               // pair record index; ncols is a multiple of 4
            if (2 * p < ncols) {
                float x0, y0, z0, x1, y1, z1;
                if (src.col_cm) {
                    const float2 xs = *reinterpret_cast<const float2 *>(&sm.craw[s][2 * p]);
                    const float2 ys = *reinterpret_cast<const float2 *>(&sm.craw[s][kMaxColTile + 2 * p]);
                    const float2 zs = *reinterpret_cast<const float2 *>(&sm.craw[s][2 * kMaxColTile + 2 * p]);
                    x0 = xs.x; x1 = xs.y; y0 = ys.x; y1 = ys.y; z0 = zs.x; z1 = zs.y;
                } else {
                    const float2 *f = reinterpret_cast<const float2 *>(&sm.craw[s][6 * p]);
                    const float2 a = f[0], bb = f[1], c = f[2];
                    x0 = a.x; y0 = a.y; z0 = bb.x; x1 = bb.y; y1 = c.x; z1 = c.y;
                }
                const float n0 = sq_norm3(src.norm_kind, x0, y0, z0), n1 = sq_norm3(src.norm_kind, x1, y1, z1);
                sm.tile[d][2 * p] = make_float4(x0, x1, y0, y1);
                sm.tile[d][2 * p + 1] = make_float4(z0, z1, n0, n1);
            }
        }
    };
    if (tid == 0) {
        mbar_init(&sm.full[0], 1);
        mbar_init(&sm.full[1], 1);
        if constexpr (RAW) mbar_init(&sm.rfull, 1);
        fence_mbar_init();
        fence_proxy_async();
        issue(0);
        issue(1);
        issue_rows(u0 / nq);
    }
    __syncthreads();
    if constexpr (RAW) {
        // tile 0: convert in front of the loop; its raw buffer is then free for tile 2
        mbar_wait(&sm.full[0], 0);
        convert(0, 0, seg_len(u0) * kQuad);
        __syncthreads();
        if (tid == 0) issue(0);
    }

    float qx[R], qy[R], qz[R], qn[R], best[R];
    uint32_t btag[R];
    int cur_bq = -1;
    size_t row_base = 0;
    uint32_t rpar = 0;
    bool armed = !RAW;     // RAW: griddepcontrol.wait not executed yet (keys are armed by our predecessor)
    const float pinf = __int_as_float(0x7f800000);
    // publish the running row minima of the current row tile
    auto flush_rows = [&]() {
#pragma unroll
        for (int r = 0; r < R; ++r) atomicMin(&rowkey[row_base + r * 32], make_key(best[r], btag[r]));
    };
#ifdef PCD_SWEEP_TRACE
    long long t_row = 0, t_comp = 0, t_bar = 0, t_flush = 0, t_mark = clock64();
#define PCD_PHASE(acc) do { const long long _n = clock64(); acc += _n - t_mark; t_mark = _n; } while (0)
#else
#define PCD_PHASE(acc) do { } while (0)
#endif
    int it = 0;
    for (int u = u0; u < u1; ++it) {
        const int buf = it & 1;
        const int bq = u / nq, q0 = u - bq * nq;
        const int b = bq / nqt, qt = bq - b * nqt;
        const int nseg = seg_len(u);
        bool pulled = false;

        if (bq != cur_bq) {
            if (cur_bq >= 0) flush_rows();
            cur_bq = bq;
            row_base = (size_t)b * Npad + (size_t)qt * QT + warp * QW + lane;    // key slot of row r: + r*32
            if constexpr (RAW) {
                mbar_wait(&sm.rfull, rpar);
                rpar ^= 1u;
                pulled = true;
                const int l0 = warp * QW + lane * R;            // first of this lane's rows inside the tile
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    float x = 0.f, y = 0.f, z = 0.f, n = __int_as_float(0x7f800000);
                    if (qt * QT + l0 + r < N) {
                        if (src.row_cm) { x = sm.rraw[l0 + r]; y = sm.rraw[QT + l0 + r]; z = sm.rraw[2 * QT + l0 + r]; }
                        else { x = sm.rraw[(l0 + r) * 3]; y = sm.rraw[(l0 + r) * 3 + 1]; z = sm.rraw[(l0 + r) * 3 + 2]; }
                        n = sq_norm3(src.norm_kind, x, y, z);
                    }
                    qx[r] = -2.f * x; qy[r] = -2.f * y; qz[r] = -2.f * z; qn[r] = n;
                    best[r] = __int_as_float(0x7f800000);
                    btag[r] = 0;
                }
            } else {
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const float4 q = __ldg(&src.rowpp[row_base + r * 32]);
                    qx[r] = q.x; qy[r] = q.y; qz[r] = q.z; qn[r] = q.w;
                    best[r] = __int_as_float(0x7f800000);
                    btag[r] = 0;
                }
            }
        }

        if constexpr (!RAW) mbar_wait(&sm.full[buf], (it >> 1) & 1);
#ifdef PCD_SWEEP_TRACE
        if (trace && tid == 0 && it == 0) trace[blockIdx.x * 8 + 4] = globaltimer_ns();
#endif
        PCD_PHASE(t_row);

        const float4 *t4 = sm.tile[buf];
        uint2 *cp = sm.colpart[buf][warp];
        float4 A = t4[0], Bv = t4[1];                       // operands of the step about to run
        uint2 pend_lo = make_uint2(0x7f800000u, 0u), pend_hi = pend_lo;   // column results of the previous step
        int pend_at = -1;
        int qd = 0;                                          // quad cursor inside the segment
        while (qd < nseg) {
            // piece = the quads of this segment that fall into one 32-column chunk
            const int chunk = (q0 + qd) / kQuadsPerChunk;
            int pe = (chunk + 1) * kQuadsPerChunk - q0;
            if (pe > nseg) pe = nseg;
            float m[R];
#pragma unroll
            for (int r = 0; r < R; ++r) m[r] = __int_as_float(0x7f800000);
            for (; qd < pe; ++qd) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int step = qd * 2 + h;
                    const float4 An = t4[step * 2 + 2], Bn = t4[step * 2 + 3];   // prefetch (pad keeps it in bounds)
                    const f32x2 X = pack2(A.x, A.y), Y = pack2(A.z, A.w);
                    const f32x2 Z = pack2(Bv.x, Bv.y), Nn = pack2(Bv.z, Bv.w);
                    float lo[R], hi[R];
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const f32x2 d = pair_dist_x2<FORM>(qx[r], qy[r], qz[r], qn[r], X, Y, Z, Nn);
                        unpack2(d, lo[r], hi[r]);
                        m[r] = min3(m[r], lo[r], hi[r]);
                    }
                    float clo = lo[0], chi = hi[0];
#pragma unroll
                    for (int r = 1; r + 1 < R; r += 2) {
                        clo = min3(clo, lo[r], lo[r + 1]);
                        chi = min3(chi, hi[r], hi[r + 1]);
                    }
                    if ((R & 1) == 0) {
                        clo = fminf(clo, lo[R - 1]);
                        chi = fminf(chi, hi[R - 1]);
                    }
                    // retire the previous step's column results (their CREDUX latency is long gone)
                    if (pend_at >= 0) *reinterpret_cast<uint4 *>(&cp[pend_at]) = make_uint4(pend_lo.x, pend_lo.y, pend_hi.x, pend_hi.y);
                    const float vlo = warp_min_f32(clo), vhi = warp_min_f32(chi);
                    pend_lo = make_uint2(__float_as_uint(vlo), __ballot_sync(0xffffffffu, clo == vlo));
                    pend_hi = make_uint2(__float_as_uint(vhi), __ballot_sync(0xffffffffu, chi == vhi));
                    pend_at = 2 * step;
                    A = An; Bv = Bn;
                }
            }
#pragma unroll
            for (int r = 0; r < R; ++r) {
                if (m[r] < best[r]) {
                    best[r] = m[r];
                    btag[r] = (uint32_t)chunk;
                }
            }
        }
        *reinterpret_cast<uint4 *>(&cp[pend_at]) = make_uint4(pend_lo.x, pend_lo.y, pend_hi.x, pend_hi.y);
        PCD_PHASE(t_comp);

        if constexpr (RAW) {
            // next tile: raw xyz -> pair records, in front of the barrier that ends this tile
            // (tile[buf^1] was last read one barrier ago)
            if (u + nseg < u1) {
                mbar_wait(&sm.full[buf ^ 1], ((it + 1) >> 1) & 1);
                convert(buf ^ 1, buf ^ 1, seg_len(u + nseg) * kQuad);
            }
        }
        __syncthreads();  // tile[buf] fully read, colpart[buf] fully written, RAW: tile[buf^1] converted, craw[buf^1] and rraw free
        PCD_PHASE(t_bar);

        if (tid == 0) {
            if constexpr (RAW) {
                issue(buf ^ 1);                                   // raw tile it+3 into the buffer just converted
                if (pulled && (long long)(bq + 1) * nq < u1) issue_rows(bq + 1);
            } else {
                issue(buf);
            }
        }
        if (!armed) {
            pdl_wait();   // keys are reset by the kernel in front of us; everything up to here overlapped it
            armed = true;
        }
        // column flush: min over the CTA's warps (lowest warp on ties), lowest lane of its ballot
        const int ncols = nseg * kQuad;
        for (int col = tid; col < ncols; col += kSweepThreads) {
            uint2 e = sm.colpart[buf][0][col];
            float v = __uint_as_float(e.x);
            uint32_t w = 0, msk = e.y;
#pragma unroll
            for (int k = 1; k < kSweepWarps; ++k) {
                const uint2 o = sm.colpart[buf][k][col];
                const float ov = __uint_as_float(o.x);
                if (ov < v) { v = ov; w = k; msk = o.y; }
            }
            const uint32_t ctag = (((uint32_t)qt * kSweepWarps + w) << 5) + (uint32_t)((__ffs(msk) - 1) & 31);
            if (v < pinf) atomicMin(&colkey[(size_t)b * Mpad + (size_t)q0 * kQuad + col], make_key(v, ctag));
        }
        u += nseg;
        PCD_PHASE(t_flush);
    }
#ifdef PCD_SWEEP_TRACE
    if (trace && tid == 0) {
        trace[blockIdx.x * 8 + 1] = globaltimer_ns();
        // phase cycles of warp 0: row switch | compute | convert + barrier wait | flush  (16 bits each, in units of 64 cycles)
        trace[blockIdx.x * 8 + 5] = (unsigned long long)t_row; trace[blockIdx.x * 8 + 6] = (unsigned long long)t_comp;
        trace[blockIdx.x * 8 + 7] = ((unsigned long long)t_bar << 32) | (unsigned long long)(t_flush & 0xffffffffll);
    }
#endif
    flush_rows();
#ifdef PCD_SWEEP_TRACE
    __syncthreads();
    if (trace && tid == 0) trace[blockIdx.x * 8 + 2] = globaltimer_ns();
#endif
}

// --------------------------------------------------------------------- fix-up + reduction
__device__ __forceinline__ float apply_transform(int transform, float v) {
    return transform == PCD_VALUE_SQRT_CLAMP ? sqrtf(fmaxf(v, 0.0f)) : v;
}

__device__ __forceinline__ void reduce_smf(float &s, float &mx, int &am) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        const float om = __shfl_xor_sync(0xffffffffu, mx, o);
        const int oa = __shfl_xor_sync(0xffffffffu, am, o);
        if (om > mx || (om == mx && oa < am)) { mx = om; am = oa; }
    }
}

struct FixupArgs {
    // operands: RAW = the caller's tensors (element strides), PACKED = nn1_prep's records
    const float *rows; long long r_sb, r_sp, r_sc;
    const float *cols; long long c_sb, c_sp, c_sc;
    const float4 *rowpk, *colpk;
    int col_vec;                  // RAW: 1 = point-major dense columns, 2 = channel-major dense columns (16-byte loads)
    int norm_kind;
    const unsigned long long *rowkey, *colkey;
    int *counters;                // [B] octets finished per sample (armed to 0)
    float4 *partials;             // [B][slots]: per 32-point unit (rows first, then columns) the (sum, max, bits of argmax) of its minima
    int slots;                    // units per sample
    int nwarps;                   // participating warps W (<= number of octets U)
    int upw, urem;                // U / W, U % W: warp w owns upw (+1 if w < urem) consecutive octets
    int nrowgroups;               // ceil(N / 32R): valid range of the lane-group part of a column tag
    int nchunks;                  // ceil(M / 32): valid range of a row tag
    int N, M, Npad, Mpad, R, transform, B;
    float *row_min; int32_t *row_arg; float *col_min; int32_t *col_arg;
    float row_scale, col_scale;
    float *stats_f; int32_t *stats_i;
    float4 *zero0; size_t nzero0; float4 *zero1; size_t nzero1;     // optional buffers to clear (float4 counts)
    int pruned;                   // keys from nn1_pruned_sweep: at the original index, tag = the arg-min itself
};


// Persistent, barrier-free fix-up, ONE LANE PER POINT.  A row point re-evaluates the 32 columns of its
// winning chunk, a column point the R rows of its winning lane -- with the sweep's exact arithmetic --
// and takes the lowest index whose distance equals the minimum.  The scan of a point is a straight
// stream of 16-byte loads and scalar math in its own lane (groups of four candidates, highest first so
// that the lowest match is the one that sticks): no cross-lane traffic, every lane busy -- the earlier
// four-lanes-per-point kernels spent five of six instructions on addressing and shuffles.
// Work unit = 32 consecutive points of one side of one sample; every warp owns a contiguous range of
// units (sample-major, rows then columns) and requests the key and the own coordinates of unit u+1
// before it evaluates unit u, so the key -> chunk round trips of consecutive units overlap.
// A key that was never lowered (every distance through the point NaN or +inf) decodes to
// (NaN, tag 0xffffffff): nothing is dereferenced through such a tag, the point gets arg 0.
// Per-sample statistics: lane-local running (sum, max, first argmax) over the warp's units of one
// sample and side, one xor-tree per segment, one partial per (sample, side, warp); the warp whose
// completion count closes a sample folds that sample's partials -- all in a fixed order, so the
// sums are run-to-run deterministic.
// Statistics of one sample from its unit partials, by one warp per side: lane-strided over the units in
// index order, then the xor tree -- an order that depends on nothing but (N, M), so a sample's sums are
// bit-identical whatever the batch size, the launch geometry or the operand path.
__device__ __forceinline__ void fold_sample_side(const FixupArgs &a, int b, int side, int lane) {
    const float ninf = -__int_as_float(0x7f800000);
    const int urow = (a.N + 31) >> 5, ucol = (a.M + 31) >> 5;
    const int first = side ? urow : 0, count = side ? ucol : urow;
    float sv = 0.f, mx = ninf;
    int am = 0x7fffffff;
    for (int k = lane; k < count; k += 32) {
        const float4 t = __ldcg(&a.partials[(size_t)b * a.slots + first + k]);
        sv += t.x;
        const int ta = __float_as_int(t.z);
        if (t.y > mx || (t.y == mx && ta < am)) { mx = t.y; am = ta; }
    }
    reduce_smf(sv, mx, am);
    if (lane == 0) {
        a.stats_f[(side * 2 + 0) * a.B + b] = sv * (side ? a.col_scale : a.row_scale);
        a.stats_f[(side * 2 + 1) * a.B + b] = mx;
        a.stats_i[side * a.B + b] = am == 0x7fffffff ? 0 : am;
    }
}
// the partial of one unit: xor tree over its 32 lanes (dead lanes are neutral)
__device__ __forceinline__ void store_unit_partial(const FixupArgs &a, int b, int unit_in_sample, bool live, float val, int p, int lane) {
    float sv = live ? val : 0.f, mx = live ? val : -__int_as_float(0x7f800000);
    int am = live ? p : 0x7fffffff;
    reduce_smf(sv, mx, am);
    if (lane == 0) a.partials[(size_t)b * a.slots + unit_in_sample] = make_float4(sv, mx, __int_as_float(am), 0.f);
}

struct FixPt {
    int b, p;
    bool live, is_col;
    unsigned long long key;
    float ox, oy, oz, on;
};

// lowest column j in [j0, j0+32) with d(row record, column j) == v   (0x7fffffff: none)
template <int FORM, bool RAW, int NORM>
__device__ __forceinline__ int fixup_scan_cols(const FixupArgs &a, int b, int j0, float qx, float qy, float qz, float qn, float v) {
    int arg = 0x7fffffff;
    if (RAW) {
        int ng = (a.M - j0 + 3) >> 2;                 // valid groups of 4 columns (M % 4 == 0)
        if (ng > 8) ng = 8;
        if (a.col_vec == 1) {                         // point-major: 4 columns = 12 consecutive floats
            const float4 *g = reinterpret_cast<const float4 *>(a.cols + (size_t)b * a.c_sb + (size_t)j0 * 3);
#pragma unroll 4
            for (int k = ng - 1; k >= 0; --k) {
                const float4 f0 = __ldg(g + 3 * k), f1 = __ldg(g + 3 * k + 1), f2 = __ldg(g + 3 * k + 2);
                const float cx[4] = {f0.x, f0.w, f1.z, f2.y}, cy[4] = {f0.y, f1.x, f1.w, f2.z}, cz[4] = {f0.z, f1.y, f2.x, f2.w};
#pragma unroll
                for (int t = 3; t >= 0; --t)
                    if (pair_dist_scalar<FORM>(qx, qy, qz, qn, cx[t], cy[t], cz[t], sq_norm3(NORM, cx[t], cy[t], cz[t])) == v) arg = j0 + 4 * k + t;
            }
        } else {                                      // channel-major: 4 columns = one float4 per channel
            const float *g = a.cols + (size_t)b * a.c_sb + j0;
#pragma unroll 4
            for (int k = ng - 1; k >= 0; --k) {
                const float4 fx = __ldg(reinterpret_cast<const float4 *>(g) + k);
                const float4 fy = __ldg(reinterpret_cast<const float4 *>(g + a.c_sc) + k);
                const float4 fz = __ldg(reinterpret_cast<const float4 *>(g + 2 * a.c_sc) + k);
                const float cx[4] = {fx.x, fx.y, fx.z, fx.w}, cy[4] = {fy.x, fy.y, fy.z, fy.w}, cz[4] = {fz.x, fz.y, fz.z, fz.w};
#pragma unroll
                for (int t = 3; t >= 0; --t)
                    if (pair_dist_scalar<FORM>(qx, qy, qz, qn, cx[t], cy[t], cz[t], sq_norm3(NORM, cx[t], cy[t], cz[t])) == v) arg = j0 + 4 * k + t;
            }
        }
    } else {                                          // packed pair records {x0,x1,y0,y1},{z0,z1,n0,n1}; padded, inert beyond M
        const float4 *rec = a.colpk + (size_t)b * a.Mpad + j0;
#pragma unroll 4
        for (int k = 7; k >= 0; --k) {
            const float4 a0 = __ldg(rec + 4 * k), c0 = __ldg(rec + 4 * k + 1), a1 = __ldg(rec + 4 * k + 2), c1 = __ldg(rec + 4 * k + 3);
            const int j = j0 + 4 * k;
            if (pair_dist_scalar<FORM>(qx, qy, qz, qn, a1.y, a1.w, c1.y, c1.w) == v) arg = j + 3;
            if (pair_dist_scalar<FORM>(qx, qy, qz, qn, a1.x, a1.z, c1.x, c1.z) == v) arg = j + 2;
            if (pair_dist_scalar<FORM>(qx, qy, qz, qn, a0.y, a0.w, c0.y, c0.w) == v) arg = j + 1;
            if (pair_dist_scalar<FORM>(qx, qy, qz, qn, a0.x, a0.z, c0.x, c0.z) == v) arg = j;
        }
    }
    return arg;
}

// lowest row i in [i0, i0+R) with d(row i, column record) == v
template <int FORM, bool RAW, int NORM>
__device__ __forceinline__ int fixup_scan_rows(const FixupArgs &a, int b, int i0, float cx, float cy, float cz, float cn, float v) {
    int arg = 0x7fffffff;
    const int R = a.R, N = a.N;
    if (RAW) {
        if (R >= 4) {                                 // groups of 4 rows: three 16-byte loads in either dense layout (N % 4 == 0)
            int ng = (N - i0 + 3) >> 2;
            if (ng > (R >> 2)) ng = R >> 2;
            if (a.r_sp == 3) {
                const float4 *g = reinterpret_cast<const float4 *>(a.rows + (size_t)b * a.r_sb + (size_t)i0 * 3);
#pragma unroll 4
                for (int k = ng - 1; k >= 0; --k) {
                    const float4 f0 = __ldg(g + 3 * k), f1 = __ldg(g + 3 * k + 1), f2 = __ldg(g + 3 * k + 2);
                    const float x[4] = {f0.x, f0.w, f1.z, f2.y}, y[4] = {f0.y, f1.x, f1.w, f2.z}, z[4] = {f0.z, f1.y, f2.x, f2.w};
#pragma unroll
                    for (int t = 3; t >= 0; --t)
                        if (pair_dist_scalar<FORM>(-2.f * x[t], -2.f * y[t], -2.f * z[t], sq_norm3(NORM, x[t], y[t], z[t]), cx, cy, cz, cn) == v) arg = i0 + 4 * k + t;
                }
            } else {
                const float *g = a.rows + (size_t)b * a.r_sb + i0;
#pragma unroll 4
                for (int k = ng - 1; k >= 0; --k) {
                    const float4 fx = __ldg(reinterpret_cast<const float4 *>(g) + k);
                    const float4 fy = __ldg(reinterpret_cast<const float4 *>(g + a.r_sc) + k);
                    const float4 fz = __ldg(reinterpret_cast<const float4 *>(g + 2 * a.r_sc) + k);
                    const float x[4] = {fx.x, fx.y, fx.z, fx.w}, y[4] = {fy.x, fy.y, fy.z, fy.w}, z[4] = {fz.x, fz.y, fz.z, fz.w};
#pragma unroll
                    for (int t = 3; t >= 0; --t)
                        if (pair_dist_scalar<FORM>(-2.f * x[t], -2.f * y[t], -2.f * z[t], sq_norm3(NORM, x[t], y[t], z[t]), cx, cy, cz, cn) == v) arg = i0 + 4 * k + t;
                }
            }
        } else {                                      // R = 2
            for (int t = R - 1; t >= 0; --t) {
                const int i = i0 + t;
                if (i < N) {
                    const float *s = a.rows + (size_t)b * a.r_sb + (size_t)i * a.r_sp;
                    const float x = __ldg(s), y = __ldg(s + a.r_sc), z = __ldg(s + 2 * a.r_sc);
                    if (pair_dist_scalar<FORM>(-2.f * x, -2.f * y, -2.f * z, sq_norm3(NORM, x, y, z), cx, cy, cz, cn) == v) arg = i;
                }
            }
        }
    } else {
        const float4 *rq = a.rowpk + (size_t)b * a.Npad + i0;
#pragma unroll 4
        for (int t = R - 1; t >= 0; --t) {
            const float4 q = __ldg(rq + t);
            if (i0 + t < N && pair_dist_scalar<FORM>(q.x, q.y, q.z, q.w, cx, cy, cz, cn) == v) arg = i0 + t;
        }
    }
    return arg;
}

template <int FORM, bool RAW, int NORM>
__global__ void __launch_bounds__(kFixupThreads, kFixupCtasPerSm)
nn1_fixup_kernel(FixupArgs a) {
    const int tid = threadIdx.x, lane = tid & 31;
    const int N = a.N, M = a.M, R = a.R;
    const float ninf = -__int_as_float(0x7f800000);

    if (!RAW) pdl_wait();     // PACKED: the records come from nn1_prep (complete once the sweep has started its math)
    // optional zero fill (gradient buffers of the coming backward); independent of the kernels in front of us
    {
        const size_t nthreads = (size_t)gridDim.x * kFixupThreads;
        const size_t t0 = (size_t)blockIdx.x * kFixupThreads + tid;
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        for (size_t t = t0; t < a.nzero0; t += nthreads) a.zero0[t] = z;
        for (size_t t = t0; t < a.nzero1; t += nthreads) a.zero1[t] = z;
    }
    const int w = blockIdx.x * (kFixupThreads / 32) + (tid >> 5);
    if (w >= a.nwarps) return;
    const int urow = (N + 31) >> 5, ucol = (M + 31) >> 5, Us = urow + ucol;    // units per sample
    // warp w owns the units [w*upw + min(w, urem), ... + upw (+1 if w < urem)): no division in the hot path
    const int u_begin = w * a.upw + min(w, a.urem), u_end = u_begin + a.upw + (w < a.urem ? 1 : 0);
    // request everything of unit (b, o) that does not depend on another load: key and own coordinates of this lane's point
    auto fetch = [&](int b_, int o) -> FixPt {
        FixPt f;
        f.b = b_;
        f.is_col = o >= urow;
        f.p = (f.is_col ? o - urow : o) * 32 + lane;
        f.live = f.p < (f.is_col ? M : N);
        f.key = 0ull; f.ox = f.oy = f.oz = f.on = 0.f;
        if (f.live) {
            f.key = f.is_col ? a.colkey[(size_t)f.b * a.Mpad + f.p]
                             : a.rowkey[(size_t)f.b * a.Npad + (a.pruned ? f.p : row_slot(f.p, R))];
            if (RAW) {
                const float *s = f.is_col ? a.cols + (size_t)f.b * a.c_sb + (size_t)f.p * a.c_sp
                                          : a.rows + (size_t)f.b * a.r_sb + (size_t)f.p * a.r_sp;
                const long long sc = f.is_col ? a.c_sc : a.r_sc;
                f.ox = __ldg(s); f.oy = __ldg(s + sc); f.oz = __ldg(s + 2 * sc);
            } else if (f.is_col) {
                const float *rec = reinterpret_cast<const float *>(a.colpk) + ((size_t)f.b * a.Mpad + (f.p & ~1)) * 4 + (f.p & 1);
                f.ox = rec[0]; f.oy = rec[2]; f.oz = rec[4]; f.on = rec[6];
            } else {
                const float4 q = __ldg(&a.rowpk[(size_t)f.b * a.Npad + f.p]);
                f.ox = q.x; f.oy = q.y; f.oz = q.z; f.on = q.w;
            }
        }
        return f;
    };

    if (RAW) pdl_wait();      // the keys: the sweep has completed and flushed

    // close the warp's segment of sample b: completion count, and -- if we are last -- the sample's statistics
    auto finish_sample = [&](int b) {
        const int s0 = b * Us, s1 = s0 + Us;                                     // the sample's unit range
        int last = 0;
        if (lane == 0) {
            const int done = min(u_end, s1) - max(u_begin, s0);
            __threadfence();
            last = atomicAdd(&a.counters[b], done) + done == Us;
        }
        last = __shfl_sync(0xffffffffu, last, 0);
        if (!last) return;
        __threadfence();
        fold_sample_side(a, b, 0, lane);
        fold_sample_side(a, b, 1, lane);
    };

    int nb = u_begin / Us, no = u_begin - nb * Us;        // (sample, unit in sample) of the NEXT unit to fetch
    FixPt cur = fetch(nb, no);
    for (int u = u_begin; u < u_end; ++u) {
        FixPt nxt = cur;
        if (++no == Us) { no = 0; ++nb; }
        if (u + 1 < u_end) nxt = fetch(nb, no);
        const int b = cur.b, p = cur.p;
        float val = 0.f;
        if (cur.live) {
            const float v = ordered_to_f32((uint32_t)(cur.key >> 32));
            const uint32_t tag = (uint32_t)cur.key;
            float ox = cur.ox, oy = cur.oy, oz = cur.oz, on = cur.on;
            if (RAW) on = sq_norm3(NORM, ox, oy, oz);
            int arg = 0x7fffffff;
            const bool finite = v < __int_as_float(0x7f800000);       // a non-finite minimum has no arg-min (arg 0)
            if (!cur.is_col && RAW) { ox *= -2.f; oy *= -2.f; oz *= -2.f; }
            if (RAW && a.pruned) {
                if (finite) arg = (int)tag;
            } else if (!cur.is_col) {
                if (finite && tag < (uint32_t)a.nchunks) arg = fixup_scan_cols<FORM, RAW, NORM>(a, b, (int)tag * kColChunk, ox, oy, oz, on, v);
            } else if (finite && (tag >> 5) < (uint32_t)a.nrowgroups) {
                arg = fixup_scan_rows<FORM, RAW, NORM>(a, b, (int)(tag >> 5) * (32 * R) + (int)(tag & 31u) * R, ox, oy, oz, on, v);
            }
            if (arg == 0x7fffffff) arg = 0;        // no finite minimum (NaN / inf inputs)
            val = apply_transform(a.transform, v);
            if (!cur.is_col) { a.row_min[(size_t)b * N + p] = val; a.row_arg[(size_t)b * N + p] = arg; }
            else { a.col_min[(size_t)b * M + p] = val; a.col_arg[(size_t)b * M + p] = arg; }
        }
        store_unit_partial(a, b, u - b * Us, cur.live, val, p, lane);
        if (u + 1 == u_end || nxt.b != b) finish_sample(b);       // warp-uniform: every lane of a unit is in the same sample
        cur = nxt;
    }
}

// ---------------------------------------------------------------- fix-up, shared-memory staged
// The lane-per-point fix-up above is bound by L1 tag look-ups: every lane of a 16-byte load touches its
// own cache line (winning chunks of neighbouring points are unrelated), 4.7 M tag cycles at BASELINE
// config 2 = 16 us.  When the cloud that is being re-scanned fits into shared memory (N, M <= 16 K
// points) it is staged there once per CTA by bulk copies -- issued BEFORE the dependency wait, so
// they overlap the tail of the sweep -- and the scans become bank-conflict-free LDS.128 streams:
//   job    = (sample b, side): side 0 = the rows re-scan columns (stage the column cloud),
//                              side 1 = the columns re-scan rows (stage the row cloud)
//   slice  = `parts` equal unit ranges per job (unit = 32 points, one per lane); one CTA per slice
//   order  = lane l visits its point's candidate groups rotated by l (group (l + i) mod G): the lanes of a
//            quarter warp then sit in different banks; the lowest matching index is kept with min().
// Statistics: lane-local -> warp xor-tree -> CTA (fixed warp order) -> one partial per slice; the CTA
// whose completion count closes a sample folds the 2 x parts partials in a fixed order.
struct StagedArgs {
    FixupArgs f;
    int parts_row, parts_col;   // slices per (sample, side): a row point scans 32 candidates, a column point R, so the
                                // sides get slice counts in proportion to their work
    int stage_stride;           // channel-major staging: floats between the channel rows (multiple of 32)
};

template <int FORM, int NORM>
__global__ void __launch_bounds__(kFixupThreads, 3)
nn1_fixup_staged_kernel(StagedArgs sa) {
    const FixupArgs &a = sa.f;
    extern __shared__ __align__(128) float stage[];
    __shared__ uint64_t bar;
    __shared__ int s_last;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int N = a.N, M = a.M, R = a.R;
    const int per_sample = sa.parts_row + sa.parts_col;
    const int b = blockIdx.x / per_sample, rem = blockIdx.x - b * per_sample;
    const int side = rem >= sa.parts_row ? 1 : 0, q = side ? rem - sa.parts_row : rem;
    const int parts = side ? sa.parts_col : sa.parts_row;
    const int n_own = side ? M : N, n_opp = side ? N : M;            // points of this side / candidates
    const float *own = side ? a.cols + (size_t)b * a.c_sb : a.rows + (size_t)b * a.r_sb;
    const long long own_sp = side ? a.c_sp : a.r_sp, own_sc = side ? a.c_sc : a.r_sc;
    const float *opp = side ? a.rows + (size_t)b * a.r_sb : a.cols + (size_t)b * a.c_sb;
    const bool opp_cm = (side ? a.r_sp : a.c_sp) == 1;
    const long long opp_sc = side ? a.r_sc : a.c_sc;

    if (tid == 0) {
        mbar_init(&bar, 1);
        fence_mbar_init();
        fence_proxy_async();
        mbar_expect_tx(&bar, (uint32_t)n_opp * 12u);
        if (opp_cm) {
#pragma unroll
            for (int c = 0; c < 3; ++c) tma_load_1d(stage + (size_t)c * sa.stage_stride, opp + (size_t)c * opp_sc, (uint32_t)n_opp * 4u, &bar);
        } else {
            tma_load_1d(stage, opp, (uint32_t)n_opp * 12u, &bar);
        }
    }
    {   // optional zero fill (gradient buffers of the coming backward)
        const size_t nthreads = (size_t)gridDim.x * kFixupThreads;
        const size_t t0 = (size_t)blockIdx.x * kFixupThreads + tid;
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        for (size_t t = t0; t < a.nzero0; t += nthreads) a.zero0[t] = z;
        for (size_t t = t0; t < a.nzero1; t += nthreads) a.zero1[t] = z;
    }
    __syncthreads();          // the barrier is initialised
    pdl_wait();               // the keys: the sweep has completed and flushed
    mbar_wait(&bar, 0);       // the candidate cloud is in shared memory

    const int units = (n_own + 31) >> 5;
    const int u0 = (int)((long long)units * q / parts), u1 = (int)((long long)units * (q + 1) / parts);
    const unsigned long long *keys = side ? a.colkey + (size_t)b * a.Mpad : a.rowkey + (size_t)b * a.Npad;
    float *out_min = side ? a.col_min + (size_t)b * M : a.row_min + (size_t)b * N;
    int32_t *out_arg = side ? a.col_arg + (size_t)b * M : a.row_arg + (size_t)b * N;

    // the key and the coordinates of a point are requested here, a unit ahead of its evaluation
    unsigned long long key = 0ull;
    float px = 0.f, py = 0.f, pz = 0.f;
    auto fetch = [&](int u, unsigned long long &k, float &x, float &y, float &z) {
        const int p = u * 32 + lane;
        k = 0ull; x = y = z = 0.f;
        if (u < u1 && p < n_own) {
            k = keys[side ? p : row_slot(p, R)];
            const float *s = own + (size_t)p * own_sp;
            x = __ldg(s); y = __ldg(s + own_sc); z = __ldg(s + 2 * own_sc);
        }
    };
    // four candidates j .. j+3 against one fixed point (m2 = -2 * its coordinates, fn = its norm): exact distances
    auto eval4 = [&](int j, float m2x, float m2y, float m2z, float fn, float &e0, float &e1, float &e2, float &e3) {
        f32x2 X0, X1, Y0, Y1, Z0, Z1;
        if (opp_cm) {
            const float4 fx = *reinterpret_cast<const float4 *>(stage + j);
            const float4 fy = *reinterpret_cast<const float4 *>(stage + sa.stage_stride + j);
            const float4 fz = *reinterpret_cast<const float4 *>(stage + 2 * sa.stage_stride + j);
            X0 = pack2(fx.x, fx.y); X1 = pack2(fx.z, fx.w);
            Y0 = pack2(fy.x, fy.y); Y1 = pack2(fy.z, fy.w);
            Z0 = pack2(fz.x, fz.y); Z1 = pack2(fz.z, fz.w);
        } else {
            const float4 *g = reinterpret_cast<const float4 *>(stage + (size_t)j * 3);
            const float4 f0 = g[0], f1 = g[1], f2 = g[2];
            X0 = pack2(f0.x, f0.w); X1 = pack2(f1.z, f2.y);
            Y0 = pack2(f0.y, f1.x); Y1 = pack2(f1.w, f2.z);
            Z0 = pack2(f0.z, f1.y); Z1 = pack2(f2.x, f2.w);
        }
        const f32x2 d0 = pair_dist_fixed_x2<FORM>(side == 0, m2x, m2y, m2z, fn, X0, Y0, Z0, sq_norm3_x2(NORM, X0, Y0, Z0));
        const f32x2 d1 = pair_dist_fixed_x2<FORM>(side == 0, m2x, m2y, m2z, fn, X1, Y1, Z1, sq_norm3_x2(NORM, X1, Y1, Z1));
        unpack2(d0, e0, e1); unpack2(d1, e2, e3);
    };
    fetch(u0 + warp, key, px, py, pz);
    for (int u = u0 + warp; u < u1; u += kFixupThreads / 32) {
        unsigned long long nkey; float nx, ny, nz;
        fetch(u + kFixupThreads / 32, nkey, nx, ny, nz);
        const int p = u * 32 + lane;
        float val = 0.f;
        const float pn = sq_norm3(NORM, px, py, pz);
        const float m2x = -2.f * px, m2y = -2.f * py, m2z = -2.f * pz;
        float bv = __int_as_float(0x7f800000);
        int arg = 0x7fffffff;
        if (p < n_own) {
            const float v = ordered_to_f32((uint32_t)(key >> 32));
            const uint32_t tag = (uint32_t)key;
            // Candidates come in groups of four (three LDS.128 in either dense layout) and are evaluated two at a time with the
            // sweep's packed instruction sequence; the fixed point carries the exact factor -2 whichever side it is on.
            int c0 = 0, ngroups = 0;                         // first candidate, groups of 4
            const bool scan = v < __int_as_float(0x7f800000);       // a non-finite minimum has no arg-min (arg 0)
            if (!scan) {
            } else if (side == 0) {
                if (tag < (uint32_t)a.nchunks) { c0 = (int)tag * kColChunk; ngroups = 8; }              // the 32 columns of the winning chunk
            } else if ((tag >> 5) < (uint32_t)a.nrowgroups) {
                c0 = (int)(tag >> 5) * (32 * R) + (int)(tag & 31u) * R;                                  // the R rows of the winning lane
                ngroups = R >> 2;
            }
            if (ngroups > 0) {
#pragma unroll 4
                for (int i = 0; i < ngroups; ++i) {
                    const int k = (lane + i) & (ngroups - 1), j = c0 + 4 * k;                             // rotated start: conflict-free banks
                    if (j < n_opp) {                                                                      // n_opp % 4 == 0: whole groups
                        float e0, e1, e2, e3;
                        eval4(j, m2x, m2y, m2z, pn, e0, e1, e2, e3);
                        if (e3 == v) arg = min(arg, j + 3);
                        if (e2 == v) arg = min(arg, j + 2);
                        if (e1 == v) arg = min(arg, j + 1);
                        if (e0 == v) arg = min(arg, j);
                    }
                }
            } else if (scan && side == 1 && R < 4 && (tag >> 5) < (uint32_t)a.nrowgroups) {
                for (int t = 0; t < R; ++t) {                                                             // R = 2
                    const int i = c0 + t;
                    if (i < n_opp) {
                        float x, y, z;
                        if (opp_cm) { x = stage[i]; y = stage[sa.stage_stride + i]; z = stage[2 * sa.stage_stride + i]; }
                        else { x = stage[3 * i]; y = stage[3 * i + 1]; z = stage[3 * i + 2]; }
                        const float e = pair_dist_scalar<FORM>(-2.f * x, -2.f * y, -2.f * z, sq_norm3(NORM, x, y, z), px, py, pz, pn);
                        if (e == v) arg = min(arg, i);
                    }
                }
            }
            bv = v;
        }
        if (p < n_own) {
            if (arg == 0x7fffffff) arg = 0;        // no finite minimum (NaN / inf inputs)
            val = apply_transform(a.transform, bv);
            out_min[p] = val; out_arg[p] = arg;
        }
        store_unit_partial(a, b, (side ? (N + 31) >> 5 : 0) + u, p < n_own, val, p, lane);
        key = nkey; px = nx; py = ny; pz = nz;
    }
    if (lane == 0) __threadfence();       // this warp's unit partials are visible before the CTA reports completion
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(&a.counters[b], 1) == per_sample - 1;
    __syncthreads();
    if (!s_last || warp >= 2) return;
    __threadfence();
    fold_sample_side(a, b, warp, lane);   // last CTA of sample b: one warp per side
}

// -------------------------------------------------------------------------------- backward
struct BwdArgs {
    const float *rows; int64_t r_sb, r_sp, r_sc;
    const float *cols; int64_t c_sb, c_sp, c_sc;
    int B, N, M, swap_norms, transform;
    const int32_t *row_arg, *col_arg;
    const float *row_min, *col_min;
    const float *g_row, *g_col;
    const float *w_row_all, *w_row_max; const int32_t *row_argmax;
    const float *w_col_all, *w_col_max; const int32_t *col_argmax;
    int64_t ws0, ws1, ws2, ws3;     // element strides of the four w arrays (0 = broadcast scalar)
    float row_scale, col_scale;
    float *grad_rows; int64_t gr_sb, gr_sp, gr_sc;
    float *grad_cols; int64_t gc_sb, gc_sp, gc_sc;
};

__device__ __forceinline__ float3 ld3(const float *base, int64_t sc) {
    return make_float3(base[0], base[sc], base[2 * sc]);
}
// upstream gradient of minimum (b,p) on one side
__device__ __forceinline__ float upstream(const float *g, const float *w_all, int64_t s_all, const float *w_max,
                                          int64_t s_max, const int32_t *argmax, int b, int p, int n, float scale) {
    float r = 0.f;
    if (g) r += g[(size_t)b * n + p];
    if (w_all) r += w_all[b * s_all] * scale;
    if (w_max && argmax[b] == p) r += w_max[b * s_max];
    return r;
}
// d(value)/d(d2) factor: squared -> 2 * g (applied to (p - q)); sqrt -> g / v, 0 at v == 0
__device__ __forceinline__ float chain_factor(int transform, float g, const float *vals, size_t off) {
    if (transform == PCD_VALUE_SQRT_CLAMP) {
        const float v = vals[off];
        return v > 0.f ? g / v : 0.f;
    }
    return 2.f * g;
}

// MODE 0 (plain stores, writes every gradient element): the terms indexed by the thread's own
// point.  MODE 1 (atomics): the terms that land on the argmin partner.  MODE 2 = both in one
// launch with atomics only, for gradients the host has zeroed (dense outputs: one memset +
// one kernel instead of two dependent kernels).
template <int MODE>
__device__ __forceinline__ void emit3(float *gp, int64_t sc, float x, float y, float z) {
    if (MODE == 0) {
        gp[0] = x; gp[sc] = y; gp[2 * sc] = z;
    } else {
        atomicAdd(gp, x); atomicAdd(gp + sc, y); atomicAdd(gp + 2 * sc, z);
    }
}

template <int MODE>
__global__ void __launch_bounds__(256) nn1_bwd_kernel(BwdArgs a) {
    constexpr bool OWN = MODE != 1, SCAT = MODE != 0;
    const long long total = (long long)a.B * (a.N + a.M);
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const int b = (int)(t / (a.N + a.M));
        const int p = (int)(t - (long long)b * (a.N + a.M));
        const float *rb = a.rows + b * a.r_sb, *cb = a.cols + b * a.c_sb;
        if (p < a.N) {
            const int i = p;
            const float g = upstream(a.g_row, a.w_row_all, a.ws0, a.w_row_max, a.ws1, a.row_argmax, b, i, a.N, a.row_scale);
            const int j = a.row_arg[(size_t)b * a.N + i];
            const float3 r = ld3(rb + i * a.r_sp, a.r_sc), c = ld3(cb + j * a.c_sp, a.c_sc);
            const float f = chain_factor(a.transform, g, a.row_min, (size_t)b * a.N + i);
            if (OWN && a.grad_rows) {
                float3 o;
                if (a.swap_norms) {
                    // entry (i,j): -f c_j ; column-direction entry (i*, j=i): +f' r_i, f' the chain factor of column i
                    const float g2 = upstream(a.g_col, a.w_col_all, a.ws2, a.w_col_max, a.ws3, a.col_argmax, b, i, a.M, a.col_scale);
                    const float f2 = chain_factor(a.transform, g2, a.col_min, (size_t)b * a.M + i);
                    o = make_float3(-f * c.x + f2 * r.x, -f * c.y + f2 * r.y, -f * c.z + f2 * r.z);
                } else {
                    o = make_float3(f * (r.x - c.x), f * (r.y - c.y), f * (r.z - c.z));
                }
                emit3<MODE>(a.grad_rows + b * a.gr_sb + i * a.gr_sp, a.gr_sc, o.x, o.y, o.z);
            }
            if (SCAT && g != 0.f) {
                if (a.grad_cols) {
                    float *gp = a.grad_cols + b * a.gc_sb + j * a.gc_sp;
                    if (a.swap_norms) emit3<1>(gp, a.gc_sc, -f * r.x, -f * r.y, -f * r.z);
                    else emit3<1>(gp, a.gc_sc, -f * (r.x - c.x), -f * (r.y - c.y), -f * (r.z - c.z));
                }
                if (a.swap_norms && a.grad_rows) {   // |rows_j|^2 term of entry (i,j)
                    const float3 rj = ld3(rb + j * a.r_sp, a.r_sc);
                    emit3<1>(a.grad_rows + b * a.gr_sb + j * a.gr_sp, a.gr_sc, f * rj.x, f * rj.y, f * rj.z);
                }
            }
        } else {
            const int j = p - a.N;
            const float g = upstream(a.g_col, a.w_col_all, a.ws2, a.w_col_max, a.ws3, a.col_argmax, b, j, a.M, a.col_scale);
            const int i = a.col_arg[(size_t)b * a.M + j];
            const float3 r = ld3(rb + i * a.r_sp, a.r_sc), c = ld3(cb + j * a.c_sp, a.c_sc);
            const float f = chain_factor(a.transform, g, a.col_min, (size_t)b * a.M + j);
            if (OWN && a.grad_cols) {
                float3 o;
                if (a.swap_norms) {
                    // entry (i*,j): -f' r_i* ; row-direction entry (i=j, j*): +f c_j, f the chain factor of row j
                    const float g1 = upstream(a.g_row, a.w_row_all, a.ws0, a.w_row_max, a.ws1, a.row_argmax, b, j, a.N, a.row_scale);
                    const float f1 = chain_factor(a.transform, g1, a.row_min, (size_t)b * a.N + j);
                    o = make_float3(-f * r.x + f1 * c.x, -f * r.y + f1 * c.y, -f * r.z + f1 * c.z);
                } else {
                    o = make_float3(f * (c.x - r.x), f * (c.y - r.y), f * (c.z - r.z));
                }
                emit3<MODE>(a.grad_cols + b * a.gc_sb + j * a.gc_sp, a.gc_sc, o.x, o.y, o.z);
            }
            if (SCAT && g != 0.f) {
                if (a.grad_rows) {
                    float *gp = a.grad_rows + b * a.gr_sb + i * a.gr_sp;
                    if (a.swap_norms) emit3<1>(gp, a.gr_sc, -f * c.x, -f * c.y, -f * c.z);
                    else emit3<1>(gp, a.gr_sc, -f * (c.x - r.x), -f * (c.y - r.y), -f * (c.z - r.z));
                }
                if (a.swap_norms && a.grad_cols) {   // |cols_i*|^2 term of entry (i*,j)
                    const float3 ci = ld3(cb + i * a.c_sp, a.c_sc);
                    emit3<1>(a.grad_cols + b * a.gc_sb + i * a.gc_sp, a.gc_sc, f * ci.x, f * ci.y, f * ci.z);
                }
            }
        }
    }
}

// ----------------------------------------------------------------------------- host helpers
template <bool RAW>
static cudaError_t launch_sweep(int form, int R, const SweepSrc &src, unsigned long long *rowkey, unsigned long long *colkey,
                                int B, int N, int M, int Npad, int Mpad, int mt, int sms, cudaStream_t st) {
    const auto launch = [&](auto FORM, auto RR) -> cudaError_t {
        const auto kernel = nn1_sweep_kernel<FORM, RR, RAW>;
        const size_t smem = sizeof(typename std::conditional<RAW, SweepSmem<RR>, SweepSmemPacked<RR>>::type);
        const int QT = kSweepWarps * 32 * RR;
        const int nqt = (N + QT - 1) / QT;                       // fully inert row tiles are skipped
        const int nq = (M + kQuad - 1) / kQuad;                  // ... and fully inert column quads
        const long long units = (long long)B * nqt * nq;
        if (units >= (1LL << 31)) return cudaErrorInvalidValue;
        // ask for the shared-memory carve-out explicitly: the register-limited residency (2 CTAs at R = 16) needs
        // 2 x 55 KB, more than the default split provides
        cudaError_t e = opt_in_smem(kernel, smem, true);
        int occ = 0;
        if (e == cudaSuccess) e = ctas_per_sm(kernel, kSweepThreads, smem, &occ);
        if (e != cudaSuccess) return e;
        long long grid = (long long)sms * occ;
        if (grid > units) grid = units;
        return launch_kernel(kernel, dim3((unsigned)grid), dim3(kSweepThreads), smem, st, true,
                             src, rowkey, colkey, N, Npad, Mpad, mt / kQuad, nqt, nq, (int)units);
    };
    return with_form(form, [&](auto FORM) {
        switch (R) {
        case 16: return launch(FORM, IntC<16>{});
        case 8: return launch(FORM, IntC<8>{});
        case 4: return launch(FORM, IntC<4>{});
        default: return launch(FORM, IntC<2>{});
        }
    });
}

template <int ITEMS>
static cudaError_t launch_bucket(const BucketArgs &a, int B, cudaStream_t st) {
    const auto kernel = nn1_bucket_kernel<ITEMS>;
    const size_t smem = bucket_smem_bytes<ITEMS>();
    cudaError_t e = opt_in_smem(kernel, smem);
    if (e != cudaSuccess) return e;
    return launch_kernel(kernel, dim3((unsigned)(2 * B)), dim3(kBucketThreads), smem, st, false, a);
}

static cudaError_t launch_pruned_sweep(int form, const PruneArgs &a, int sms, cudaStream_t st) {
    return with_form(form, [&](auto FORM) {
        const auto kernel = nn1_pruned_sweep_kernel<FORM>;
        int occ = 0;
        const cudaError_t e = ctas_per_sm(kernel, kPruneThreads, 0, &occ);
        if (e != cudaSuccess) return e;
        const long long items = (long long)a.B * (((a.N + 31) >> 5) + ((a.M + 31) >> 5));
        long long grid = (long long)sms * occ, wpc = kPruneThreads / 32;
        if (grid * wpc > items) grid = (items + wpc - 1) / wpc;
        return launch_kernel(kernel, dim3((unsigned)grid), dim3(kPruneThreads), 0, st, true, a);
    });
}

static cudaError_t launch_fixup(int form, bool raw, const FixupArgs &a, dim3 grid, cudaStream_t st) {
    const auto kernel = with_form(form, [&](auto FORM) {
        // the norm rounding is a template parameter of the streamed variant only (the packed records carry their norms)
        if (!raw) return nn1_fixup_kernel<FORM, false, PCD_NORM_MULSUM>;
        return with_norm(a.norm_kind, [&](auto NORM) { return nn1_fixup_kernel<FORM, true, NORM>; });
    });
    return launch_kernel(kernel, grid, dim3(kFixupThreads), 0, st, true, a);
}

// Shared-memory staged fix-up (dense clouds of up to kStageMaxBytes): see nn1_fixup_staged_kernel.
constexpr size_t kStageMaxBytes = 200 * 1024;

// One CTA per (sample, side, slice); `parts` slices per job are chosen so that the whole grid is resident at once
// (a second wave of CTAs would wait for the first one to drain: +40 % at BASELINE config 2).
static cudaError_t launch_fixup_staged(int form, int norm_kind, StagedArgs sa, int B, int sms, size_t smem, cudaStream_t st) {
    const auto kernel = with_form(form, [&](auto FORM) {
        return with_norm(norm_kind, [&](auto NORM) { return nn1_fixup_staged_kernel<FORM, NORM>; });
    });
    cudaError_t e = opt_in_smem(kernel, kStageMaxBytes, true);
    // residency for this staging size: 1 .. 3 CTAs per SM (register bound 3)
    int per_sm = 0;
    if (e == cudaSuccess) e = ctas_per_sm(kernel, kFixupThreads, smem, &per_sm);
    if (e != cudaSuccess) return e;
    // slices per sample, split between the sides in proportion to their scan work (32 candidates per row point, R per column point)
    const int urow = (sa.f.N + 31) / 32, ucol = (sa.f.M + 31) / 32;
    int total = sms * per_sm / B;
    if (total < 2) total = 2;
    const double wr = 32.0 * sa.f.N, wc = (double)sa.f.R * sa.f.M;
    int pr = (int)(total * wr / (wr + wc) + 0.5);
    if (pr < 1) pr = 1;
    if (pr > total - 1) pr = total - 1;
    int pc = total - pr;
    // a slice should give every warp of its CTA at least one unit (each CTA stages the whole candidate cloud)
    const int wpc = kFixupThreads / 32;
    if (pr > (urow + wpc - 1) / wpc) pr = (urow + wpc - 1) / wpc;
    if (pc > (ucol + wpc - 1) / wpc) pc = (ucol + wpc - 1) / wpc;
    sa.parts_row = pr; sa.parts_col = pc;
    return launch_kernel(kernel, dim3((unsigned)(B * (pr + pc))), dim3(kFixupThreads), smem, st, true, sa);
}

// Tile-shape heuristic.  R rows per lane (register blocking: the per-step overhead -- operand
// LDS, CREDUX, ballots, stores -- is amortised over 2R pairs) against padding waste and the
// number of chunks each CTA of the persistent grid gets.
static void choose_tiling(int B, int N, int M, int sms, int force_R, int force_mt, int *R_out, int *mt_out) {
    static const int occ_of[5] = {6, 5, 4, 2, 0};       // CTAs/SM for R = 2, 4, 8, 16
    const long long nch = (M + kColChunk - 1) / kColChunk;
    int R = 16, oi = 3;
    while (R > 2) {
        const long long qtiles = (long long)B * ((N + 128 * R - 1) / (128 * R));
        const long long padded = qtiles * 128 * R;
        const bool waste = padded * 8 > (long long)B * N * 9;                 // > 12.5 % inert rows
        const bool starved = qtiles * nch < 6LL * sms * occ_of[oi];            // < 6 chunks per CTA
        if (!waste && !starved) break;
        R >>= 1; --oi;
    }
    int mt = kMaxColTile;
    // explicit per-call overrides (tests and tuning sweeps); the library reads no environment
    if (force_R == 2 || force_R == 4 || force_R == 8 || force_R == 16) R = force_R;
    if (force_mt >= 32 && force_mt <= 256 && (force_mt & (force_mt - 1)) == 0) mt = force_mt;
    *R_out = R; *mt_out = mt;
}

// A cloud the sweep can stream as it lies in the caller's tensor: point-major [.,N,3] (sp = 3, sc = 1)
// or channel-major [.,3,N] (sp = 1), 16-byte aligned rows / tiles.
static bool dense_layout(const float *p, int64_t sb, int64_t sp, int64_t sc, int n, int *cm) {
    if ((reinterpret_cast<uintptr_t>(p) & 15) != 0 || (n & 3) != 0 || (sb & 3) != 0 || sb < 0) return false;
    if (sp == 3 && sc == 1) { *cm = 0; return true; }
    if (sp == 1 && sc >= n && (sc & 3) == 0) { *cm = 1; return true; }
    return false;
}

}  // namespace pcd

// =================================================================================== C ABI
using namespace pcd;

#ifdef PCD_SWEEP_TRACE
extern "C" int pcd_debug_set_sweep_trace(void *buf) {
    unsigned long long *p = (unsigned long long *)buf;
    PCD_CUDA_CHECK(cudaMemcpyToSymbol(g_sweep_trace, &p, sizeof(p)));
    return PCD_OK;
}
// buf: 4 zeroed uint64 counters the pruned sweep adds to (items, evaluated chunks, arg-min re-scans, tie passes); NULL stops
extern "C" int pcd_debug_set_prune_counters(void *buf) {
    unsigned long long *p = (unsigned long long *)buf;
    PCD_CUDA_CHECK(cudaMemcpyToSymbol(g_prune_count, &p, sizeof(p)));
    return PCD_OK;
}
#endif

extern "C" size_t pcd_nn1_workspace_bytes(int B, int N, int M, int sweep_mode) {
    (void)sweep_mode;      // kept for ABI compatibility: every mode needs the same workspace
    if (B <= 0 || N <= 0 || M <= 0) return 0;
    return nn1_layout(B, N, M).total;
}

extern "C" int pcd_nn1_query_tiling(int B, int N, int M, int *rows_per_lane, int *col_tile) {
    if (B <= 0 || N <= 0 || M <= 0 || !rows_per_lane || !col_tile) {
        set_error("pcd_nn1_query_tiling: bad argument");
        return PCD_ERR_ARG;
    }
    const int sms = num_sms();
    if (sms <= 0) return cuda_fail(cudaGetLastError(), "no CUDA device");
    choose_tiling(B, N, M, sms, 0, 0, rows_per_lane, col_tile);
    return PCD_OK;
}

extern "C" int pcd_nn1_forward(const float *rows, int64_t r_sb, int64_t r_sp, int64_t r_sc,
                               const float *cols, int64_t c_sb, int64_t c_sp, int64_t c_sc,
                               int B, int N, int M, int form, int norm_kind, int swap_norms, int transform,
                               float row_sum_scale, float col_sum_scale,
                               float *row_min, int32_t *row_arg, float *col_min, int32_t *col_arg,
                               float *stats_f, int32_t *stats_i,
                               float *zero0, size_t zero0_floats, float *zero1, size_t zero1_floats,
                               void *workspace, size_t workspace_bytes, int rows_per_lane, int col_tile, int sweep_mode,
                               void *sweep_start_event, void *sweep_stop_event, void *stream) {
    if (!rows || !cols || !row_min || !row_arg || !col_min || !col_arg || !stats_f || !stats_i || !workspace) {
        set_error("pcd_nn1_forward: NULL pointer argument");
        return PCD_ERR_ARG;
    }
    if (B <= 0 || N <= 0 || M <= 0 || form < 0 || form > 2 || norm_kind < 0 || norm_kind > 1 || transform < 0 ||
        transform > 1 || B > 65535 || sweep_mode < 0 || sweep_mode > 2) {
        set_error("pcd_nn1_forward: bad argument B=%d N=%d M=%d form=%d norm=%d transform=%d sweep_mode=%d", B, N, M, form,
                  norm_kind, transform, sweep_mode);
        return PCD_ERR_ARG;
    }
    if (swap_norms && N != M) {
        set_error("pcd_nn1_forward: swap_norms requires N == M (got %d, %d), as the reference's broadcast does", N, M);
        return PCD_ERR_ARG;
    }
    if ((zero0_floats && (!zero0 || (zero0_floats & 3) || (reinterpret_cast<uintptr_t>(zero0) & 15))) ||
        (zero1_floats && (!zero1 || (zero1_floats & 3) || (reinterpret_cast<uintptr_t>(zero1) & 15)))) {
        set_error("pcd_nn1_forward: zero-fill buffers must be 16-byte aligned with a multiple of 4 floats");
        return PCD_ERR_ARG;
    }
    const int sms = num_sms();
    if (sms <= 0) return cuda_fail(cudaGetLastError(), "no CUDA device");
    const Nn1Layout L = nn1_layout(B, N, M);
    if (workspace_bytes < L.total) {
        set_error("pcd_nn1_forward: workspace %zu < required %zu bytes", workspace_bytes, L.total);
        return PCD_ERR_WORKSPACE;
    }
    if ((reinterpret_cast<uintptr_t>(workspace) & 255) != 0) {
        set_error("pcd_nn1_forward: workspace must be 256-byte aligned");
        return PCD_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    char *ws = (char *)workspace;
    float4 *rowpk = (float4 *)(ws + L.rowpk);
    float4 *rowpp = (float4 *)(ws + L.rowpp);
    float *colpk = (float *)(ws + L.colpk);
    unsigned long long *rowkey = (unsigned long long *)(ws + L.rowkey);
    unsigned long long *colkey = (unsigned long long *)(ws + L.colkey);
    int *counters = (int *)(ws + L.counters);

    int R, mt;
    choose_tiling(B, N, M, sms, rows_per_lane, col_tile, &R, &mt);

    int row_cm = 0, col_cm = 0;
    const bool raw = !swap_norms && dense_layout(rows, r_sb, r_sp, r_sc, N, &row_cm) &&
                     dense_layout(cols, c_sb, c_sp, c_sc, M, &col_cm);
    SweepSrc src{rows, (long long)r_sb, (long long)r_sc, cols, (long long)c_sb, (long long)c_sc, row_cm, col_cm, norm_kind,
                 rowpp, (const float4 *)colpk};

    const int nmax = N > M ? N : M;
    const size_t stage_stride = align_up((size_t)nmax, 32);
    const size_t stage_bytes = stage_stride * 12;
    const bool staged = raw && stage_bytes <= kStageMaxBytes;
    // the pruned chain: dense clouds the bucketing sorts in shared memory, large enough that its bucketing pass pays off
    // (DESIGN.md section 4.0); an explicit tiling keeps the full sweep
    const bool pruned = raw && nmax <= kPruneMaxPoints && (N < M ? N : M) >= kPruneMinPoints && B >= kPruneMinBatch &&
                        rows_per_lane == 0 && col_tile == 0;
    int *bperm = (int *)(ws + L.bperm);
    if (pruned) {
        const BucketArgs ba{rows, (long long)r_sb, (long long)r_sp, (long long)r_sc, cols, (long long)c_sb, (long long)c_sp,
                            (long long)c_sc, N, M, norm_kind, L.bslots, (float4 *)(ws + L.brec), (float4 *)(ws + L.bbox), bperm,
                            counters, (int *)(ws + L.queue)};
        PCD_CUDA_CHECK(nmax <= 4 * kBucketThreads ? launch_bucket<4>(ba, B, st) : launch_bucket<16>(ba, B, st));
    } else if (raw) {
        PCD_CUDA_CHECK(launch_kernel(nn1_arm_kernel, dim3((unsigned)(sms * 2)), dim3(256), 0, st, false,
                                     (ulonglong2 *)rowkey, L.nkeys / 2, counters, B));
    } else {
        const int grid = capped_grid((long long)B * (L.Npad + L.Mpad), 256, (long long)sms * 8);
        PCD_CUDA_CHECK(launch_kernel(nn1_prep_kernel, dim3(grid), dim3(256), 0, st, false, rows, r_sb, r_sp, r_sc, cols, c_sb,
                                     c_sp, c_sc, B, N, M, L.Npad, L.Mpad, R, norm_kind, swap_norms, rowpk, rowpp, colpk, rowkey,
                                     colkey, counters));
    }
    // an event between two kernels turns the programmatic edge into a full dependency: timing the sweep
    // alone (bench.py's roofline) costs the overlap, nothing else
    if (sweep_start_event) PCD_CUDA_CHECK(cudaEventRecord((cudaEvent_t)sweep_start_event, st));
    if (pruned) {
        const PruneArgs pa{(const float4 *)(ws + L.brec), (const float4 *)(ws + L.bbox), bperm, (int *)(ws + L.queue),
                           rowkey, colkey, B, N, M, L.Npad, L.Mpad, L.bslots};
        PCD_CUDA_CHECK(launch_pruned_sweep(form, pa, sms, st));
    } else {
        PCD_CUDA_CHECK(raw ? launch_sweep<true>(form, R, src, rowkey, colkey, B, N, M, L.Npad, L.Mpad, mt, sms, st)
                           : launch_sweep<false>(form, R, src, rowkey, colkey, B, N, M, L.Npad, L.Mpad, mt, sms, st));
    }
    if (sweep_stop_event) PCD_CUDA_CHECK(cudaEventRecord((cudaEvent_t)sweep_stop_event, st));
    {
        // persistent grid: every warp of every resident CTA owns a contiguous range of units (32 points of one side)
        const long long octets = (long long)B * ((N + 31) / 32 + (M + 31) / 32);
        if (octets >= (1LL << 31)) {
            set_error("pcd_nn1_forward: B * (N + M) too large");
            return PCD_ERR_ARG;
        }
        long long nwarps = (long long)sms * kFixupCtasPerSm * (kFixupThreads / 32);
        if (nwarps > kFixupMaxWarps) nwarps = kFixupMaxWarps;
        if (nwarps > octets) nwarps = octets;
        FixupArgs a{rows, (long long)r_sb, (long long)r_sp, (long long)r_sc, cols, (long long)c_sb, (long long)c_sp, (long long)c_sc,
                    rowpk, (const float4 *)colpk, col_cm ? 2 : 1, norm_kind, rowkey, colkey, counters,
                    (float4 *)(ws + L.partials), L.partial_slots, (int)nwarps, (int)(octets / nwarps), (int)(octets % nwarps),
                    (N + 32 * R - 1) / (32 * R), (M + kColChunk - 1) / kColChunk, N, M, L.Npad, L.Mpad, R, transform, B, row_min, row_arg, col_min, col_arg,
                    row_sum_scale, col_sum_scale, stats_f, stats_i,
                    (float4 *)zero0, zero0_floats / 4, (float4 *)zero1, zero1_floats / 4, pruned ? 1 : 0};
        if (staged && !pruned) {
            // one CTA per (sample, side, slice): the re-scanned cloud is staged in shared memory
            const StagedArgs sa{a, 1, 1, (int)stage_stride};
            PCD_CUDA_CHECK(launch_fixup_staged(form, norm_kind, sa, B, sms, stage_bytes, st));
        } else {
            const dim3 grid((unsigned)((nwarps + kFixupThreads / 32 - 1) / (kFixupThreads / 32)));
            PCD_CUDA_CHECK(launch_fixup(form, raw, a, grid, st));
        }
    }
    return PCD_OK;
}

extern "C" int pcd_nn1_backward(const float *rows, int64_t r_sb, int64_t r_sp, int64_t r_sc,
                                const float *cols, int64_t c_sb, int64_t c_sp, int64_t c_sc,
                                int B, int N, int M, int swap_norms, int transform,
                                const int32_t *row_arg, const int32_t *col_arg,
                                const float *row_min, const float *col_min,
                                const float *g_row, const float *g_col,
                                const float *w_row_all, const float *w_row_max, const int32_t *row_argmax,
                                const float *w_col_all, const float *w_col_max, const int32_t *col_argmax,
                                const int64_t *w_strides, float row_sum_scale, float col_sum_scale,
                                float *grad_rows, int64_t gr_sb, int64_t gr_sp, int64_t gr_sc,
                                float *grad_cols, int64_t gc_sb, int64_t gc_sp, int64_t gc_sc,
                                int grads_prezeroed, void *stream) {
    if (!rows || !cols || !row_arg || !col_arg || B <= 0 || N <= 0 || M <= 0) {
        set_error("pcd_nn1_backward: bad argument");
        return PCD_ERR_ARG;
    }
    if ((w_row_max && !row_argmax) || (w_col_max && !col_argmax)) {
        set_error("pcd_nn1_backward: w_*_max given without *_argmax");
        return PCD_ERR_ARG;
    }
    if (transform == PCD_VALUE_SQRT_CLAMP && (!row_min || !col_min)) {
        set_error("pcd_nn1_backward: SQRT_CLAMP needs the stored minima");
        return PCD_ERR_ARG;
    }
    if (swap_norms && N != M) {
        set_error("pcd_nn1_backward: swap_norms requires N == M");
        return PCD_ERR_ARG;
    }
    if (!grad_rows && !grad_cols) return PCD_OK;
    const int sms = num_sms();
    if (sms <= 0) return cuda_fail(cudaGetLastError(), "no CUDA device");
    BwdArgs a{rows, r_sb, r_sp, r_sc, cols, c_sb, c_sp, c_sc, B, N, M, swap_norms, transform,
              row_arg, col_arg, row_min, col_min, g_row, g_col,
              w_row_all, w_row_max, row_argmax, w_col_all, w_col_max, col_argmax,
              w_strides ? w_strides[0] : 1, w_strides ? w_strides[1] : 1, w_strides ? w_strides[2] : 1,
              w_strides ? w_strides[3] : 1, row_sum_scale, col_sum_scale,
              grad_rows, gr_sb, gr_sp, gr_sc, grad_cols, gc_sb, gc_sp, gc_sc};
    const int grid = capped_grid((long long)B * (N + M), 256, (long long)sms * 16);
    cudaStream_t st = (cudaStream_t)stream;
    const bool dense_r = !grad_rows || (gr_sc == 1 && gr_sp == 3 && gr_sb == (int64_t)N * 3);
    const bool dense_c = !grad_cols || (gc_sc == 1 && gc_sp == 3 && gc_sb == (int64_t)M * 3);
    if (grads_prezeroed) {
        // the caller handed these buffers to pcd_nn1_forward's zero fill (or cleared them itself): one launch
        nn1_bwd_kernel<2><<<grid, 256, 0, st>>>(a);
        PCD_CUDA_CHECK(cudaGetLastError());
    } else if (dense_r && dense_c) {
        if (grad_rows) PCD_CUDA_CHECK(cudaMemsetAsync(grad_rows, 0, (size_t)B * N * 3 * sizeof(float), st));
        if (grad_cols) PCD_CUDA_CHECK(cudaMemsetAsync(grad_cols, 0, (size_t)B * M * 3 * sizeof(float), st));
        nn1_bwd_kernel<2><<<grid, 256, 0, st>>>(a);
        PCD_CUDA_CHECK(cudaGetLastError());
    } else {
        nn1_bwd_kernel<0><<<grid, 256, 0, st>>>(a);
        PCD_CUDA_CHECK(cudaGetLastError());
        nn1_bwd_kernel<1><<<grid, 256, 0, st>>>(a);
        PCD_CUDA_CHECK(cudaGetLastError());
    }
    return PCD_OK;
}
