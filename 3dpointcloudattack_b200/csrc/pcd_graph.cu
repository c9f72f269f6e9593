// pcd_graph.cu -- the callers either side of the k-NN path (SURVEY.md section 8f rows 2 and 3):
//
//   * edge features of a k-NN graph: DGCNN get_graph_feature (model/dgcnn.py:203-227) and
//     CurveNet LPFA.group_feature (model/curvenet_util.py:206-236) -- a gather through idx fused
//     with the centre subtraction / concatenation / permute(0,3,1,2), and its scatter-add backward;
//   * farthest point sampling (model/pointnet2_utils.py:59-81, model/curvenet_util.py:69-90):
//     the reference's Python loop of `npoint` iterations x 6 kernel launches as ONE persistent
//     CTA per sample with the points and their running distances in registers.
//
// Both are HBM / latency bound byte movers: no tensor cores, no tiles of math.
#include "pcd_common.cuh"

namespace pcd {

// ------------------------------------------------------------------------- edge features
// out[b, q*C + c, n, j] = op_q( x[b,c,n] (centre), x[b,c,idx[b,n,j]] (neighbour) ),  q < nblocks
//   CENTER   -> centre            NEIGHBOR -> neighbour            DIFF -> neighbour - centre
// ops are packed two bits per block.  The output -- the only large stream: B * nblocks*C * N*k
// floats, 5.4 GB for DGCNN's last layer at BASELINE config 4 -- is written once with streaming
// float4 stores.  A CTA stages the x rows of its CG channels in shared memory (N floats each):
// the neighbour gathers are random 4-byte reads, and from L1 they cost one tag lookup per
// lane (ncu: lg_throttle, 4.0 TB/s of stores); from shared memory they are bank accesses.
constexpr int kEdgeThreads = 256;
constexpr int kEdgeSmemFloats = 16384;       // 64 KB of staged channel rows per CTA

__device__ __forceinline__ float edge_value(int op, float ctr, float nb) {
    return op == PCD_EDGE_CENTER ? ctr : (op == PCD_EDGE_NEIGHBOR ? nb : __fadd_rn(nb, -ctr));
}

// grid (slices, channel groups, B); a slice = spt consecutive VEC-wide slots per thread-stride
template <int VEC>
__global__ void __launch_bounds__(kEdgeThreads)
edge_feature_fwd_kernel(const float *__restrict__ x, const int32_t *__restrict__ idx, int C, int N, int k, int nblocks,
                        int ops, int CG, long long slots_per_slice, float *__restrict__ out) {
    extern __shared__ float xs[];                                  // [CG][N]
    const long long NK = (long long)N * k;
    const int b = blockIdx.z;
    const int c0 = blockIdx.y * CG;
    const int ncg = (c0 + CG < C ? c0 + CG : C) - c0;
    const float *xb = x + ((size_t)b * C + c0) * N;
    for (int i = threadIdx.x; i < ncg * N; i += kEdgeThreads) xs[i] = __ldg(xb + i);
    __syncthreads();
    const long long nslots = (NK + VEC - 1) / VEC;
    const long long s_begin = (long long)blockIdx.x * slots_per_slice;
    const long long s_end = s_begin + slots_per_slice < nslots ? s_begin + slots_per_slice : nslots;
    const int32_t *ib = idx + (size_t)b * NK;
    for (long long sl = s_begin + threadIdx.x; sl < s_end; sl += kEdgeThreads) {
        const long long e0 = sl * VEC;
        int m[VEC];
        if (VEC == 4) {
            const int4 v = __ldcs(reinterpret_cast<const int4 *>(ib + e0));
            m[0] = v.x; m[1 % VEC] = v.y; m[2 % VEC] = v.z; m[3 % VEC] = v.w;
        } else {
            m[0] = __ldcs(ib + e0);
        }
        const int n = (int)(e0 / k);                               // VEC = 4 only when 4 | k: the four slots share n
#pragma unroll
        for (int i = 0; i < VEC; ++i) m[i] = min(max(m[i], 0), N - 1);      // never read outside the staged rows (the kernel is store bound)
        for (int c = 0; c < ncg; ++c) {
            const float *xr = xs + c * N;
            const float ctr = xr[n];
            float nb[VEC];
#pragma unroll
            for (int i = 0; i < VEC; ++i) nb[i] = xr[m[i]];
            for (int q = 0; q < nblocks; ++q) {
                const int op = (ops >> (2 * q)) & 3;
                float *dst = out + (((size_t)b * nblocks + q) * C + c0 + c) * NK + e0;
                if (VEC == 4) {
                    __stcs(reinterpret_cast<float4 *>(dst),
                           make_float4(edge_value(op, ctr, nb[0]), edge_value(op, ctr, nb[1 % VEC]),
                                       edge_value(op, ctr, nb[2 % VEC]), edge_value(op, ctr, nb[3 % VEC])));
                } else {
                    __stcs(dst, edge_value(op, ctr, nb[0]));
                }
            }
        }
    }
}

// Backward: gx[b,c,n] = sum_j s_ctr(n,j) + sum_{(n',j): idx[b,n',j] = n} s_nbr(n',j) with
//   s_nbr = sum of g over NEIGHBOR and DIFF blocks,  s_ctr = sum over CENTER blocks - sum over DIFF blocks.
// One CTA per (sample, channel): the N accumulators live in shared memory.  Threads walk the
// (n, j) slots in lane-linear order, so the upstream gradient -- again the only large stream,
// read once -- and the indices arrive as fully coalesced 16-byte loads; own terms and
// neighbour terms both go through shared-memory atomics.  Summation order of the scatter is
// not fixed (as in the reference's index backward): results differ run to run in the last bits.
template <int VEC>
__global__ void __launch_bounds__(kEdgeThreads, 8)       // 8 CTAs = 64 warps per SM: the CAS loops are latency bound
edge_feature_bwd_kernel(const float *__restrict__ g, const int32_t *__restrict__ idx, int C, int N, int k, int nblocks,
                        int ops, float *__restrict__ gx) {
    extern __shared__ float acc[];
    const int c = blockIdx.x, b = blockIdx.y;
    const long long NK = (long long)N * k;
    for (int i = threadIdx.x; i < N; i += kEdgeThreads) acc[i] = 0.f;
    __syncthreads();
    const int32_t *ib = idx + (size_t)b * NK;
    const long long nslots = NK / VEC;
    // warp-uniform trip count: every lane of a warp runs the same number of iterations (lanes past the end carry a
    // neutral slot), so the segmented scan below always runs converged, with the full mask
    const long long nslots_up = (nslots + 31) / 32 * 32;
    for (long long sl = threadIdx.x; sl < nslots_up; sl += kEdgeThreads) {
        const bool valid = sl < nslots;
        const long long e0 = (valid ? sl : 0) * VEC;
        int m[VEC];
        if (VEC == 4) {
            const int4 v = *reinterpret_cast<const int4 *>(ib + e0);
            m[0] = v.x; m[1 % VEC] = v.y; m[2 % VEC] = v.z; m[3 % VEC] = v.w;
        } else {
            m[0] = ib[e0];
        }
        float sn[VEC], own = 0.f;
#pragma unroll
        for (int i = 0; i < VEC; ++i) { sn[i] = 0.f; m[i] = min(max(m[i], 0), N - 1); }
        if (valid) {
            for (int q = 0; q < nblocks; ++q) {
                const int op = (ops >> (2 * q)) & 3;
                const float *gp = g + (((size_t)b * nblocks + q) * C + c) * NK + e0;
                float ga[VEC];
                if (VEC == 4) {
                    const float4 gv = __ldcs(reinterpret_cast<const float4 *>(gp));
                    ga[0] = gv.x; ga[1 % VEC] = gv.y; ga[2 % VEC] = gv.z; ga[3 % VEC] = gv.w;
                } else {
                    ga[0] = __ldcs(gp);
                }
#pragma unroll
                for (int i = 0; i < VEC; ++i) {
                    if (op != PCD_EDGE_CENTER) sn[i] += ga[i];
                    if (op == PCD_EDGE_CENTER) own += ga[i];
                    if (op == PCD_EDGE_DIFF) own -= ga[i];
                }
            }
#pragma unroll
            for (int i = 0; i < VEC; ++i) atomicAdd(&acc[m[i]], sn[i]);
        }
        // own term: consecutive lanes share the centre n (k / VEC slots each).  Shared-memory float
        // atomics are compare-and-swap loops, and same-address lanes serialise them, so the lanes of
        // a run first add up with a segmented shuffle scan and only the run's last lane touches acc[n].
        // (Batching the loads of several slots per thread ahead of the atomics was measured slower:
        // the CAS loops are latency bound and want occupancy -- 64 warps/SM -- more than load ILP.)
        const int n = valid ? (int)(e0 / k) : -1;              // -1: a run of its own that adds nothing
        const int lane = threadIdx.x & 31;
        __syncwarp();                                          // reconverge after the CAS loops
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const float up = __shfl_up_sync(0xffffffffu, own, o);
            const int nup = __shfl_up_sync(0xffffffffu, n, o);
            if (lane >= o && nup == n) own += up;
        }
        const int ndown = __shfl_down_sync(0xffffffffu, n, 1);
        const bool last = lane == 31 || ndown != n;
        if (last && valid) atomicAdd(&acc[n], own);
    }
    __syncthreads();
    float *dst = gx + ((size_t)b * C + c) * N;
    for (int i = threadIdx.x; i < N; i += kEdgeThreads) dst[i] = acc[i];
}

// ------------------------------------------------ edge-feature backward, gather form (round 2)
// The REPRODUCIBLE backward: the scatter of the atomics kernel above turned into a gather.  Per sample the k-NN graph is
// inverted once (edge_csr_build_kernel; every one of the C channel planes of the sample reuses it), then a CTA per
// (sample, channel) streams its planes of g through shared memory with 1-D TMA bulk copies and every thread sums, for
// the targets it owns, the staged values of the incoming edges -- no floating-point atomics, a fixed summation order,
// the same bits on every run (the atomics kernel and the reference's index backward are not reproducible).
//
// Chunks: the source rows are cut into chunks of S rows; a stage = the chunk's rows of every block of g plus the
// chunk's part of the inverted graph (two stages per CTA, two CTAs per SM).  The inverted graph is CHUNK-major: for
// chunk ch and target j, list[ch][sub[ch][j] .. sub[ch][j+1]) holds the slots (row_in_chunk * k + slot, ascending) of
// the chunk's edges that point at j -- 16-bit entries, a quarter of the g stream, read from L2 (all channel CTAs of a
// sample read the same lists).  Thread t owns the targets t, t + 512, ...; their sums stay in registers over the chunks;
// the own-row terms (centre / difference blocks) are row sums of the staged chunk taken by the thread that owns the row.
//
// Measured (tools/edge_bwd_bench.py, B=128, C=64, N=2048, k=20): 1.44 ms = 1.8 TB/s against 0.80 ms = 3.4 TB/s for the
// atomics kernel, + 52 us for the inversion.  It was built to beat the atomics (VERDICT r1 #7) and does not: a target
// meets S*k/N = 2.5 incoming edges per chunk on average and the lanes of a warp disagree about the count (max ~7), so
// the LDS -> LDS -> FADD trips run at a third of the lanes; smaller chunks (S=128, three CTAs per SM: 1.98 ms) and
// eight predicated loads per trip (2.01 ms) were slower -- the cost is per (target, chunk) visit and per issued LDS,
// not latency.  It therefore is the opt-in form (functional.deterministic_edge_backward), not the default.
constexpr int kEgThreads = 512;
constexpr int kEgBuildThreads = 1024;
constexpr int kEgMaxTpt = 8;                       // targets per thread: N <= 4096
constexpr size_t kEgStageBudget = 110 * 1024;      // two stages (g blocks + the chunk's lists) per CTA, two CTAs per SM

struct EgPlan {
    int S, nch, np1, tpt;
    size_t sub_bytes, ws_bytes, stage_bytes, smem_main, smem_build;
};

static bool eg_plan(int B, int N, int k, int nblocks, EgPlan *p) {
    if (N > kEgThreads * kEgMaxTpt || k > 255 || ((long long)N * k) % 4 != 0 || nblocks < 1 || nblocks > 4) return false;
    const int np1 = (N + 8) & ~7;                  // row stride of sub[] in 16-bit entries (>= N + 1, 16-byte rows)
    auto stage_bytes = [&](int S) { return (size_t)nblocks * S * k * 4 + (size_t)S * k * 2 + (size_t)np1 * 2; };
    int S = 256;
    while (S > 32 && 2 * stage_bytes(S) > kEgStageBudget) S >>= 1;
    if (2 * stage_bytes(S) > kEgStageBudget || (long long)S * k > 65535) return false;
    p->S = S;
    p->nch = (N + S - 1) / S;
    p->np1 = np1;
    p->stage_bytes = stage_bytes(S);
    p->tpt = (N + kEgThreads - 1) / kEgThreads;
    p->sub_bytes = (size_t)B * p->nch * p->np1 * 2;
    p->ws_bytes = p->sub_bytes + (size_t)B * p->nch * S * k * 2;
    p->smem_main = 128 + 2 * p->stage_bytes;
    p->smem_build = (size_t)(2 * N + 2) * 4 + (size_t)S * k * 2;
    return true;
}

// in-place ascending sort of a short list in shared memory (one thread): insertion sort, heap sort for long lists
// (a target that a whole chunk points at) so that the worst case stays O(L log L)
__device__ void sort_u16(uint16_t *a, int n) {
    if (n <= 24) {
        for (int i = 1; i < n; ++i) {
            const uint16_t v = a[i];
            int j = i - 1;
            while (j >= 0 && a[j] > v) { a[j + 1] = a[j]; --j; }
            a[j + 1] = v;
        }
        return;
    }
    auto sift = [&](int root, int end) {
        const uint16_t v = a[root];
        for (;;) {
            int ch = 2 * root + 1;
            if (ch >= end) break;
            if (ch + 1 < end && a[ch + 1] > a[ch]) ++ch;
            if (a[ch] <= v) break;
            a[root] = a[ch];
            root = ch;
        }
        a[root] = v;
    };
    for (int i = n / 2 - 1; i >= 0; --i) sift(i, n);
    for (int e = n - 1; e > 0; --e) {
        const uint16_t t = a[0]; a[0] = a[e]; a[e] = t;
        sift(0, e);
    }
}

// One CTA per sample.  Per chunk: histogram of the targets (shared-memory integer atomics), exclusive scan,
// fill, per-target sort (the fill order of the atomics is arbitrary; sorted lists make the gather's summation order
// -- and so the gradient -- reproducible bit for bit), coalesced write-out.
__global__ void __launch_bounds__(kEgBuildThreads)
edge_csr_build_kernel(const int32_t *__restrict__ idx, int N, int k, int S, int nch, int np1,
                      uint16_t *__restrict__ sub, uint16_t *__restrict__ list) {
    extern __shared__ int eg_sm[];
    int *cnt = eg_sm;                               // [N + 1] counts, then exclusive starts
    int *cur = eg_sm + (N + 1);                     // [N] fill cursors
    uint16_t *lst = reinterpret_cast<uint16_t *>(cur + N + 1);   // [S * k]
    __shared__ int wtot[32];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int SK = S * k;
    constexpr int IPT = (kEgThreads * kEgMaxTpt + kEgBuildThreads - 1) / kEgBuildThreads;   // 4 counters per thread
    for (int ch = 0; ch < nch; ++ch) {
        int rows = N - ch * S;
        if (rows > S) rows = S;
        const int ne = rows * k;
        const int32_t *ib = idx + ((size_t)b * N + (size_t)ch * S) * k;
        for (int i = tid; i <= N; i += kEgBuildThreads) cnt[i] = 0;
        __syncthreads();
        for (int e = tid; e < ne; e += kEgBuildThreads) atomicAdd(&cnt[min(max(ib[e], 0), N - 1)], 1);
        __syncthreads();
        // exclusive scan over cnt[0 .. N): thread t owns the IPT consecutive counters from t * IPT
        int v[IPT], tsum = 0;
#pragma unroll
        for (int i = 0; i < IPT; ++i) {
            const int j = tid * IPT + i;
            v[i] = j < N ? cnt[j] : 0;
            tsum += v[i];
        }
        int inc = tsum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int up = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += up;
        }
        if (lane == 31) wtot[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            int w = wtot[lane], winc = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int up = __shfl_up_sync(0xffffffffu, winc, o);
                if (lane >= o) winc += up;
            }
            wtot[lane] = winc - w;
        }
        __syncthreads();
        int run = wtot[warp] + inc - tsum;
#pragma unroll
        for (int i = 0; i < IPT; ++i) {
            const int j = tid * IPT + i;
            if (j < N) { cnt[j] = run; cur[j] = run; }
            run += v[i];
        }
        if (tid == 0) cnt[N] = ne;
        __syncthreads();
        uint16_t *srow = sub + ((size_t)b * nch + ch) * np1;
        for (int i = tid; i <= N; i += kEgBuildThreads) srow[i] = (uint16_t)cnt[i];
        for (int e = tid; e < ne; e += kEgBuildThreads) {
            const int t = min(max(ib[e], 0), N - 1);
            lst[atomicAdd(&cur[t], 1)] = (uint16_t)e;
        }
        __syncthreads();
        for (int i = tid; i < N; i += kEgBuildThreads) {
            const int lo = cnt[i], n = cnt[i + 1] - lo;
            if (n > 1) sort_u16(lst + lo, n);
        }
        __syncthreads();
        uint16_t *lrow = list + ((size_t)b * nch + ch) * SK;
        for (int e = tid; e < ne; e += kEgBuildThreads) lrow[e] = lst[e];
        __syncthreads();
    }
}

template <int TPT>
__global__ void __launch_bounds__(kEgThreads, 2)
edge_feature_bwd_gather_kernel(const float *__restrict__ g, const uint16_t *__restrict__ sub, const uint16_t *__restrict__ list,
                               int C, int N, int k, int nblocks, int ops, int S, int nch, int np1, float *__restrict__ gx) {
    extern __shared__ __align__(128) unsigned char eg_raw[];
    uint64_t *full = reinterpret_cast<uint64_t *>(eg_raw);        // [2]
    // stage: [nblocks][S * k] floats of g | [S * k] list entries | [np1] sub-list bounds   (all 16-byte multiples)
    const int c = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
    const int SK = S * k;
    const size_t NK = (size_t)N * k;
    const size_t stage_bytes = (size_t)nblocks * SK * 4 + (size_t)SK * 2 + (size_t)np1 * 2;
    unsigned char *stage0 = eg_raw + 128;
    const uint16_t *sp = sub + (size_t)b * nch * np1;
    const uint16_t *lp = list + (size_t)b * nch * SK;
    auto issue = [&](int ch) {                                    // one thread
        const int buf = ch & 1;
        int rows = N - ch * S;
        if (rows > S) rows = S;
        const uint32_t bytes = (uint32_t)rows * k * 4u;
        unsigned char *dst = stage0 + buf * stage_bytes;
        mbar_expect_tx(&full[buf], bytes * nblocks + (uint32_t)SK * 2u + (uint32_t)np1 * 2u);
        for (int q = 0; q < nblocks; ++q)
            tma_load_1d(dst + (size_t)q * SK * 4, g + (((size_t)b * nblocks + q) * C + c) * NK + (size_t)ch * SK, bytes, &full[buf]);
        tma_load_1d(dst + (size_t)nblocks * SK * 4, lp + (size_t)ch * SK, (uint32_t)SK * 2u, &full[buf]);
        tma_load_1d(dst + (size_t)nblocks * SK * 4 + (size_t)SK * 2, sp + (size_t)ch * np1, (uint32_t)np1 * 2u, &full[buf]);
    };
    if (tid == 0) {
        mbar_init(&full[0], 1);
        mbar_init(&full[1], 1);
        fence_mbar_init();
        fence_proxy_async();
        issue(0);
        if (nch > 1) issue(1);
    }
    __syncthreads();
    float acc[TPT];
#pragma unroll
    for (int s = 0; s < TPT; ++s) acc[s] = 0.f;
    for (int ch = 0; ch < nch; ++ch) {
        const int buf = ch & 1;
        int rows = N - ch * S;
        if (rows > S) rows = S;
        mbar_wait(&full[buf], (ch >> 1) & 1);
        const float *st = reinterpret_cast<const float *>(stage0 + buf * stage_bytes);
        const uint16_t *l = reinterpret_cast<const uint16_t *>(st + (size_t)nblocks * SK);
        const uint16_t *sb = l + SK;
        // incoming edges of this chunk, in list order (= ascending source slot): fixed summation order
#pragma unroll
        for (int s = 0; s < TPT; ++s) {
            const int j = tid + s * kEgThreads;
            if (j < N) {
                const int p1 = sb[j + 1];
                for (int p = sb[j]; p < p1; ++p) {
                    const int off = l[p];
                    float v = 0.f;
                    for (int q = 0; q < nblocks; ++q)
                        if (((ops >> (2 * q)) & 3) != PCD_EDGE_CENTER) v += st[(size_t)q * SK + off];
                    acc[s] += v;
                }
            }
        }
        // own-row terms: row r of the chunk is target ch*S + r, owned by thread (ch*S) % T + r in slot (ch*S) / T
        const int r = tid - (ch * S) % kEgThreads;
        if (r >= 0 && r < rows) {
            float own = 0.f;
            for (int q = 0; q < nblocks; ++q) {
                const int op = (ops >> (2 * q)) & 3;
                if (op == PCD_EDGE_NEIGHBOR) continue;
                const float *row = st + (size_t)q * SK + (size_t)r * k;
                float rs = 0.f;
                if ((k & 3) == 0) {
                    for (int kk = 0; kk < k; kk += 4) {
                        const float4 t4 = *reinterpret_cast<const float4 *>(row + kk);
                        rs += t4.x; rs += t4.y; rs += t4.z; rs += t4.w;
                    }
                } else {
                    for (int kk = 0; kk < k; ++kk) rs += row[kk];
                }
                own += op == PCD_EDGE_CENTER ? rs : -rs;
            }
            const int cs = (ch * S) / kEgThreads;
#pragma unroll
            for (int s = 0; s < TPT; ++s)
                if (s == cs) acc[s] += own;
        }
        __syncthreads();                                          // the stage has been read by everybody
        if (tid == 0 && ch + 2 < nch) {
            fence_proxy_async();
            issue(ch + 2);
        }
    }
    float *dst = gx + ((size_t)b * C + c) * N;
#pragma unroll
    for (int s = 0; s < TPT; ++s) {
        const int j = tid + s * kEgThreads;
        if (j < N) dst[j] = acc[s];
    }
}

// ----------------------------------------------------------------- farthest point sampling
// One CTA per sample.  Thread t owns the points i = t + s*T (s < PPT) and their running
// minimum distance to the chosen set in registers.  Per iteration: the new centroid is one
// broadcast load, every thread updates its PPT distances with the reference's arithmetic
// ((dx*dx + dy*dy) + dz*dz, then `dist < distance`), the block arg-max (first index on ties,
// as torch.max(dim)) is two REDUX per warp plus one shared-memory exchange -- ONE
// __syncthreads per iteration.
template <int T, int PPT>
__global__ void __launch_bounds__(T)
fps_kernel(const float *__restrict__ xyz, int64_t sb, int64_t sp, int64_t sc, int N, int npoint,
           const int32_t *__restrict__ start, int32_t *__restrict__ out) {
    constexpr int W = T / 32;
    __shared__ unsigned long long wbest[2][W];
    extern __shared__ float4 pts[];                         // [T * PPT] the cloud again: the chosen centroid is one broadcast LDS
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float *pb = xyz + b * sb;
    float px[PPT], py[PPT], pz[PPT], dist[PPT];
#pragma unroll
    for (int s = 0; s < PPT; ++s) {
        const int i = tid + s * T;
        if (i < N) {
            px[s] = pb[i * sp]; py[s] = pb[i * sp + sc]; pz[s] = pb[i * sp + 2 * sc];
            dist[s] = 1e10f;
        } else {
            px[s] = py[s] = pz[s] = 0.f;
            dist[s] = -1.f;                                 // never the maximum, never updated
        }
        pts[i] = make_float4(px[s], py[s], pz[s], 0.f);
    }
    __syncthreads();
    int far = start ? start[b] : 0;
    if (far < 0 || far >= N) far = 0;
    for (int it = 0; it < npoint; ++it) {
        if (tid == 0) out[(size_t)b * npoint + it] = far;
        if (it + 1 == npoint) break;
        const float4 c4 = pts[far];
        const float cx = c4.x, cy = c4.y, cz = c4.z;
        uint32_t bd = 0u, bi = 0xffffffffu;                  // best (distance bits, index) of this thread
#pragma unroll
        for (int s = 0; s < PPT; ++s) {
            const float dx = __fadd_rn(px[s], -cx), dy = __fadd_rn(py[s], -cy), dz = __fadd_rn(pz[s], -cz);
            const float d = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
            if (dist[s] >= 0.f && d < dist[s]) dist[s] = d;
            if (dist[s] >= 0.f) {
                const uint32_t u = __float_as_uint(dist[s]);   // dist >= 0: the bit pattern orders like the value
                if (u > bd || bi == 0xffffffffu) { bd = u; bi = (uint32_t)(tid + s * T); }   // s ascending: first index kept on ties
            }
        }
        const uint32_t wd = __reduce_max_sync(0xffffffffu, bd);
        const uint32_t wi = __reduce_min_sync(0xffffffffu, bd == wd ? bi : 0xffffffffu);
        if (lane == 0) wbest[it & 1][warp] = ((unsigned long long)wd << 32) | (0xffffffffu - wi);
        __syncthreads();
        // every warp folds the W per-warp results itself: max distance bits, then lowest index among the maxima
        const unsigned long long kw = lane < W ? wbest[it & 1][lane] : 0ull;
        const uint32_t kd = (uint32_t)(kw >> 32), ki = 0xffffffffu - (uint32_t)kw;
        const uint32_t bd2 = __reduce_max_sync(0xffffffffu, kd);
        far = (int)__reduce_min_sync(0xffffffffu, (lane < W && kd == bd2) ? ki : 0xffffffffu);
    }
}

// N beyond the register variants: running distances in shared memory, points re-read through L1.
template <int T>
__global__ void __launch_bounds__(T)
fps_large_kernel(const float *__restrict__ xyz, int64_t sb, int64_t sp, int64_t sc, int N, int npoint,
                 const int32_t *__restrict__ start, int32_t *__restrict__ out) {
    constexpr int W = T / 32;
    extern __shared__ float dist_s[];
    __shared__ unsigned long long wbest[2][W];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float *pb = xyz + b * sb;
    for (int i = tid; i < N; i += T) dist_s[i] = 1e10f;
    int far = start ? start[b] : 0;
    if (far < 0 || far >= N) far = 0;
    for (int it = 0; it < npoint; ++it) {
        if (tid == 0) out[(size_t)b * npoint + it] = far;
        if (it + 1 == npoint) break;
        const float cx = __ldg(pb + far * sp), cy = __ldg(pb + far * sp + sc), cz = __ldg(pb + far * sp + 2 * sc);
        uint32_t bd = 0u, bi = 0xffffffffu;
        for (int i = tid; i < N; i += T) {
            const float dx = __fadd_rn(__ldg(pb + i * sp), -cx), dy = __fadd_rn(__ldg(pb + i * sp + sc), -cy),
                        dz = __fadd_rn(__ldg(pb + i * sp + 2 * sc), -cz);
            const float d = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
            float cur = dist_s[i];
            if (d < cur) { cur = d; dist_s[i] = d; }
            const uint32_t u = __float_as_uint(cur);
            if (u > bd || bi == 0xffffffffu) { bd = u; bi = (uint32_t)i; }
        }
        const uint32_t wd = __reduce_max_sync(0xffffffffu, bd);
        const uint32_t wi = __reduce_min_sync(0xffffffffu, bd == wd ? bi : 0xffffffffu);
        if (lane == 0) wbest[it & 1][warp] = ((unsigned long long)wd << 32) | (0xffffffffu - wi);
        __syncthreads();
        // every warp folds the W per-warp results itself: max distance bits, then lowest index among the maxima
        const unsigned long long kw = lane < W ? wbest[it & 1][lane] : 0ull;
        const uint32_t kd = (uint32_t)(kw >> 32), ki = 0xffffffffu - (uint32_t)kw;
        const uint32_t bd2 = __reduce_max_sync(0xffffffffu, kd);
        far = (int)__reduce_min_sync(0xffffffffu, (lane < W && kd == bd2) ? ki : 0xffffffffu);
    }
}

static int pack_ops(int nblocks, const int *ops, int *packed) {
    if (nblocks < 1 || nblocks > 4 || !ops) return 0;
    int p = 0;
    for (int q = 0; q < nblocks; ++q) {
        if (ops[q] < 0 || ops[q] > 2) return 0;
        p |= ops[q] << (2 * q);
    }
    *packed = p;
    return 1;
}

}  // namespace pcd

using namespace pcd;

extern "C" int pcd_edge_feature_forward(const float *x, const int32_t *idx, int B, int C, int N, int k, int nblocks,
                                        const int *ops, float *out, void *stream) {
    int packed = 0;
    if (!x || !idx || !out || B <= 0 || C <= 0 || N <= 0 || k <= 0 || B > 65535 || !pack_ops(nblocks, ops, &packed)) {
        set_error("pcd_edge_feature_forward: bad argument B=%d C=%d N=%d k=%d nblocks=%d", B, C, N, k, nblocks);
        return PCD_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const long long NK = (long long)N * k;
    if ((size_t)N * sizeof(float) > 200 * 1024) {
        set_error("pcd_edge_feature_forward: N=%d exceeds the shared-memory row staging (N <= 51200)", N);
        return PCD_ERR_UNSUPPORTED;
    }
    // channel group: as many rows of N floats as fit 64 KB of shared memory (at least one, at most 16)
    int CG = kEdgeSmemFloats / N;
    if (CG < 1) CG = 1;
    if (CG > 16) CG = 16;
    if (CG > C) CG = C;
    const int cgroups = (C + CG - 1) / CG;
    if (cgroups > 65535) {
        set_error("pcd_edge_feature_forward: C=%d too large", C);
        return PCD_ERR_UNSUPPORTED;
    }
    const size_t smem = (size_t)CG * N * sizeof(float);
    const bool vec = (k & 3) == 0 && ((uintptr_t)out & 15) == 0 && ((uintptr_t)idx & 15) == 0;
    const long long nslots = vec ? NK / 4 : NK;
    // slices: enough CTAs for ~6 waves of 3 resident CTAs per SM, at least 4 slots per thread
    long long slices = (148LL * 3 * 6 + (long long)B * cgroups - 1) / ((long long)B * cgroups);
    const long long max_slices = (nslots + 4 * kEdgeThreads - 1) / (4 * kEdgeThreads);
    if (slices > max_slices) slices = max_slices;
    if (slices < 1) slices = 1;
    const long long sps = (nslots + slices - 1) / slices;
    const dim3 grid((unsigned)((nslots + sps - 1) / sps), cgroups, B);
    const auto kernel = vec ? edge_feature_fwd_kernel<4> : edge_feature_fwd_kernel<1>;
    if (smem > 48 * 1024) PCD_CUDA_CHECK(opt_in_smem(kernel, smem));
    kernel<<<grid, kEdgeThreads, smem, st>>>(x, idx, C, N, k, nblocks, packed, CG, sps, out);
    PCD_CUDA_CHECK(cudaGetLastError());
    return PCD_OK;
}

extern "C" size_t pcd_edge_feature_backward_workspace(int B, int N, int k, int nblocks) {
    EgPlan p;
    if (B <= 0 || N <= 0 || k <= 0 || !eg_plan(B, N, k, nblocks, &p)) return 0;
    return p.ws_bytes;
}

// A function template, not a lambda: it is instantiated at the end of the file, so the gather kernels' 128-byte aligned
// dynamic shared array is declared after those of the FPS kernels, whose dynamic shared memory it would otherwise align
// to 128 bytes as well (64 bytes more per CTA at T = 128).
template <int TPT>
static cudaError_t launch_eg_gather(const EgPlan &p, const float *g, const uint16_t *sub, const uint16_t *list, int B, int C,
                                    int N, int k, int nblocks, int packed, float *gx, cudaStream_t st) {
    if (p.smem_main > 48 * 1024) {
        const cudaError_t e = opt_in_smem(edge_feature_bwd_gather_kernel<TPT>, p.smem_main);
        if (e != cudaSuccess) return e;
    }
    edge_feature_bwd_gather_kernel<TPT><<<dim3(C, B), kEgThreads, p.smem_main, st>>>(g, sub, list, C, N, k, nblocks, packed, p.S,
                                                                                      p.nch, p.np1, gx);
    return cudaGetLastError();
}

extern "C" int pcd_edge_feature_backward(const float *g, const int32_t *idx, int B, int C, int N, int k, int nblocks,
                                         const int *ops, float *gx, void *workspace, size_t workspace_bytes, void *stream) {
    int packed = 0;
    if (!g || !idx || !gx || B <= 0 || C <= 0 || N <= 0 || k <= 0 || B > 65535 || !pack_ops(nblocks, ops, &packed)) {
        set_error("pcd_edge_feature_backward: bad argument B=%d C=%d N=%d k=%d nblocks=%d", B, C, N, k, nblocks);
        return PCD_ERR_ARG;
    }
    if (((uintptr_t)g & 15) != 0 || ((uintptr_t)idx & 15) != 0) {
        set_error("pcd_edge_feature_backward: g and idx must be 16-byte aligned");
        return PCD_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    EgPlan p;
    if (workspace && ((uintptr_t)workspace & 15) == 0 && C <= 65535 && eg_plan(B, N, k, nblocks, &p) &&
        workspace_bytes >= p.ws_bytes) {
        // gather form: invert the graph once per sample, then one CTA per (sample, channel)
        uint16_t *sub = reinterpret_cast<uint16_t *>(workspace);
        uint16_t *list = reinterpret_cast<uint16_t *>(reinterpret_cast<unsigned char *>(workspace) + p.sub_bytes);
        if (p.smem_build > 48 * 1024) PCD_CUDA_CHECK(opt_in_smem(edge_csr_build_kernel, p.smem_build));
        edge_csr_build_kernel<<<B, kEgBuildThreads, p.smem_build, st>>>(idx, N, k, p.S, p.nch, p.np1, sub, list);
        PCD_CUDA_CHECK(cudaGetLastError());
        cudaError_t e;
        if (p.tpt <= 1) e = launch_eg_gather<1>(p, g, sub, list, B, C, N, k, nblocks, packed, gx, st);
        else if (p.tpt <= 2) e = launch_eg_gather<2>(p, g, sub, list, B, C, N, k, nblocks, packed, gx, st);
        else if (p.tpt <= 4) e = launch_eg_gather<4>(p, g, sub, list, B, C, N, k, nblocks, packed, gx, st);
        else e = launch_eg_gather<8>(p, g, sub, list, B, C, N, k, nblocks, packed, gx, st);
        PCD_CUDA_CHECK(e);
        return PCD_OK;
    }
    const size_t smem = (size_t)N * sizeof(float);
    if (smem > 200 * 1024) {
        set_error("pcd_edge_feature_backward: N=%d exceeds the shared-memory accumulator (N <= 51200)", N);
        return PCD_ERR_UNSUPPORTED;
    }
    const bool vec = (k & 3) == 0;
    const auto kernel = vec ? edge_feature_bwd_kernel<4> : edge_feature_bwd_kernel<1>;
    if (smem > 48 * 1024) PCD_CUDA_CHECK(opt_in_smem(kernel, smem));
    kernel<<<dim3(C, B), kEdgeThreads, smem, st>>>(g, idx, C, N, k, nblocks, packed, gx);
    PCD_CUDA_CHECK(cudaGetLastError());
    return PCD_OK;
}

extern "C" int pcd_fps(const float *xyz, int64_t sb, int64_t sp, int64_t sc, int B, int N, int npoint,
                       const int32_t *start, int32_t *out, void *stream) {
    if (!xyz || !out || B <= 0 || N <= 0 || npoint <= 0) {
        set_error("pcd_fps: bad argument B=%d N=%d npoint=%d", B, N, npoint);
        return PCD_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    // up to 8192 points, each of T threads holds PPT points in registers (the cloud once more in shared memory, T * PPT
    // float4); beyond, the running distances live in shared memory
    const auto launch = [&](auto kernel, int threads, size_t smem) -> int {
        if (smem > 48 * 1024) PCD_CUDA_CHECK(opt_in_smem(kernel, smem));
        kernel<<<B, threads, smem, st>>>(xyz, sb, sp, sc, N, npoint, start, out);
        PCD_CUDA_CHECK(cudaGetLastError());
        return PCD_OK;
    };
    if (N <= 256) return launch(fps_kernel<128, 2>, 128, 128 * 2 * sizeof(float4));
    if (N <= 512) return launch(fps_kernel<128, 4>, 128, 128 * 4 * sizeof(float4));
    if (N <= 1024) return launch(fps_kernel<256, 4>, 256, 256 * 4 * sizeof(float4));
    if (N <= 2048) return launch(fps_kernel<256, 8>, 256, 256 * 8 * sizeof(float4));
    if (N <= 4096) return launch(fps_kernel<512, 8>, 512, 512 * 8 * sizeof(float4));
    if (N <= 8192) return launch(fps_kernel<1024, 8>, 1024, 1024 * 8 * sizeof(float4));
    const size_t smem = (size_t)N * sizeof(float);
    if (smem > 200 * 1024) {
        set_error("pcd_fps: N=%d exceeds the shared-memory distance array (N <= 51200)", N);
        return PCD_ERR_UNSUPPORTED;
    }
    return launch(fps_large_kernel<1024>, 1024, smem);
}
