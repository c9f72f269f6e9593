// pcd_knn.cu -- k-NN select sweep and ordered ball query for sm_100a.
//
// k-NN (pcd_knn_forward): every warp owns RQ query rows; its 32 lanes sweep the candidate
// columns of a shared-memory tile (TMA bulk copies for xyz clouds, channel-chunked tiles for
// C-channel DGCNN features).  Candidates that beat the row's current K-th distance are
// ballot-compacted into a per-row staging buffer; each time 32 are staged they are bitonic
// sorted across the warp and merged into the row's sorted top-K list, which lives in
// registers (one 64-bit (ordered distance, index) key per lane and list).  Keys order by
// distance first and index second, so exact ties resolve to the LOWEST index (the stable
// restatement of torch.topk the oracle uses).
//
// Reference semantics: attack/GeoA3/knn_utils.py:10-55, attack/CW/CW_utils/dist_utils.py:133-143,
// model/dgcnn.py:194-200, model/curvenet_util.py:10-26, model/pointnet2_utils.py:84-104.
#include <cstdlib>

#include "pcd_common.cuh"

namespace pcd {

constexpr int kKnnWarps = 8;
constexpr int kKnnThreads = kKnnWarps * 32;
constexpr int kKnnRQ = 4;          // query rows per warp
constexpr int kKnnTile = 512;      // xyz candidates per TMA stage (16 B each)
constexpr unsigned long long kEmptyKey = ~0ull;

static inline size_t align_up_k(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ------------------------------------------------------------------ warp-level key sorting
__device__ __forceinline__ unsigned long long shfl_xor_u64(unsigned long long v, int m) {
    return __shfl_xor_sync(0xffffffffu, v, m);
}
__device__ __forceinline__ unsigned long long shfl_u64(unsigned long long v, int src) {
    return __shfl_sync(0xffffffffu, v, src);
}
__device__ __forceinline__ unsigned long long umin64(unsigned long long a, unsigned long long b) { return a < b ? a : b; }
__device__ __forceinline__ unsigned long long umax64(unsigned long long a, unsigned long long b) { return a < b ? b : a; }

// full bitonic sort of one key per lane, ascending in lane order
__device__ __forceinline__ unsigned long long warp_sort32(unsigned long long key, int lane) {
#pragma unroll
    for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
            const unsigned long long o = shfl_xor_u64(key, j);
            const bool up = (lane & k) == 0 || k == 32;
            const bool lower = (lane & j) == 0;
            // keep the smaller key iff (lower == up): one 64-bit compare (swapping equal keys is harmless)
            key = ((o < key) == (lower == up)) ? o : key;
        }
    }
    return key;
}
// sort a bitonic sequence (one key per lane) ascending
__device__ __forceinline__ unsigned long long warp_bitonic_merge32(unsigned long long key, int lane) {
#pragma unroll
    for (int j = 16; j > 0; j >>= 1) {
        const unsigned long long o = shfl_xor_u64(key, j);
        key = ((o < key) == ((lane & j) == 0)) ? o : key;
    }
    return key;
}

// full bitonic sort of one fp32 value per lane, ascending in lane order (SHFL + FMNMX per stage)
__device__ __forceinline__ float warp_sort32_f32(float v, int lane) {
#pragma unroll
    for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
            const float o = __shfl_xor_sync(0xffffffffu, v, j);
            const bool up = (lane & k) == 0 || k == 32;
            const bool lower = (lane & j) == 0;
            v = (lower == up) ? fminf(v, o) : fmaxf(v, o);
        }
    }
    return v;
}

// Merge an ascending run `s` (one key per lane) into the NL sorted lists of a row.
template <int NL>
__device__ __forceinline__ void merge_run(unsigned long long (&L)[NL], unsigned long long s, int lane) {
#pragma unroll
    for (int l = 0; l < NL; ++l) {
        const unsigned long long rev = shfl_u64(s, 31 - lane);
        const unsigned long long lo = umin64(L[l], rev);
        const unsigned long long hi = umax64(L[l], rev);
        L[l] = warp_bitonic_merge32(lo, lane);
        if (l + 1 < NL) s = warp_bitonic_merge32(hi, lane);
    }
}

__device__ __forceinline__ float key_threshold(unsigned long long kth) {
    return kth == kEmptyKey ? __int_as_float(0x7f800000) : ordered_to_f32((uint32_t)(kth >> 32));
}

// Per-row select state shared by the xyz and the feature kernels.
//
// The heavy part -- sort the 32 staged keys, merge them into the row's sorted lists, carry the
// overflow, tighten the threshold -- is ONE out-of-line function per NL.  Inlined into every
// unrolled offer() it made the select kernels 9.5 K SASS instructions long and the instruction
// cache their bottleneck (ncu: stall_no_instruction 7.1 per issue on knnc_kernel).
template <int NL>
struct SelState {
    unsigned long long L[NL];
    float thr;
};

template <int NL>
__device__ __noinline__ SelState<NL> merge_staged(SelState<NL> s, unsigned long long *buf, int cnt, int lane, int K) {
    // cnt >= 32: buf[0..31] is merged, buf[32..cnt-1] carried to the front; cnt < 32 (final
    // flush): buf[0..cnt-1] is merged
    __syncwarp();
    const unsigned long long run = warp_sort32((cnt >= 32 || lane < cnt) ? buf[lane] : kEmptyKey, lane);
    merge_run<NL>(s.L, run, lane);
    const int rem = cnt - 32;
    const unsigned long long carry = (lane < rem) ? buf[32 + lane] : kEmptyKey;
    __syncwarp();
    if (lane < rem) buf[lane] = carry;
    unsigned long long kl = s.L[0];
#pragma unroll
    for (int l = 1; l < NL; ++l)
        if (((K - 1) >> 5) == l) kl = s.L[l];
    s.thr = fminf(s.thr, key_threshold(shfl_u64(kl, (K - 1) & 31)));   // only ever tightens (thr may start below +inf)
    __syncwarp();
    return s;
}

template <int NL>
struct RowSelect {
    SelState<NL> st;
    int cnt;
    __device__ __forceinline__ void init() {
#pragma unroll
        for (int l = 0; l < NL; ++l) st.L[l] = kEmptyKey;
        st.thr = __int_as_float(0x7f800000);
        cnt = 0;
    }
    // stage the passing lanes of one 32-candidate step; merge when 32 are staged
    // (buf holds 63 keys: at most 31 waiting + 32 new)
    __device__ __forceinline__ void offer(float d, int j, unsigned long long *buf, int lane, int K) {
        const bool pass = d < st.thr;
        const unsigned mask = __ballot_sync(0xffffffffu, pass);
        if (mask == 0) return;
        if (pass) buf[cnt + __popc(mask & ((1u << lane) - 1u))] = make_key(d, (uint32_t)j);
        cnt += __popc(mask);
        if (cnt >= 32) {
            st = merge_staged<NL>(st, buf, cnt, lane, K);
            cnt -= 32;
        }
    }
    // Four candidates per lane (indices j..j+3) in one out-of-line compaction (stage4 below).
    __device__ __forceinline__ void offer4(const float (&d)[4], int j, unsigned long long *buf, int lane, int K);
    __device__ __forceinline__ void finish(unsigned long long *buf, int lane, int K) {
        if (cnt > 0) {
            st = merge_staged<NL>(st, buf, cnt, lane, K);
            cnt = 0;
        }
    }
    __device__ __forceinline__ void store(float *dists, int32_t *idx, size_t base, int lane, int K) const {
#pragma unroll
        for (int l = 0; l < NL; ++l) {
            const int k = l * 32 + lane;
            if (k < K) {
                if (dists) dists[base + k] = ordered_to_f32((uint32_t)(st.L[l] >> 32));
                idx[base + k] = (int32_t)(uint32_t)st.L[l];
            }
        }
    }
};

// Stage the passing ones of four candidates per lane (indices j..j+3) with ONE compaction: the
// per-lane pass counts (0..4) are prefix-summed over the warp with three bit-plane ballots.
// When more than 32 pass (the staging buffer holds 31 waiting + 32 new keys) the candidates go
// through four single rounds.  Out of line for the same instruction-cache reason as merge_staged.
template <int NL>
struct SelStateCnt {
    SelState<NL> st;
    int cnt;
};

template <int NL>
__device__ __noinline__ SelStateCnt<NL> stage4(SelStateCnt<NL> s, float d0, float d1, float d2, float d3, int j,
                                               unsigned long long *buf, int lane, int K) {
    const float thr = s.st.thr;
    const bool p0 = d0 < thr, p1 = d1 < thr, p2 = d2 < thr, p3 = d3 < thr;
    const int c = (int)p0 + (int)p1 + (int)p2 + (int)p3;
    const unsigned b0 = __ballot_sync(0xffffffffu, c & 1), b1 = __ballot_sync(0xffffffffu, c & 2),
                   b2 = __ballot_sync(0xffffffffu, c & 4);
    const int total = __popc(b0) + 2 * __popc(b1) + 4 * __popc(b2);
    if (total == 0) return s;
    if (total <= 32) {
        const unsigned lt = (1u << lane) - 1u;
        int pos = s.cnt + __popc(b0 & lt) + 2 * __popc(b1 & lt) + 4 * __popc(b2 & lt);
        if (p0) buf[pos++] = make_key(d0, (uint32_t)j);
        if (p1) buf[pos++] = make_key(d1, (uint32_t)(j + 1));
        if (p2) buf[pos++] = make_key(d2, (uint32_t)(j + 2));
        if (p3) buf[pos] = make_key(d3, (uint32_t)(j + 3));
        s.cnt += total;
        if (s.cnt >= 32) {
            s.st = merge_staged<NL>(s.st, buf, s.cnt, lane, K);
            s.cnt -= 32;
        }
        return s;
    }
    const float dd[4] = {d0, d1, d2, d3};
#pragma unroll 1
    for (int e = 0; e < 4; ++e) {
        const bool pass = dd[e] < s.st.thr;
        const unsigned mask = __ballot_sync(0xffffffffu, pass);
        if (mask == 0) continue;
        if (pass) buf[s.cnt + __popc(mask & ((1u << lane) - 1u))] = make_key(dd[e], (uint32_t)(j + e));
        s.cnt += __popc(mask);
        if (s.cnt >= 32) {
            s.st = merge_staged<NL>(s.st, buf, s.cnt, lane, K);
            s.cnt -= 32;
        }
    }
    return s;
}

template <int NL>
__device__ __forceinline__ void RowSelect<NL>::offer4(const float (&d)[4], int j, unsigned long long *buf, int lane, int K) {
    SelStateCnt<NL> s;
    s.st = st; s.cnt = cnt;
    s = stage4<NL>(s, d[0], d[1], d[2], d[3], j, buf, lane, K);
    st = s.st; cnt = s.cnt;
}

// K-th smallest (0-based rank K-1 < 32) of one fp32 value per lane, bumped to the next float up
// (thresholds are tested with d < thr and d == kth must pass); +inf / NaN stay +inf.  Out of line.
__device__ __noinline__ float warp_kth_bound(float v, int lane, int K) {
    const float kth = __shfl_sync(0xffffffffu, warp_sort32_f32(v, lane), K - 1);
    return kth < __int_as_float(0x7f800000) ? ordered_to_f32(f32_to_ordered(kth) + 1u) : __int_as_float(0x7f800000);
}

// -------------------------------------------------------------------------- prep (xyz clouds)
// rowq[b][i] = (-2x,-2y,-2z,nrow)   colq[b][j] = (x,y,z,ncol)   padded points inert (n = +inf)
__global__ void knn3_prep_kernel(const float *__restrict__ rows, int64_t r_sb, int64_t r_sp, int64_t r_sc,
                                 const float *__restrict__ cols, int64_t c_sb, int64_t c_sp, int64_t c_sc,
                                 int B, int N, int M, int Npad, int Mpad, int norm_kind, int swap_norms,
                                 float4 *__restrict__ rowq, float4 *__restrict__ colq, float *__restrict__ colpk,
                                 int *__restrict__ ovf_cnt) {
    const long long per_b = (long long)Npad + Mpad;
    const long long total = per_b * B;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const int b = (int)(t / per_b);
        const int p = (int)(t - (long long)b * per_b);
        if (p == 0 && ovf_cnt) ovf_cnt[b] = 0;           // overflow list of the collect pipeline (was a separate memset)
        const bool is_row = p < Npad;
        const int i = is_row ? p : p - Npad;
        const int n_own = is_row ? N : M;
        float x = 0.f, y = 0.f, z = 0.f, n = __int_as_float(0x7f800000);
        if (i < n_own) {
            const float *s = is_row ? rows + b * r_sb + i * r_sp : cols + b * c_sb + i * c_sp;
            const int64_t sc = is_row ? r_sc : c_sc;
            x = s[0]; y = s[sc]; z = s[2 * sc];
            if (swap_norms) {
                const float *o = is_row ? cols + b * c_sb + i * c_sp : rows + b * r_sb + i * r_sp;
                const int64_t oc = is_row ? c_sc : r_sc;
                n = sq_norm3(norm_kind, o[0], o[oc], o[2 * oc]);
            } else {
                n = sq_norm3(norm_kind, x, y, z);
            }
        }
        if (is_row) {
            rowq[(size_t)b * Npad + i] = make_float4(-2.f * x, -2.f * y, -2.f * z, n);
        } else {
            colq[(size_t)b * Mpad + i] = make_float4(x, y, z, n);
            float *rec = colpk + ((size_t)b * Mpad + (i & ~1)) * 4 + (i & 1);   // pair records for the pre-pass
            rec[0] = x; rec[2] = y; rec[4] = z; rec[6] = n;
        }
    }
}

// ------------------------------------------------------- pre-pass: chunk minima -> tight thresholds
// The K-th smallest distance of a row is <= the K-th smallest of its per-chunk minima (each
// chunk minimum is a distinct candidate).  A cheap row sweep (rows in lanes, packed math, one
// FMNMX3 per two pairs -- the NN-1 sweep without its column side) yields the chunk minima, a
// thread per row takes their K-th smallest, and the select kernel starts from that threshold
// instead of +inf: only ~1.2 K candidates per row ever reach the staging buffer, so the bitonic
// merges (the dominant cost of a cold-start select) almost disappear.  Exactness is unaffected:
// the threshold is a true upper bound of the K-th distance and the select kernel keeps every
// candidate with d <= threshold.
constexpr int kPreR = 4;          // rows per lane
constexpr int kPreTile = 256;     // columns per TMA stage
constexpr int kPreMaxChunks = 64;

struct PreSmem {
    float4 tile[2][kPreTile + 2];
    uint64_t full[2];
};

template <int FORM>
__global__ void __launch_bounds__(128)
knn3_chunkmin_kernel(const float4 *__restrict__ rowq, const float4 *__restrict__ colpk, int Npad, int Mpad, int M_all,
                     int W /* columns per chunk, even */, int G, int cps /* chunks per column split */,
                     float *__restrict__ cm /* [B][G][Npad] */) {
    constexpr int R = kPreR;
    __shared__ __align__(128) PreSmem sm;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.y;
    const int row0 = blockIdx.x * (128 * R) + warp * (32 * R) + lane;       // rows row0 + 32 r
    // column split blockIdx.z owns the chunks [c0, c1): columns [c0 W, min(M, c1 W)); stages are counted
    // from its first column (W is even, so pair records stay aligned; the workspace has one stage of slack)
    const int c0 = blockIdx.z * cps;
    const int c1 = (c0 + cps < G) ? c0 + cps : G;
    const int col_begin = c0 * W;
    const int col_end = (c1 * W < M_all) ? c1 * W : M_all;
    const int M = col_end - col_begin;                                       // columns of this split
    if (M <= 0) return;
    const int ntiles = (M + kPreTile - 1) / kPreTile;
    const float4 *src = colpk + (size_t)b * Mpad + col_begin;
    const uint32_t tile_bytes = kPreTile * 16u;
    if (tid == 0) {
        mbar_init(&sm.full[0], 1);
        mbar_init(&sm.full[1], 1);
        fence_mbar_init();
        fence_proxy_async();
        mbar_expect_tx(&sm.full[0], tile_bytes);
        tma_load_1d(sm.tile[0], src, tile_bytes, &sm.full[0]);
        if (ntiles > 1) {
            mbar_expect_tx(&sm.full[1], tile_bytes);
            tma_load_1d(sm.tile[1], src + kPreTile, tile_bytes, &sm.full[1]);
        }
    }
    if (tid < 4) sm.tile[tid >> 1][kPreTile + (tid & 1)] = make_float4(0.f, 0.f, 0.f, 0.f);
    __syncthreads();

    float qx[R], qy[R], qz[R], qn[R], m[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const float4 q = __ldg(&rowq[(size_t)b * Npad + row0 + 32 * r]);
        qx[r] = q.x; qy[r] = q.y; qz[r] = q.z; qn[r] = q.w;
        m[r] = __int_as_float(0x7f800000);
    }
    float *out = cm + (size_t)b * G * Npad + row0;
    int chunk = c0, left = W / 2;                      // packed steps left in the current chunk
    const int total_steps = (M + 1) / 2;
    int done = 0;
    for (int t = 0; t < ntiles; ++t) {
        const int buf = t & 1;
        mbar_wait(&sm.full[buf], (t >> 1) & 1);
        const float4 *t4 = sm.tile[buf];
        int nsteps = total_steps - done;
        if (nsteps > kPreTile / 2) nsteps = kPreTile / 2;
        float4 A = t4[0], Bv = t4[1];
        for (int s = 0; s < nsteps; ++s) {
            const float4 An = t4[2 * s + 2], Bn = t4[2 * s + 3];
            const f32x2 X = pack2(A.x, A.y), Y = pack2(A.z, A.w);
            const f32x2 Z = pack2(Bv.x, Bv.y), Nn = pack2(Bv.z, Bv.w);
#pragma unroll
            for (int r = 0; r < R; ++r) {
                f32x2 d;
                if (FORM == PCD_FORM_COL_ROW) {
                    // d = (t + ncol) + nrow: the row norm is the outer term and fl(. + nrow) is monotone,
                    // so the chunk minimum of d is fl(min(t + ncol) + nrow): add it once per chunk
                    f32x2 tt = mul2_s(qx[r], X);
                    tt = fma2_s(qy[r], Y, tt);
                    tt = fma2_s(qz[r], Z, tt);
                    d = add2(tt, Nn);
                } else {
                    d = pair_dist_x2<FORM>(qx[r], qy[r], qz[r], qn[r], X, Y, Z, Nn);
                }
                float lo, hi;
                unpack2(d, lo, hi);
                m[r] = min3(m[r], lo, hi);
            }
            A = An; Bv = Bn;
            if (--left == 0) {
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    out[(size_t)chunk * Npad + 32 * r] = (FORM == PCD_FORM_COL_ROW) ? __fadd_rn(m[r], qn[r]) : m[r];
                    m[r] = __int_as_float(0x7f800000);
                }
                ++chunk;
                left = W / 2;
            }
        }
        done += nsteps;
        __syncthreads();
        if (tid == 0 && t + 2 < ntiles) {
            mbar_expect_tx(&sm.full[buf], tile_bytes);
            tma_load_1d(sm.tile[buf], src + (size_t)(t + 2) * kPreTile, tile_bytes, &sm.full[buf]);
        }
    }
    if (chunk < c1) {      // last, partial chunk
#pragma unroll
        for (int r = 0; r < R; ++r)
            out[(size_t)chunk * Npad + 32 * r] = (FORM == PCD_FORM_COL_ROW) ? __fadd_rn(m[r], qn[r]) : m[r];
    }
}

// thread per row: K-th smallest of the G <= GP chunk minima with a fully unrolled bitonic sorting
// network over registers (no shared memory, no divergence; 2 FMNMX per compare-exchange).  The
// shared-memory insertion list it replaces took longer than the chunk-minima sweep itself.
template <int GP>
__global__ void __launch_bounds__(128)
knn_threshold_kernel(const float *__restrict__ cm, int Npad, int G, int K, float *__restrict__ thr0) {
    const int b = blockIdx.y, i = blockIdx.x * 128 + threadIdx.x;
    const float *src = cm + (size_t)b * G * Npad + i;
    const float inf = __int_as_float(0x7f800000);
    float v[GP];
#pragma unroll
    for (int g = 0; g < GP; ++g) v[g] = g < G ? src[(size_t)g * Npad] : inf;
#pragma unroll
    for (int k = 2; k <= GP; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
#pragma unroll
            for (int e = 0; e < GP; ++e) {
                const int l = e ^ j;
                if (l > e) {
                    const float x = v[e], y = v[l];
                    const bool up = (e & k) == 0;
                    v[e] = up ? fminf(x, y) : fmaxf(x, y);
                    v[l] = up ? fmaxf(x, y) : fminf(x, y);
                }
            }
        }
    }
    float kth = inf;
#pragma unroll
    for (int g = 0; g < GP; ++g)
        if (g == K - 1) kth = v[g];
    // smallest float above kth: candidates are tested with d < thr, and d == kth must pass
    thr0[(size_t)b * Npad + i] = kth < inf ? ordered_to_f32(f32_to_ordered(kth) + 1u) : inf;
}

// ------------------------------------------------- collect pass: candidates below the threshold
// Rows in lanes, packed math -- the chunk-minima sweep again -- but now every row knows a tight
// exact upper bound thr of its K-th distance, so only ~1.2 K of its M candidates matter.
//   phase 1 (per 256-column stage): the minimum of every 8-column group is compared with the
//     row's bound; hits are pushed to a lane-private byte queue in shared memory (predicated
//     store, no branch).  For form COL_ROW the outer row norm is moved into the bound
//     (4 instead of 5 math instructions per pair); the moved bound is widened by a few ulp so
//     the filter can only err towards extra hits.
//   phase 2: each lane drains its queue: the 8 columns of a hit are re-evaluated with the exact
//     arithmetic of `FORM`, and those with d < thr are appended (as (ordered distance, index)
//     keys) to the row's candidate list in the workspace -- lane-private rows and per-split
//     lists, so no atomics.
// knn3_final_kernel then keeps the K smallest keys of every row (thread per row, insertion
// network in registers).  A row whose list overflows is handed to knn3_kernel (the warp-per-row
// select) through a per-sample overflow list, so the result is exact for any input.
constexpr int kColGroup = 8;                                   // columns per tested group
constexpr int kColGroups = kPreTile / kColGroup;               // 32 groups per stage

struct CollectSmem {
    float4 tile[2][kPreTile + 2];
    uint64_t full[2];
    unsigned int cnt[kPreR][128];
    float4 rowrec[kPreR][128];                       // the lane's row records and bounds for phase 2 (dynamic row index)
    float rowthr[kPreR][128];
    unsigned char queue[kColGroups * kPreR][128];
};

template <int FORM>
__global__ void __launch_bounds__(128)
knn3_collect_kernel(const float4 *__restrict__ rowq, const float4 *__restrict__ colpk, const float *__restrict__ thr0,
                    int B, int Npad, int Mpad, int M, int nsplit, int tps /* stages per split */, int caps,
                    unsigned long long *__restrict__ cand, unsigned int *__restrict__ cnt_g) {
    constexpr int R = kPreR;
    __shared__ __align__(128) CollectSmem sm;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.y;
    const int rt = blockIdx.x / nsplit, sp = blockIdx.x - rt * nsplit;
    const int row0 = rt * (128 * R) + warp * (32 * R) + lane;               // rows row0 + 32 r
    const int ntiles_all = (M + kPreTile - 1) / kPreTile;
    const int t_begin = sp * tps;
    const int t_end = (t_begin + tps < ntiles_all) ? t_begin + tps : ntiles_all;
    const int ntiles = t_end - t_begin;
    const float4 *src = colpk + (size_t)b * Mpad + (size_t)t_begin * kPreTile;
    const uint32_t tile_bytes = kPreTile * 16u;
    if (tid == 0) {
        mbar_init(&sm.full[0], 1);
        mbar_init(&sm.full[1], 1);
        fence_mbar_init();
        fence_proxy_async();
        if (ntiles > 0) {
            mbar_expect_tx(&sm.full[0], tile_bytes);
            tma_load_1d(sm.tile[0], src, tile_bytes, &sm.full[0]);
        }
        if (ntiles > 1) {
            mbar_expect_tx(&sm.full[1], tile_bytes);
            tma_load_1d(sm.tile[1], src + kPreTile, tile_bytes, &sm.full[1]);
        }
    }
    __syncthreads();

    const float inf = __int_as_float(0x7f800000);
    float qx[R], qy[R], qz[R], qn[R], bound[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const float4 q = __ldg(&rowq[(size_t)b * Npad + row0 + 32 * r]);
        const float thr = __ldg(&thr0[(size_t)b * Npad + row0 + 32 * r]);
        qx[r] = q.x; qy[r] = q.y; qz[r] = q.z; qn[r] = q.w;
        if (FORM == PCD_FORM_COL_ROW) {
            // fl(u + n) < thr  ==>  u < (thr - n) + ulp(thr):  widen the computed difference by 2^-21 of the magnitudes
            const float c = __fadd_rn(thr, -q.w);
            bound[r] = __fadd_rn(c, __fmaf_rn(__fadd_rn(fabsf(c), fabsf(thr)), 4.76837158e-7f, 1e-37f));
        } else {
            bound[r] = thr;
        }
        sm.cnt[r][tid] = 0u;
        sm.rowrec[r][tid] = q;
        sm.rowthr[r][tid] = thr;
    }
    const size_t list_base = ((size_t)sp * B + b) * (size_t)caps * Npad;     // + slot * Npad + row

    for (int t = 0; t < ntiles; ++t) {
        const int buf = t & 1;
        mbar_wait(&sm.full[buf], (t >> 1) & 1);
        const float4 *t4 = sm.tile[buf];
        // ---- phase 1
        int qcount = 0;
#pragma unroll 1
        for (int g = 0; g < kColGroups; ++g) {
            float m[R];
#pragma unroll
            for (int r = 0; r < R; ++r) m[r] = inf;
#pragma unroll
            for (int s4 = 0; s4 < kColGroup / 2; ++s4) {
                const int step = g * (kColGroup / 2) + s4;
                const float4 A = t4[2 * step], Bv = t4[2 * step + 1];
                const f32x2 X = pack2(A.x, A.y), Y = pack2(A.z, A.w);
                const f32x2 Z = pack2(Bv.x, Bv.y), Nn = pack2(Bv.z, Bv.w);
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    f32x2 d;
                    if (FORM == PCD_FORM_COL_ROW) {
                        f32x2 tt = mul2_s(qx[r], X);
                        tt = fma2_s(qy[r], Y, tt);
                        tt = fma2_s(qz[r], Z, tt);
                        d = add2(tt, Nn);
                    } else {
                        d = pair_dist_x2<FORM>(qx[r], qy[r], qz[r], qn[r], X, Y, Z, Nn);
                    }
                    float lo, hi;
                    unpack2(d, lo, hi);
                    m[r] = min3(m[r], lo, hi);
                }
            }
#pragma unroll
            for (int r = 0; r < R; ++r) {
                if (m[r] < bound[r]) {
                    sm.queue[qcount][tid] = (unsigned char)(r * kColGroups + g);
                    ++qcount;
                }
            }
        }
        // ---- phase 2
        const int jbase = (t_begin + t) * kPreTile;
        for (int e = 0; e < qcount; ++e) {
            const int code = sm.queue[e][tid];
            const int r = code / kColGroups, g = code - r * kColGroups;
            const int row = row0 + 32 * r;
            const float4 q = sm.rowrec[r][tid];
            const float thr = sm.rowthr[r][tid];
            unsigned int slot = sm.cnt[r][tid];
            unsigned long long *dst = cand + list_base + row;
            float dd[kColGroup];
            unsigned int pm = 0u;                            // bit = column offset inside the group
#pragma unroll
            for (int s4 = 0; s4 < kColGroup / 2; ++s4) {
                // lanes visit the four pair records of their group in rotated order: the groups are 128 B
                // apart (one bank row), unrotated every lane would hit the same four banks
                const int rs = (s4 + lane) & (kColGroup / 2 - 1);
                const int step = g * (kColGroup / 2) + rs;
                const float4 A = t4[2 * step], Bv = t4[2 * step + 1];
                const f32x2 d = pair_dist_x2<FORM>(q.x, q.y, q.z, q.w, pack2(A.x, A.y), pack2(A.z, A.w),
                                                   pack2(Bv.x, Bv.y), pack2(Bv.z, Bv.w));
                unpack2(d, dd[2 * s4], dd[2 * s4 + 1]);
                pm |= ((dd[2 * s4] < thr ? 1u : 0u) | (dd[2 * s4 + 1] < thr ? 2u : 0u)) << (2 * rs);
            }
            while (pm) {                                     // usually one pass: the group's single candidate
                const int co = __ffs(pm) - 1;
                pm &= pm - 1u;
                const int k = 2 * (((co >> 1) - lane) & (kColGroup / 2 - 1)) + (co & 1);     // register holding column co
                float v = dd[0];
#pragma unroll
                for (int u = 1; u < kColGroup; ++u) v = (k == u) ? dd[u] : v;
                if (slot < (unsigned)caps) dst[(size_t)slot * Npad] = make_key(v, (uint32_t)(jbase + g * kColGroup + co));
                ++slot;
            }
            sm.cnt[r][tid] = slot;
        }
        __syncthreads();                                   // stage fully read by every warp
        if (tid == 0 && t + 2 < ntiles) {
            mbar_expect_tx(&sm.full[buf], tile_bytes);
            tma_load_1d(sm.tile[buf], src + (size_t)(t + 2) * kPreTile, tile_bytes, &sm.full[buf]);
        }
    }
#pragma unroll
    for (int r = 0; r < R; ++r)
        cnt_g[((size_t)sp * B + b) * Npad + row0 + 32 * r] = sm.cnt[r][tid];
}

// thread per row: the K smallest of the row's candidate keys, ascending (insertion network over
// KT >= K registers).  Rows with an overflowed list go to the per-sample overflow list instead
// (knn3_kernel rewrites their outputs afterwards).  Results leave through shared memory so that
// a warp writes its 32 x K outputs as one contiguous, coalesced block.
template <int KT>
__global__ void __launch_bounds__(128, (KT <= 20) ? 8 : ((KT <= 24) ? 6 : ((KT <= 32) ? 5 : 3)))     // occupancy hides the candidate-load latency
knn3_final_kernel(const unsigned long long *__restrict__ cand, const unsigned int *__restrict__ cnt_g, int B, int N,
                  int Npad, int nsplit, int caps, int K, float *__restrict__ dists, int32_t *__restrict__ idx,
                  int *__restrict__ ovf_cnt, int *__restrict__ ovf_rows) {
    extern __shared__ uint32_t stage_dyn[];                  // [4 warps][32 * K] output staging
    __shared__ unsigned short s_n[16][128];
    const int b = blockIdx.y, i = blockIdx.x * 128 + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long L[KT];
#pragma unroll
    for (int k = 0; k < KT; ++k) L[k] = kEmptyKey;
    if (i < N) {
        // all list lengths first (independent loads), kept in shared memory for the flat walk below
        unsigned int total = 0;
        bool over = false;
        for (int sp = 0; sp < nsplit; ++sp) {
            const unsigned int n = cnt_g[((size_t)sp * B + b) * Npad + i];
            s_n[sp][threadIdx.x] = (unsigned short)(n > 0xffffu ? 0xffffu : n);
            over |= n > (unsigned)caps;
            total += n;
        }
        if (over) {
            const int pos = atomicAdd(&ovf_cnt[b], 1);
            ovf_rows[(size_t)b * Npad + pos] = i;
        } else {
            // One flat walk over the row's lists (a warp iterates max-over-lanes of the TOTAL count, not
            // the sum of per-list maxima); the next key is in flight while the current one is inserted.
            // Insertion = shift: every position compares and selects independently (no serial
            // min/max chain through the KT registers), ONE instance of the network in the kernel.
            const size_t split_stride = (size_t)B * caps * Npad;
            const unsigned long long *src = cand + (size_t)b * caps * Npad + i;
            int sp = 0;
            unsigned int s = 0, n_cur = s_n[0][threadIdx.x], fetched = 0;
            auto fetch = [&]() -> unsigned long long {       // next key of the flat walk (kEmptyKey past the end)
                if (fetched >= total) return kEmptyKey;
                while (s >= n_cur && sp + 1 < nsplit) { ++sp; s = 0; n_cur = s_n[sp][threadIdx.x]; src += split_stride; }
                const unsigned long long v = src[(size_t)s * Npad];
                ++s; ++fetched;
                return v;
            };
            auto insert = [&](unsigned long long c) {
                if (c < L[KT - 1]) {
#pragma unroll
                    for (int k = KT - 1; k >= 0; --k) {
                        const bool pk = c < L[k];
                        const bool pk1 = k > 0 ? (c < L[k > 0 ? k - 1 : 0]) : false;
                        L[k] = pk ? (pk1 ? L[k > 0 ? k - 1 : 0] : c) : L[k];
                    }
                }
            };
            // four keys in flight: a key is loaded four insertions (~1 us of ALU work) before it is needed
            unsigned long long k0 = fetch(), k1 = fetch(), k2 = fetch(), k3 = fetch();
#pragma unroll 1
            for (unsigned int t = 0; t < total; t += 4) {
                insert(k0); k0 = fetch();
                insert(k1); k1 = fetch();
                insert(k2); k2 = fetch();
                insert(k3); k3 = fetch();
            }
        }
    }
    const int i0 = blockIdx.x * 128 + warp * 32;             // first row of this warp
    const int nvalid = N - i0 < 32 ? N - i0 : 32;
    if (nvalid <= 0) return;
    const size_t base = ((size_t)b * N + i0) * K;
    uint32_t *sg = stage_dyn + (size_t)warp * 32 * K;
    if (dists) {
#pragma unroll
        for (int k = 0; k < KT; ++k)
            if (k < K) sg[lane * K + k] = __float_as_uint(ordered_to_f32((uint32_t)(L[k] >> 32)));
        __syncwarp();
        for (int e = lane; e < nvalid * K; e += 32) dists[base + e] = __uint_as_float(sg[e]);
        __syncwarp();
    }
#pragma unroll
    for (int k = 0; k < KT; ++k)
        if (k < K) sg[lane * K + k] = (uint32_t)L[k];
    __syncwarp();
    for (int e = lane; e < nvalid * K; e += 32) idx[base + e] = (int32_t)sg[e];
}

// ------------------------------------------------------------------------- xyz k-NN kernel
struct Knn3Smem {
    float4 tile[2][kKnnTile];                              // 2 x 8 KB candidate tiles (TMA)
    unsigned long long stage[kKnnWarps][kKnnRQ][64];       // 16 KB staging buffers
    uint64_t full[2];
};

template <int FORM, int NL>
__global__ void __launch_bounds__(kKnnThreads)
knn3_kernel(const float4 *__restrict__ rowq, const float4 *__restrict__ colq, const float *__restrict__ thr0,
            int N, int M, int Npad, int Mpad, int K, float *__restrict__ dists, int32_t *__restrict__ idx,
            const int *__restrict__ ovf_cnt, const int *__restrict__ ovf_rows) {
    __shared__ __align__(128) Knn3Smem sm;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.y;
    // overflow mode (ovf_rows != NULL): the CTA serves 32 entries of the sample's overflow list
    const int nlist = ovf_rows ? ovf_cnt[b] : 0;
    if (ovf_rows && (int)blockIdx.x * kKnnWarps * kKnnRQ >= nlist) return;
    const int row0 = (blockIdx.x * kKnnWarps + warp) * kKnnRQ;
    const int ntiles = (M + kKnnTile - 1) / kKnnTile;
    const float4 *src = colq + (size_t)b * Mpad;
    const uint32_t tile_bytes = kKnnTile * 16u;

    if (tid == 0) {
        mbar_init(&sm.full[0], 1);
        mbar_init(&sm.full[1], 1);
        fence_mbar_init();
        fence_proxy_async();
        mbar_expect_tx(&sm.full[0], tile_bytes);
        tma_load_1d(sm.tile[0], src, tile_bytes, &sm.full[0]);
        if (ntiles > 1) {
            mbar_expect_tx(&sm.full[1], tile_bytes);
            tma_load_1d(sm.tile[1], src + kKnnTile, tile_bytes, &sm.full[1]);
        }
    }
    __syncthreads();

    float4 q[kKnnRQ];
    int rowi[kKnnRQ];
    RowSelect<NL> sel[kKnnRQ];
#pragma unroll
    for (int r = 0; r < kKnnRQ; ++r) {
        rowi[r] = row0 + r;                                  // rows are padded to a multiple of 32 per CTA
        if (ovf_rows) rowi[r] = (row0 + r < nlist) ? ovf_rows[(size_t)b * Npad + row0 + r] : N;   // N: padded row, never stored
        q[r] = __ldg(&rowq[(size_t)b * Npad + (rowi[r] < Npad ? rowi[r] : 0)]);
        sel[r].init();
        if (thr0) sel[r].st.thr = __ldg(&thr0[(size_t)b * Npad + (rowi[r] < Npad ? rowi[r] : 0)]);
    }

    for (int t = 0; t < ntiles; ++t) {
        const int buf = t & 1;
        mbar_wait(&sm.full[buf], (t >> 1) & 1);
        const float4 *tile = sm.tile[buf];
        const int jbase = t * kKnnTile;
#pragma unroll 2
        for (int s = 0; s < kKnnTile / 32; ++s) {
            const float4 c = tile[s * 32 + lane];
            const int j = jbase + s * 32 + lane;
#pragma unroll
            for (int r = 0; r < kKnnRQ; ++r) {
                const float d = pair_dist_scalar<FORM>(q[r].x, q[r].y, q[r].z, q[r].w, c.x, c.y, c.z, c.w);
                sel[r].offer(d, j, sm.stage[warp][r], lane, K);
            }
        }
        __syncthreads();
        if (tid == 0 && t + 2 < ntiles) {
            mbar_expect_tx(&sm.full[buf], tile_bytes);
            tma_load_1d(sm.tile[buf], src + (size_t)(t + 2) * kKnnTile, tile_bytes, &sm.full[buf]);
        }
    }
#pragma unroll
    for (int r = 0; r < kKnnRQ; ++r) {
        sel[r].finish(sm.stage[warp][r], lane, K);
        const int i = rowi[r];
        if (i < N) sel[r].store(dists, idx, ((size_t)b * N + i) * K, lane, K);
    }
}

// ------------------------------------------------------------- C-channel (feature) k-NN
constexpr int kFcRows = 8;                          // query rows per warp
constexpr int kFcCtaRows = kKnnWarps * kFcRows;     // 64 query rows per CTA
constexpr int kFcTile = 128;                        // candidates per stage (4 per lane)
constexpr int kFcStage = 63;                        // staging keys per row (31 waiting + 32 new - 1)
// Workspace: rowT[b][C][Npad] (= -2 * feature, channel-major), rown[b][Npad], and the candidates
// in STAGE-major order colS[b][Mpad/128][C+1][128] -- the C channel rows of a 128-candidate
// stage followed by its norms -- so that one 1-D TMA bulk copy fetches a whole stage.
__global__ void knnc_prep_kernel(const float *__restrict__ rows, int64_t r_sb, int64_t r_sp, int64_t r_sc,
                                 const float *__restrict__ cols, int64_t c_sb, int64_t c_sp, int64_t c_sc,
                                 int B, int N, int M, int C, int Npad, int Mpad, int norm_kind, int swap_norms,
                                 float *__restrict__ rowT, float *__restrict__ rown,
                                 float *__restrict__ colS) {
    const long long per_b = (long long)Npad + Mpad;
    const long long total = per_b * B;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const int b = (int)(t / per_b);
        const int p = (int)(t - (long long)b * per_b);
        const bool is_row = p < Npad;
        const int i = is_row ? p : p - Npad;
        const int n_own = is_row ? N : M;
        const bool live = i < n_own;
        const float *own = is_row ? rows + b * r_sb + i * r_sp : cols + b * c_sb + i * c_sp;
        const int64_t osc = is_row ? r_sc : c_sc;
        const float *nsrc = own;
        int64_t nsc = osc;
        if (swap_norms) {
            nsrc = is_row ? cols + b * c_sb + i * c_sp : rows + b * r_sb + i * r_sp;
            nsc = is_row ? c_sc : r_sc;
        }
        float n = __int_as_float(0x7f800000);
        if (live) {
            const float v0 = nsrc[0];
            n = __fmul_rn(v0, v0);
            for (int k = 1; k < C; ++k) {
                const float v = nsrc[k * nsc];
                n = (norm_kind == PCD_NORM_FMA) ? __fmaf_rn(v, v, n) : __fadd_rn(n, __fmul_rn(v, v));
            }
        }
        if (is_row) {
            for (int k = 0; k < C; ++k) rowT[((size_t)b * C + k) * Npad + i] = live ? -2.f * own[k * osc] : 0.f;
            rown[(size_t)b * Npad + i] = n;
        } else {
            float *dst = colS + ((size_t)b * (Mpad / kFcTile) + i / kFcTile) * (size_t)(C + 1) * kFcTile + i % kFcTile;
            for (int k = 0; k < C; ++k) dst[(size_t)k * kFcTile] = live ? own[k * osc] : 0.f;
            dst[(size_t)C * kFcTile] = n;
        }
    }
}

// Register blocking: a warp owns 8 query rows, a lane 4 consecutive candidates of the 128-wide
// stage -> 32 accumulators per lane held as 16 packed pairs; per channel 2 broadcast LDS.128
// (8 query values) + 1 LDS.128 (4 candidates) feed 16 FFMA2 (the 4 x 2 blocking it replaces fed
// 8 FFMA from 3 LDS and ran at 28 % of the FMA peak).  Every pair is still the sequential fp32
// chain fmul, fma, fma, ... over the channels (packed halves round independently), then the two
// norm additions in the order of `form`: bit-identical to the oracle.
// Candidate stages (C channel rows of 512 B + the norms, contiguous in the workspace) arrive by
// one 1-D TMA bulk copy each behind an mbarrier, double buffered.  A row's four candidates are
// tested against its threshold with ONE vote per row, all eight votes issued before the first
// branch, so the common "nothing passes" case is a short branch-free sequence.

static inline size_t knnc_smem_bytes(int C) {
    return 128 + (size_t)C * kFcCtaRows * 4 + 2 * ((size_t)C * kFcTile + kFcTile) * 4 +
           (size_t)kFcCtaRows * kFcStage * 8;
}

template <int NL>
__global__ void __launch_bounds__(kKnnThreads)
knnc_kernel(const float *__restrict__ rowT, const float *__restrict__ rown, const float *__restrict__ colS,
            int N, int M, int C, int Npad, int Mpad, int K, int form,
            float *__restrict__ dists, int32_t *__restrict__ idx) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    // layout: full[2], empty[2] | qs[C][64] | ct[2][C*128 + 128] | stage[64 rows][63] u64
    uint64_t *full = reinterpret_cast<uint64_t *>(smem_raw);
    uint64_t *empty = full + 2;                  // one arrival per warp when it has finished reading a stage
    float *qs = reinterpret_cast<float *>(smem_raw + 128);
    float *ct = qs + (size_t)C * kFcCtaRows;
    const size_t ct_stride = (size_t)C * kFcTile + kFcTile;
    unsigned long long *stage = reinterpret_cast<unsigned long long *>(ct + 2 * ct_stride);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.y;
    const int cta_row0 = blockIdx.x * kFcCtaRows;
    const int row0 = cta_row0 + warp * kFcRows;
    const int ntiles = (M + kFcTile - 1) / kFcTile;
    const float *cbase = colS + (size_t)b * (Mpad / kFcTile) * ct_stride;
    const uint32_t stage_bytes = (uint32_t)ct_stride * 4u;

    auto issue = [&](int t) {                    // one thread
        const int buf = t & 1;
        mbar_expect_tx(&full[buf], stage_bytes);
        tma_load_1d(ct + buf * ct_stride, cbase + (size_t)t * ct_stride, stage_bytes, &full[buf]);
    };
    if (tid == 0) {
        mbar_init(&full[0], 1);
        mbar_init(&full[1], 1);
        mbar_init(&empty[0], kKnnWarps);
        mbar_init(&empty[1], kKnnWarps);
        fence_mbar_init();
        fence_proxy_async();
    }
    __syncthreads();
    if (tid == 0) {
        issue(0);
        if (ntiles > 1) issue(1);
    }
    // the CTA's query rows, channel-major: qs[k][r]
    for (int e = tid; e < C * kFcCtaRows; e += kKnnThreads) {
        const int k = e / kFcCtaRows, r = e - k * kFcCtaRows;
        qs[e] = rowT[((size_t)b * C + k) * Npad + cta_row0 + r];
    }
    float qn[kFcRows];
    RowSelect<NL> sel[kFcRows];
#pragma unroll
    for (int r = 0; r < kFcRows; ++r) {
        qn[r] = rown[(size_t)b * Npad + row0 + r];
        sel[r].init();
    }
    unsigned long long *mystage = stage + (size_t)warp * kFcRows * kFcStage;
    __syncthreads();

    const float4 *q4 = reinterpret_cast<const float4 *>(qs) + warp * 2;          // + k * 16
    for (int t = 0; t < ntiles; ++t) {
        const int buf = t & 1;
        // No CTA barrier in the loop: the warps drift apart by up to one stage.  The producer
        // refills the stage of tile t-1 with tile t+1 once all eight warps have released it.
        if (tid == 0 && t >= 1 && t + 1 < ntiles) {
            mbar_wait(&empty[buf ^ 1], ((t - 1) >> 1) & 1);
            fence_proxy_async();
            issue(t + 1);
        }
        mbar_wait(&full[buf], (t >> 1) & 1);
        const float *tile = ct + buf * ct_stride;
        const float4 *c4p = reinterpret_cast<const float4 *>(tile) + lane;       // + k * 32
        f32x2 acc[kFcRows][2];
        {
            const float4 qa = q4[0], qb = q4[1], c = c4p[0];
            const f32x2 c01 = pack2(c.x, c.y), c23 = pack2(c.z, c.w);
            const float q[kFcRows] = {qa.x, qa.y, qa.z, qa.w, qb.x, qb.y, qb.z, qb.w};
#pragma unroll
            for (int r = 0; r < kFcRows; ++r) { acc[r][0] = mul2_s(q[r], c01); acc[r][1] = mul2_s(q[r], c23); }
        }
#pragma unroll 4
        for (int k = 1; k < C; ++k) {
            const float4 qa = q4[k * 16], qb = q4[k * 16 + 1], c = c4p[k * 32];
            const f32x2 c01 = pack2(c.x, c.y), c23 = pack2(c.z, c.w);
            const float q[kFcRows] = {qa.x, qa.y, qa.z, qa.w, qb.x, qb.y, qb.z, qb.w};
#pragma unroll
            for (int r = 0; r < kFcRows; ++r) { acc[r][0] = fma2_s(q[r], c01, acc[r][0]); acc[r][1] = fma2_s(q[r], c23, acc[r][1]); }
        }
        const float4 n4 = reinterpret_cast<const float4 *>(tile + (size_t)C * kFcTile)[lane];
        const f32x2 n01 = pack2(n4.x, n4.y), n23 = pack2(n4.z, n4.w);
        const int j = t * kFcTile + lane * 4;
        float d[kFcRows][4];
        unsigned hit[kFcRows];
#pragma unroll
        for (int r = 0; r < kFcRows; ++r) {
            f32x2 d01, d23;
            if (form == PCD_FORM_ROW_COL) {
                d01 = add2(add2_s(qn[r], acc[r][0]), n01); d23 = add2(add2_s(qn[r], acc[r][1]), n23);
            } else if (form == PCD_FORM_COL_ROW) {
                d01 = add2_s(qn[r], add2(acc[r][0], n01)); d23 = add2_s(qn[r], add2(acc[r][1], n23));
            } else {
                d01 = add2(add2_s(qn[r], n01), acc[r][0]); d23 = add2(add2_s(qn[r], n23), acc[r][1]);
            }
            unpack2(d01, d[r][0], d[r][1]); unpack2(d23, d[r][2], d[r][3]);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[buf]);  // this warp is done with the stage (distances are in registers)
        if (NL == 1 && t == 0) {
            // First stage: instead of staging all 128 candidates against thr = +inf (four sort +
            // merge rounds per row), start from a cheap exact upper bound of the K-th distance:
            // the K-th smallest of the 32 lane minima (32 distinct candidates; K <= 32 here).
#pragma unroll
            for (int r = 0; r < kFcRows; ++r) {
                sel[r].st.thr = warp_kth_bound(fminf(min3(d[r][0], d[r][1], d[r][2]), d[r][3]), lane, K);
            }
        }
#pragma unroll
        for (int r = 0; r < kFcRows; ++r) {
            const float thr = sel[r].st.thr;
            hit[r] = __ballot_sync(0xffffffffu, (d[r][0] < thr) | (d[r][1] < thr) | (d[r][2] < thr) | (d[r][3] < thr));
        }
#pragma unroll
        for (int r = 0; r < kFcRows; ++r) {
            if (hit[r]) sel[r].offer4(d[r], j, mystage + r * kFcStage, lane, K);
        }
    }
#pragma unroll
    for (int r = 0; r < kFcRows; ++r) {
        sel[r].finish(mystage + r * kFcStage, lane, K);
        const int i = row0 + r;
        if (i < N) sel[r].store(dists, idx, ((size_t)b * N + i) * K, lane, K);
    }
}

// ------------------------------------------------------------------------ k-NN backward
// dists[b,i,k] = d(i, j=idx[b,i,k]) ; own-index terms with plain stores, partner terms with
// atomics (same two-pass scheme as the NN-1 backward).
struct KnnBwdArgs {
    const float *rows; int64_t r_sb, r_sp, r_sc;
    const float *cols; int64_t c_sb, c_sp, c_sc;
    int B, N, M, K, swap_norms;
    const int32_t *idx; const float *g;
    float *grad_rows; int64_t gr_sb, gr_sp, gr_sc;
    float *grad_cols; int64_t gc_sb, gc_sp, gc_sc;
};

template <bool SCATTER>
__global__ void __launch_bounds__(256) knn_bwd_kernel(KnnBwdArgs a) {
    const long long total = (long long)a.B * (a.N + a.M);
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const int b = (int)(t / (a.N + a.M));
        const int p = (int)(t - (long long)b * (a.N + a.M));
        const float *rb = a.rows + b * a.r_sb, *cb = a.cols + b * a.c_sb;
        if (p < a.N) {
            const int i = p;
            const float rx = rb[i * a.r_sp], ry = rb[i * a.r_sp + a.r_sc], rz = rb[i * a.r_sp + 2 * a.r_sc];
            float ox = 0.f, oy = 0.f, oz = 0.f, gsum = 0.f;
            for (int k = 0; k < a.K; ++k) {
                const size_t e = ((size_t)b * a.N + i) * a.K + k;
                const float g2 = 2.f * a.g[e];
                const int j = a.idx[e];
                const float cx = cb[j * a.c_sp], cy = cb[j * a.c_sp + a.c_sc], cz = cb[j * a.c_sp + 2 * a.c_sc];
                gsum += g2;
                if (!SCATTER) {
                    if (a.swap_norms) { ox -= g2 * cx; oy -= g2 * cy; oz -= g2 * cz; }
                    else { ox += g2 * (rx - cx); oy += g2 * (ry - cy); oz += g2 * (rz - cz); }
                } else if (g2 != 0.f) {
                    if (a.grad_cols) {
                        float *gp = a.grad_cols + b * a.gc_sb + j * a.gc_sp;
                        if (a.swap_norms) {
                            atomicAdd(gp, -g2 * rx); atomicAdd(gp + a.gc_sc, -g2 * ry); atomicAdd(gp + 2 * a.gc_sc, -g2 * rz);
                        } else {
                            atomicAdd(gp, -g2 * (rx - cx)); atomicAdd(gp + a.gc_sc, -g2 * (ry - cy));
                            atomicAdd(gp + 2 * a.gc_sc, -g2 * (rz - cz));
                        }
                    }
                    if (a.swap_norms && a.grad_rows) {   // |rows_j|^2 term
                        const float jx = rb[j * a.r_sp], jy = rb[j * a.r_sp + a.r_sc], jz = rb[j * a.r_sp + 2 * a.r_sc];
                        float *gp = a.grad_rows + b * a.gr_sb + j * a.gr_sp;
                        atomicAdd(gp, g2 * jx); atomicAdd(gp + a.gr_sc, g2 * jy); atomicAdd(gp + 2 * a.gr_sc, g2 * jz);
                    }
                }
            }
            if (!SCATTER && a.grad_rows) {
                float *gp = a.grad_rows + b * a.gr_sb + i * a.gr_sp;
                gp[0] = ox; gp[a.gr_sc] = oy; gp[2 * a.gr_sc] = oz;
            }
        } else if (!SCATTER && a.grad_cols) {
            // own-index term of a column point: only the swapped-norm |cols_i|^2 term (N == M)
            const int j = p - a.N;
            float ox = 0.f, oy = 0.f, oz = 0.f;
            if (a.swap_norms) {
                float gsum = 0.f;
                for (int k = 0; k < a.K; ++k) gsum += 2.f * a.g[((size_t)b * a.N + j) * a.K + k];
                ox = gsum * cb[j * a.c_sp]; oy = gsum * cb[j * a.c_sp + a.c_sc]; oz = gsum * cb[j * a.c_sp + 2 * a.c_sc];
            }
            float *gp = a.grad_cols + b * a.gc_sb + j * a.gc_sp;
            gp[0] = ox; gp[a.gc_sc] = oy; gp[2 * a.gc_sc] = oz;
        }
    }
}

// ------------------------------------------------------------------------------ ball query
// One warp per query row; lanes sweep 32 columns per step in ascending index order and
// ballot-compact the hits, so the output is already ordered and the sweep stops as soon as
// nsample hits are found (the reference sorts all N indices per row instead).
__global__ void __launch_bounds__(256)
ball_query_kernel(const float *__restrict__ xyz, int64_t x_sb, int64_t x_sp, int64_t x_sc,
                  const float *__restrict__ qry, int64_t q_sb, int64_t q_sp, int64_t q_sc,
                  int B, int N, int S, float r2, int nsample, int32_t *__restrict__ idx) {
    const int lane = threadIdx.x & 31;
    const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < (long long)B * S; w += warps) {
        const int b = (int)(w / S), i = (int)(w - (long long)b * S);
        const float *qp = qry + b * q_sb + i * q_sp;
        const float qx = qp[0], qy = qp[q_sc], qz = qp[2 * q_sc];
        const float qn = sq_norm3(PCD_NORM_MULSUM, qx, qy, qz);
        const float mx = -2.f * qx, my = -2.f * qy, mz = -2.f * qz;
        int32_t *out = idx + ((size_t)b * S + i) * nsample;
        int cnt = 0, first = N;
        for (int j0 = 0; j0 < N && cnt < nsample; j0 += 32) {
            const int j = j0 + lane;
            bool hit = false;
            if (j < N) {
                const float *cp = xyz + b * x_sb + j * x_sp;
                const float cx = cp[0], cy = cp[x_sc], cz = cp[2 * x_sc];
                const float d = pair_dist_scalar<PCD_FORM_ROW_COL>(mx, my, mz, qn, cx, cy, cz,
                                                                   sq_norm3(PCD_NORM_MULSUM, cx, cy, cz));
                hit = !(d > r2);
            }
            const unsigned mask = __ballot_sync(0xffffffffu, hit);
            if (mask) {
                if (cnt == 0) first = j0 + __ffs(mask) - 1;
                const int pos = cnt + __popc(mask & ((1u << lane) - 1u));
                if (hit && pos < nsample) out[pos] = j;
                cnt += __popc(mask);
            }
        }
        for (int s = (cnt < nsample ? cnt : nsample) + lane; s < nsample; s += 32) out[s] = first;
    }
}

struct KnnLayout {
    int Npad, Mpad;
    size_t a, b, c, d, e, total;   // xyz: a=rowq b=colq c=colpk d=cm e=thr0 ; features: a=rowT b=rown c=colS
    // xyz pre-pass + collect plan
    bool prepass;
    int W, G, nsplit, tps, caps;
    size_t cand, cnt, ovf_cnt, ovf_rows;
};
constexpr int kPlanSMs = 148;     // B200; the plan must not depend on a device query (workspace sizes are host-only)

static KnnLayout knn_layout(int B, int N, int M, int C, int K) {
    KnnLayout L;
    L.prepass = false;
    L.W = L.G = L.nsplit = L.tps = L.caps = 0;
    L.cand = L.cnt = L.ovf_cnt = L.ovf_rows = 0;
    size_t off = 0;
    L.e = 0;
    if (C == 3) {
        // pre-pass: chunk width W so that 3K <= G <= 64 chunks where possible; skipped when M is too small
        int W = (M / (3 * (K > 0 ? K : 1))) & ~1;
        const int wmin = ((M + kPreMaxChunks - 1) / kPreMaxChunks + 1) & ~1;
        if (W < wmin) W = wmin;
        if (W < 2) W = 2;
        L.W = W;
        L.G = (M + W - 1) / W;
        L.prepass = K >= 1 && L.G >= K && L.G <= kPreMaxChunks && M >= 256;
        // rows-in-lanes passes want 512-row tiles; the warp-per-row select alone only 32 (small clouds, big batches)
        L.Npad = (int)align_up_k((size_t)N, L.prepass ? 128 * kPreR : kKnnWarps * kKnnRQ);
        L.Mpad = (int)align_up_k((size_t)M, kKnnTile);
        L.a = off; off = align_up_k(off + (size_t)B * L.Npad * 16, 256);
        L.b = off; off = align_up_k(off + (size_t)B * L.Mpad * 16, 256);
        L.c = off; off = align_up_k(off + (size_t)B * L.Mpad * 16 + kPreTile * 16, 256);   // + one stage of slack (chunk-aligned stages)
        L.d = off;
        if (L.prepass) off = align_up_k(off + (size_t)B * L.G * L.Npad * 4, 256);            // chunk minima [B][G][Npad]
        L.e = off; off = align_up_k(off + (size_t)B * L.Npad * 4, 256);
        if (L.prepass) {
            // collect pass: split the column stages of a row tile over nsplit CTAs until the grid fills the GPU
            const int ntiles = (M + kPreTile - 1) / kPreTile;
            const long long base = (long long)B * (L.Npad / (128 * kPreR));
            // (>= 4 full waves of 8 resident CTAs per SM, or one stage per CTA)
            long long want = ((long long)kPlanSMs * 8 * 4 + base - 1) / base;
            if (want < 1) want = 1;
            if (want > 16) want = 16;
            if (want > ntiles) want = ntiles;
            L.tps = (ntiles + (int)want - 1) / (int)want;
            L.nsplit = (ntiles + L.tps - 1) / L.tps;
            L.caps = (2 * K + L.nsplit - 1) / L.nsplit + 12;           // expected ~1.2 K / nsplit candidates per list
            L.cand = off; off = align_up_k(off + (size_t)L.nsplit * B * L.caps * L.Npad * 8, 256);
            L.cnt = off; off = align_up_k(off + (size_t)L.nsplit * B * L.Npad * 4, 256);
            L.ovf_cnt = off; off = align_up_k(off + (size_t)B * 4, 256);
            L.ovf_rows = off; off = align_up_k(off + (size_t)B * L.Npad * 4, 256);
        }
    } else {
        L.Npad = (int)align_up_k((size_t)N, kFcCtaRows);
        L.Mpad = (int)align_up_k((size_t)M, kFcTile);
        L.a = off; off = align_up_k(off + (size_t)B * L.Npad * C * 4, 256);
        L.b = off; off = align_up_k(off + (size_t)B * L.Npad * 4, 256);
        L.c = off; off = align_up_k(off + (size_t)B * L.Mpad * (C + 1) * 4, 256);
        L.d = off;
    }
    L.total = off;
    return L;
}

}  // namespace pcd

using namespace pcd;

extern "C" size_t pcd_knn_workspace_bytes(int B, int N, int M, int C, int K) {
    if (B <= 0 || N <= 0 || M <= 0 || C <= 0) return 0;
    return knn_layout(B, N, M, C, K).total;
}

extern "C" int pcd_knn_forward(const float *rows, int64_t r_sb, int64_t r_sp, int64_t r_sc,
                               const float *cols, int64_t c_sb, int64_t c_sp, int64_t c_sc,
                               int B, int N, int M, int C, int K, int form, int norm_kind, int swap_norms,
                               float *dists, int32_t *idx, void *workspace, size_t workspace_bytes, int strategy, void *stream) {
    if (!rows || !cols || !idx || !workspace) {
        set_error("pcd_knn_forward: NULL pointer argument");
        return PCD_ERR_ARG;
    }
    if (B <= 0 || N <= 0 || M <= 0 || form < 0 || form > 2 || norm_kind < 0 || norm_kind > 1 || B > 65535) {
        set_error("pcd_knn_forward: bad argument B=%d N=%d M=%d form=%d norm=%d", B, N, M, form, norm_kind);
        return PCD_ERR_ARG;
    }
    if (K < 1 || K > M || K > PCD_KNN_MAX_K || C < 1 || C > PCD_KNN_MAX_C) {
        set_error("pcd_knn_forward: unsupported K=%d (1..min(M,%d)) or C=%d (1..%d)", K, PCD_KNN_MAX_K, C, PCD_KNN_MAX_C);
        return PCD_ERR_UNSUPPORTED;
    }
    if (swap_norms && N != M) {
        set_error("pcd_knn_forward: swap_norms requires N == M");
        return PCD_ERR_ARG;
    }
    const KnnLayout L = knn_layout(B, N, M, C, K);
    if (workspace_bytes < L.total) {
        set_error("pcd_knn_forward: workspace %zu < required %zu bytes", workspace_bytes, L.total);
        return PCD_ERR_WORKSPACE;
    }
    const int sms = num_sms();
    if (sms <= 0) return cuda_fail(cudaGetLastError(), "no CUDA device");
    cudaStream_t st = (cudaStream_t)stream;
    char *ws = (char *)workspace;
    const int pgrid = capped_grid((long long)B * (L.Npad + L.Mpad), 256, (long long)sms * 8);
    const dim3 grid(L.Npad / (kKnnWarps * kKnnRQ), B);
    const int NL = (K + 31) / 32;
    if (C == 3) {
        float4 *rowq = (float4 *)(ws + L.a), *colq = (float4 *)(ws + L.b);
        float *colpk = (float *)(ws + L.c), *cm = (float *)(ws + L.d), *thr0 = (float *)(ws + L.e);
        knn3_prep_kernel<<<pgrid, 256, 0, st>>>(rows, r_sb, r_sp, r_sc, cols, c_sb, c_sp, c_sc, B, N, M, L.Npad, L.Mpad,
                                                norm_kind, swap_norms, rowq, colq, colpk,
                                                L.prepass ? (int *)(ws + L.ovf_cnt) : nullptr);
        PCD_CUDA_CHECK(cudaGetLastError());
        // strategy (per call; the library reads no environment): 0 = chunk-minima bound + collect + final,
        // 1 = bound + warp-per-row select (no collect pass), 2 = warp-per-row select alone.  Same results.
        const bool prepass = L.prepass && strategy != PCD_KNN_SELECT_ONLY;
        const bool collect = prepass && strategy != PCD_KNN_BOUND_SELECT;
        int *ovf_cnt = (int *)(ws + L.ovf_cnt), *ovf_rows = (int *)(ws + L.ovf_rows);
        if (prepass) {
            const int W = L.W, G = L.G;
            // column splits at chunk granularity until the grid holds >= 4 waves of 8 CTAs per SM
            const long long base = (long long)B * (L.Npad / (128 * kPreR));
            long long csplit = ((long long)sms * 32 + base - 1) / base;
            const int max_split = (M + 2 * kPreTile - 1) / (2 * kPreTile);        // at least two stages per split
            if (csplit > max_split) csplit = max_split;
            if (csplit > G) csplit = G;
            if (csplit < 1) csplit = 1;
            const int cps = (G + (int)csplit - 1) / (int)csplit;
            const dim3 pg(L.Npad / (128 * kPreR), B, (G + cps - 1) / cps);
            with_form(form, [&](auto F) { knn3_chunkmin_kernel<F><<<pg, 128, 0, st>>>(rowq, (const float4 *)colpk, L.Npad, L.Mpad, M, W, G, cps, cm); });
            PCD_CUDA_CHECK(cudaGetLastError());
            if (G <= 32) knn_threshold_kernel<32><<<dim3(L.Npad / 128, B), 128, 0, st>>>(cm, L.Npad, G, K, thr0);
            else knn_threshold_kernel<64><<<dim3(L.Npad / 128, B), 128, 0, st>>>(cm, L.Npad, G, K, thr0);
            PCD_CUDA_CHECK(cudaGetLastError());
        }
        const float *thr_arg = prepass ? thr0 : nullptr;
        // warp-per-row select: of every row, or of the rows listed in (ovf_cnt, ovf_rows)
        const auto launch_select = [&](const int *oc, const int *orows) {
            with_form(form, [&](auto F) {
                if (NL == 1) knn3_kernel<F, 1><<<grid, kKnnThreads, 0, st>>>(rowq, colq, thr_arg, N, M, L.Npad, L.Mpad, K, dists, idx, oc, orows);
                else knn3_kernel<F, 2><<<grid, kKnnThreads, 0, st>>>(rowq, colq, thr_arg, N, M, L.Npad, L.Mpad, K, dists, idx, oc, orows);
            });
        };
        if (collect) {
            unsigned long long *cand = (unsigned long long *)(ws + L.cand);
            unsigned int *cnt_g = (unsigned int *)(ws + L.cnt);
            const dim3 cg((L.Npad / (128 * kPreR)) * L.nsplit, B);
            with_form(form, [&](auto F) {
                knn3_collect_kernel<F><<<cg, 128, 0, st>>>(rowq, (const float4 *)colpk, thr0, B, L.Npad, L.Mpad, M, L.nsplit, L.tps, L.caps, cand, cnt_g);
            });
            PCD_CUDA_CHECK(cudaGetLastError());
            const dim3 fg((N + 127) / 128, B);
            const auto launch_final = [&](auto KT) {
                knn3_final_kernel<KT><<<fg, 128, (size_t)128 * K * sizeof(uint32_t), st>>>(cand, cnt_g, B, N, L.Npad, L.nsplit, L.caps, K,
                                                                                            dists, idx, ovf_cnt, ovf_rows);
            };
            switch ((K + 3) / 4) {                           // KT = K rounded up to a multiple of 4 (48 / 64 beyond 32)
                case 1: launch_final(IntC<4>{}); break;
                case 2: launch_final(IntC<8>{}); break;
                case 3: launch_final(IntC<12>{}); break;
                case 4: launch_final(IntC<16>{}); break;
                case 5: launch_final(IntC<20>{}); break;
                case 6: launch_final(IntC<24>{}); break;
                case 7: launch_final(IntC<28>{}); break;
                case 8: launch_final(IntC<32>{}); break;
                default: if (K <= 48) launch_final(IntC<48>{}); else launch_final(IntC<64>{}); break;
            }
            PCD_CUDA_CHECK(cudaGetLastError());
            // rows whose candidate lists overflowed (none for randomly ordered clouds): warp-per-row select
            launch_select(ovf_cnt, ovf_rows);
        } else {
            launch_select(nullptr, nullptr);
        }
        PCD_CUDA_CHECK(cudaGetLastError());
    } else {
        float *rowf = (float *)(ws + L.a), *rown = (float *)(ws + L.b);
        float *colS = (float *)(ws + L.c);
        knnc_prep_kernel<<<pgrid, 256, 0, st>>>(rows, r_sb, r_sp, r_sc, cols, c_sb, c_sp, c_sc, B, N, M, C, L.Npad,
                                                L.Mpad, norm_kind, swap_norms, rowf, rown, colS);
        PCD_CUDA_CHECK(cudaGetLastError());
        const size_t smem = knnc_smem_bytes(C);
        const dim3 fgrid(L.Npad / kFcCtaRows, B);
        const auto kernel = NL == 1 ? knnc_kernel<1> : knnc_kernel<2>;
        PCD_CUDA_CHECK(opt_in_smem(kernel, smem));
        kernel<<<fgrid, kKnnThreads, smem, st>>>(rowf, rown, colS, N, M, C, L.Npad, L.Mpad, K, form, dists, idx);
        PCD_CUDA_CHECK(cudaGetLastError());
    }
    return PCD_OK;
}

extern "C" int pcd_knn_backward(const float *rows, int64_t r_sb, int64_t r_sp, int64_t r_sc,
                                const float *cols, int64_t c_sb, int64_t c_sp, int64_t c_sc,
                                int B, int N, int M, int K, int swap_norms, const int32_t *idx, const float *g_dists,
                                float *grad_rows, int64_t gr_sb, int64_t gr_sp, int64_t gr_sc,
                                float *grad_cols, int64_t gc_sb, int64_t gc_sp, int64_t gc_sc, void *stream) {
    if (!rows || !cols || !idx || !g_dists || B <= 0 || N <= 0 || M <= 0 || K <= 0) {
        set_error("pcd_knn_backward: bad argument");
        return PCD_ERR_ARG;
    }
    if (swap_norms && N != M) {
        set_error("pcd_knn_backward: swap_norms requires N == M");
        return PCD_ERR_ARG;
    }
    if (!grad_rows && !grad_cols) return PCD_OK;
    const int sms = num_sms();
    if (sms <= 0) return cuda_fail(cudaGetLastError(), "no CUDA device");
    KnnBwdArgs a{rows, r_sb, r_sp, r_sc, cols, c_sb, c_sp, c_sc, B, N, M, K, swap_norms, idx, g_dists,
                 grad_rows, gr_sb, gr_sp, gr_sc, grad_cols, gc_sb, gc_sp, gc_sc};
    const int grid = capped_grid((long long)B * (N + M), 256, (long long)sms * 16);
    cudaStream_t st = (cudaStream_t)stream;
    knn_bwd_kernel<false><<<grid, 256, 0, st>>>(a);
    PCD_CUDA_CHECK(cudaGetLastError());
    knn_bwd_kernel<true><<<grid, 256, 0, st>>>(a);
    PCD_CUDA_CHECK(cudaGetLastError());
    return PCD_OK;
}

extern "C" int pcd_ball_query(const float *xyz, int64_t x_sb, int64_t x_sp, int64_t x_sc,
                              const float *new_xyz, int64_t q_sb, int64_t q_sp, int64_t q_sc,
                              int B, int N, int S, float radius2, int nsample, int32_t *idx, void *stream) {
    if (!xyz || !new_xyz || !idx || B <= 0 || N <= 0 || S <= 0 || nsample <= 0) {
        set_error("pcd_ball_query: bad argument");
        return PCD_ERR_ARG;
    }
    const int sms = num_sms();
    if (sms <= 0) return cuda_fail(cudaGetLastError(), "no CUDA device");
    const int grid = capped_grid((long long)B * S, 8, (long long)sms * 8);     // a warp per query row
    ball_query_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(xyz, x_sb, x_sp, x_sc, new_xyz, q_sb, q_sp, q_sc, B, N, S,
                                                             radius2, nsample, idx);
    PCD_CUDA_CHECK(cudaGetLastError());
    return PCD_OK;
}
