// pcd_common.cuh -- shared device helpers for the sm_100a point-set distance kernels.
//
// The one rule every kernel here obeys: a pair distance is ALWAYS evaluated with the same
// fp32 instruction sequence (pair_dist_scalar / pair_dist_x2 below), so a value recomputed in
// the fix-up, k-NN or ball-query kernels is bit-identical to the one the sweep saw.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "../../include/pcdist.h"

namespace pcd {

// ----------------------------------------------------------------------------- error state
void set_error(const char *fmt, ...);
int cuda_fail(cudaError_t e, const char *what);
#define PCD_CUDA_CHECK(expr)                                              \
    do {                                                                  \
        cudaError_t _e = (expr);                                          \
        if (_e != cudaSuccess) return ::pcd::cuda_fail(_e, #expr);        \
    } while (0)

// ------------------------------------------------------------------- packed fp32x2 (Blackwell)
// sm_100 executes two IEEE fp32 FMAs per lane in one FFMA2/FADD2/FMUL2 issue slot; each half
// rounds independently (RN), so results equal the scalar ops bit for bit.  A {s,s} pack folds
// into a scalar-broadcast operand (Rn.F32) in SASS, so query coordinates cost one register.
typedef unsigned long long f32x2;

__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
    f32x2 d;
    asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "f"(lo), "f"(hi));
    return d;
}
__device__ __forceinline__ f32x2 bcast2(float s) { return pack2(s, s); }
__device__ __forceinline__ void unpack2(f32x2 v, float &lo, float &hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
    f32x2 d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
    f32x2 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
    f32x2 d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
// scalar-broadcast variants: the {s,s} pack lives inside the asm block so that it cannot be
// hoisted into a loop-invariant register PAIR; ptxas folds it into the Rn.F32 operand form.
__device__ __forceinline__ f32x2 mul2_s(float s, f32x2 b) {
    f32x2 d;
    asm("{\n.reg .b64 q;\nmov.b64 q, {%1, %1};\nmul.rn.f32x2 %0, q, %2;\n}" : "=l"(d) : "f"(s), "l"(b));
    return d;
}
__device__ __forceinline__ f32x2 fma2_s(float s, f32x2 b, f32x2 c) {
    f32x2 d;
    asm("{\n.reg .b64 q;\nmov.b64 q, {%1, %1};\nfma.rn.f32x2 %0, q, %2, %3;\n}" : "=l"(d) : "f"(s), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ f32x2 add2_s(float s, f32x2 b) {
    f32x2 d;
    asm("{\n.reg .b64 q;\nmov.b64 q, {%1, %1};\nadd.rn.f32x2 %0, q, %2;\n}" : "=l"(d) : "f"(s), "l"(b));
    return d;
}
// three-input min (FMNMX3, sm_100)
__device__ __forceinline__ float min3(float a, float b, float c) {
    float d;
    asm("min.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}
// warp-wide fp32 min in one instruction (CREDUX.MIN.F32, sm_100a)
__device__ __forceinline__ float warp_min_f32(float v) {
    float d;
    asm volatile("redux.sync.min.f32 %0, %1, 0xffffffff;" : "=f"(d) : "f"(v));
    return d;
}

// ------------------------------------------------------------------------ pair arithmetic
// Query side carries (x', y', z', n) with x' = -2x (exact), column side (x, y, z, n).
template <int FORM>
__device__ __forceinline__ float pair_dist_scalar(float qx, float qy, float qz, float qn,
                                                  float cx, float cy, float cz, float cn) {
    float t = __fmul_rn(qx, cx);
    t = __fmaf_rn(qy, cy, t);
    t = __fmaf_rn(qz, cz, t);
    if (FORM == PCD_FORM_ROW_COL) return __fadd_rn(__fadd_rn(t, qn), cn);
    if (FORM == PCD_FORM_COL_ROW) return __fadd_rn(__fadd_rn(t, cn), qn);
    return __fadd_rn(__fadd_rn(qn, cn), t);
}
template <int FORM>
__device__ __forceinline__ f32x2 pair_dist_x2(float qx, float qy, float qz, float qn,
                                              f32x2 cx, f32x2 cy, f32x2 cz, f32x2 cn) {
    f32x2 t = mul2_s(qx, cx);
    t = fma2_s(qy, cy, t);
    t = fma2_s(qz, cz, t);
    if (FORM == PCD_FORM_ROW_COL) return add2(add2_s(qn, t), cn);
    if (FORM == PCD_FORM_COL_ROW) return add2_s(qn, add2(t, cn));
    return add2(add2_s(qn, cn), t);
}
__device__ __forceinline__ float pair_dist_dyn(int form, float qx, float qy, float qz, float qn,
                                               float cx, float cy, float cz, float cn) {
    if (form == PCD_FORM_ROW_COL) return pair_dist_scalar<PCD_FORM_ROW_COL>(qx, qy, qz, qn, cx, cy, cz, cn);
    if (form == PCD_FORM_COL_ROW) return pair_dist_scalar<PCD_FORM_COL_ROW>(qx, qy, qz, qn, cx, cy, cz, cn);
    return pair_dist_scalar<PCD_FORM_SUM_FIRST>(qx, qy, qz, qn, cx, cy, cz, cn);
}

// |p|^2 of two points at once, same roundings as sq_norm3.  The mul-then-add form is evaluated with the scalar
// round-to-nearest intrinsics: ptxas CONTRACTS mul.rn.f32x2 + add.rn.f32x2 into FFMA2 (observed with CUDA 12.9, --fmad=false
// notwithstanding), which would change the rounding of (x*x + y*y) + z*z; __fmul_rn / __fadd_rn are never fused.
__device__ __forceinline__ f32x2 sq_norm3_x2(int kind, f32x2 x, f32x2 y, f32x2 z) {
    if (kind == PCD_NORM_FMA) return fma2(z, z, fma2(y, y, mul2(x, x)));
    float x0, x1, y0, y1, z0, z1;
    unpack2(x, x0, x1); unpack2(y, y0, y1); unpack2(z, z0, z1);
    return pack2(__fadd_rn(__fadd_rn(__fmul_rn(x0, x0), __fmul_rn(y0, y0)), __fmul_rn(z0, z0)),
                 __fadd_rn(__fadd_rn(__fmul_rn(x1, x1), __fmul_rn(y1, y1)), __fmul_rn(z1, z1)));
}
// Two distances between ONE fixed point f (coordinates fx, fy, fz, norm fn) and two candidates (packed coordinates X, Y, Z,
// norms NN).  `row_is_fixed` says which side the fixed point is on; the factor -2 of the row operand is exact, so it is
// applied to the fixed scalars either way: fl((-2 r).c) == fl(r.(-2 c)).  m2x etc. = -2 * the fixed coordinates.
template <int FORM>
__device__ __forceinline__ f32x2 pair_dist_fixed_x2(bool row_is_fixed, float m2x, float m2y, float m2z, float fn,
                                                    f32x2 X, f32x2 Y, f32x2 Z, f32x2 NN) {
    f32x2 t = mul2_s(m2x, X);
    t = fma2_s(m2y, Y, t);
    t = fma2_s(m2z, Z, t);
    // nrow / ncol: the fixed point's norm is the row norm when row_is_fixed, else the column norm
    if (FORM == PCD_FORM_SUM_FIRST) return add2(add2_s(fn, NN), t);                               // (nrow + ncol) + t
    if (FORM == PCD_FORM_ROW_COL) return row_is_fixed ? add2(add2_s(fn, t), NN) : add2_s(fn, add2(t, NN));   // (t + nrow) + ncol
    return row_is_fixed ? add2_s(fn, add2(t, NN)) : add2(add2_s(fn, t), NN);                       // (t + ncol) + nrow
}

__device__ __forceinline__ float sq_norm3(int kind, float x, float y, float z) {
    if (kind == PCD_NORM_FMA) return __fmaf_rn(z, z, __fmaf_rn(y, y, __fmul_rn(x, x)));
    return __fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z));
}

// --------------------------------------------------------------------------- ordered keys
// Monotone map fp32 -> u32 so that (value, index) pairs can be min-reduced with one u64
// atomicMin: lower value first, then lower index.  -0.0 is canonicalised to +0.0 first.
__device__ __forceinline__ uint32_t f32_to_ordered(float f) {
    uint32_t u = __float_as_uint(__fadd_rn(f, 0.0f));
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ordered_to_f32(uint32_t o) {
    return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}
__device__ __forceinline__ unsigned long long make_key(float v, uint32_t tag) {
    return ((unsigned long long)f32_to_ordered(v) << 32) | tag;
}

// ------------------------------------------------------------- TMA bulk copy + mbarrier
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}
// 1-D bulk async copy global -> shared (SASS: UBLKCP), completion on an mbarrier.
__device__ __forceinline__ void tma_load_1d(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(smem_dst)),
        "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// ------------------------------------------------------------------- block-wide reduction
// Sum over a block of THREADS threads (a multiple of 32) in a fixed order: an xor butterfly per warp, then one over the
// warp totals.  sh holds THREADS / 32 values.  Every thread gets the total.
template <typename T, int THREADS>
__device__ __forceinline__ T block_sum(T v, T *sh) {
    static_assert(THREADS % 32 == 0 && THREADS <= 1024, "block_sum: whole warps, at most 32");
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();                   // sh may still be read from the previous call
    if (lane == 0) sh[warp] = v;
    __syncthreads();
    T t = lane < THREADS / 32 ? sh[lane] : T(0);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    return t;
}

// ------------------------------------------------- programmatic dependent launch (sm_90+)
// A kernel launched with the programmatic-stream-serialization attribute may become resident
// while its predecessor in the stream is still running; it must execute pdl_wait() before it
// touches anything the predecessor writes.  pdl_launch_dependents() in the predecessor allows the
// successor's CTAs to be scheduled from that point on.  Both are no-ops in a normal launch.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
static inline cudaError_t launch_kernel(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                        bool programmatic, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
#ifdef PCD_NO_PDL            // development builds only (tools/): measure the chain without programmatic launches
    programmatic = false;
#endif
    cfg.numAttrs = programmatic ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// Per-device cache of the SM count: the query costs microseconds and the answer differs between the devices of one process.
struct PerDeviceInt {
    int v[64];
};
static inline int current_device() {
    int dev = 0;
    return cudaGetDevice(&dev) == cudaSuccess && dev >= 0 && dev < 64 ? dev : -1;
}
static inline int num_sms() {
    static PerDeviceInt cache = {};
    const int dev = current_device();
    if (dev < 0) return 0;
    if (cache.v[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
        cache.v[dev] = n;
    }
    return cache.v[dev];
}

// Opt a kernel in to more than 48 KB of dynamic shared memory ONCE per (kernel, device) and size: the attribute call
// costs microseconds and the entry points are meant to be allocation- and configuration-free in steady state.  The memo is
// keyed by the kernel's ADDRESS (instantiations of one template share their pointer type, so a per-type static would
// let one instantiation's opt-in stand for another's).  max_carveout also asks for the largest shared-memory carve-out
// (residency limited by registers may need more shared memory than the default split); the occupancy that ctas_per_sm
// reports depends on it, so opt in before the first ctas_per_sm of that kernel.
cudaError_t opt_in_smem_fn(const void *kernel, size_t bytes, bool max_carveout);     // pcd_host.cu
template <typename K>
static inline cudaError_t opt_in_smem(K kernel, size_t bytes, bool max_carveout = false) {
    return opt_in_smem_fn(reinterpret_cast<const void *>(kernel), bytes, max_carveout);
}
// Resident CTAs per SM (at least 1) of `kernel` at `threads` threads and `smem` bytes of dynamic shared memory, queried once
// per (kernel, device, threads, smem).
cudaError_t ctas_per_sm_fn(const void *kernel, int threads, size_t smem, int *ctas);  // pcd_host.cu
template <typename K>
static inline cudaError_t ctas_per_sm(K kernel, int threads, size_t smem, int *ctas) {
    return ctas_per_sm_fn(reinterpret_cast<const void *>(kernel), threads, smem, ctas);
}

// Grid of a grid-stride kernel: one CTA per `per_cta` work items, at most `cap` CTAs.
static inline int capped_grid(long long work, int per_cta, long long cap) {
    const long long want = (work + per_cta - 1) / per_cta;
    return (int)(want < cap ? want : cap);
}

// Runtime value -> template argument: call the generic lambda `fn` with std::integral_constant<int, value>, which converts
// to a template argument inside it (fn(F) ... kernel<F><<<...>>>).  fn is instantiated for every value, and with it every
// kernel it names.
template <int V> using IntC = std::integral_constant<int, V>;
template <typename Fn>
static inline decltype(auto) with_form(int form, Fn &&fn) {
    if (form == PCD_FORM_ROW_COL) return fn(IntC<PCD_FORM_ROW_COL>{});
    if (form == PCD_FORM_COL_ROW) return fn(IntC<PCD_FORM_COL_ROW>{});
    return fn(IntC<PCD_FORM_SUM_FIRST>{});
}
template <typename Fn>
static inline decltype(auto) with_norm(int norm_kind, Fn &&fn) {
    if (norm_kind == PCD_NORM_FMA) return fn(IntC<PCD_NORM_FMA>{});
    return fn(IntC<PCD_NORM_MULSUM>{});
}

}  // namespace pcd
