// tc_ptx.cuh -- raw PTX wrappers, operand layouts and small kernels shared by the tcgen05 rollouts (rollout_tc2.cu,
// rollout_tcw.cu): mbarrier, bulk / TMA copies, tcgen05 alloc / mma / ld / st / commit, shared-memory descriptors, packed
// float32x2 arithmetic, the tanh forms and the float16 hi + lo split.  Everything is in an anonymous namespace: each
// translation unit inlines its own copy.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include "common.cuh"

#ifndef T2_TANH_FORM
#define T2_TANH_FORM 1         // accurate tanh of the split kernel: 0 = (1 - e) / (1 + e) with e = 2^(-2 log2e |x|), 1 = 1 - 2 / (1 + e^2x)
                               // (measured, K = 10 000: form 0 2.508 ms, form 1 2.421 ms; error against float64 unchanged on the
                               //  Humanoid shape, 1.6e-6 of the fitness spread)
#endif
#ifndef T2_NEWTON_MASK
#define T2_NEWTON_MASK 0x0     // of the four value pairs of an 8-column batch: bit e set -> pair e takes the FMA-pipe reciprocal
                               // (measured, K = 10 000: mask 0x0 2.445 ms, 0x5 2.462, 0x7 2.476, 0xF 2.594 -- see tanh_acc2)
#endif

namespace {

constexpr uint32_t TC_SPIN_LIMIT = 1u << 28;   // mbarrier watchdog: trap instead of hanging the GPU
constexpr int TC_MT = 128, TC_KC = 64;         // time steps per MMA tile (M), K chunk (one 128-byte swizzled row of float16)
constexpr int TC_STAGE = TC_MT * 128;          // 16 KB: one observation stage, 128 rows x 64 f16

// ---- raw PTX wrappers ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try(bar, parity)) {
        if (++spins > TC_SPIN_LIMIT) __trap();            // watchdog: trap instead of hanging the GPU
    }
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// 3-D TMA tensor copy (tile mode): coordinates {element, origin unit, row}
__device__ __forceinline__ void tma_load_3d(void* dst_smem, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 ::"r"(smem_u32(dst_smem)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t* result_in_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(result_in_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]^T, f16 inputs, f32 accumulate
__device__ __forceinline__ void umma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem desc]^T: A = 128 lanes x 8 columns (16 f16 along K, element 2j in the low half of column j)
__device__ __forceinline__ void umma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st4(uint32_t taddr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
template <int N> __device__ __forceinline__ void reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N> __device__ __forceinline__ void reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }

// packed float32x2 arithmetic (one issue slot for two values)
__device__ __forceinline__ unsigned long long pk(float a, float b) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ void unpk(unsigned long long v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ unsigned long long fma2(unsigned long long a, unsigned long long b, unsigned long long c) {
    unsigned long long d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ unsigned long long add2(unsigned long long a, unsigned long long b) {
    unsigned long long d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ unsigned long long mul2(unsigned long long a, unsigned long long b) {
    unsigned long long d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ float tanh_fast(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
// tanh of two values to float32 accuracy: tanh|x| = (1 - e) / (1 + e), e = 2^(-2 log2(e) |x|) (no cancellation: e in (0, 1]);
// max abs error 1.4e-7, mean error ~1e-11 (tools/bench_src/tc_micro.cu).  The elementwise arithmetic is packed.
// NEWTON (a compile-time constant after unrolling) = false: 1 / (1 + e) by rcp.approx (2 MUFU per tanh).  NEWTON = true: the reciprocal on the FMA pipe instead
// (d = 1 + e in (1, 2]: quadratic minimax start, relative error 1.0e-2, two Newton steps -> 1e-8 before rounding; 7 packed
// FMA-pipe operations for two values).  ncu shows the split kernel at 62 % XU / 30 % FMA pipe utilisation, but moving
// reciprocals to the FMA pipe made it SLOWER (2.445 ms -> 2.594 ms with every reciprocal moved): the kernel is bound by issue
// slots and the per-tile dependency chain, not by the XU pipe.  Kept as a compile-time option (T2_NEWTON_MASK), off.
__device__ __forceinline__ void tanh_acc2(float x0, float x1, float& t0, float& t1, const bool NEWTON) {
#if T2_TANH_FORM == 1
    // tanh x = 1 - 2 / (1 + e^(2x)): 7 instructions for two values (mul2, 2 ex2, add2, 2 rcp, fma2) instead of 12; no sign
    // handling (e -> 0 / inf gives -1 / +1), same absolute-error class (cancellation near 0 as in the other form)
    float y0, y1;
    unpk(mul2(pk(x0, x1), pk(2.885390081777927f, 2.885390081777927f)), y0, y1);
    float d0, d1;
    unpk(add2(pk(ex2_approx(y0), ex2_approx(y1)), pk(1.0f, 1.0f)), d0, d1);
    unpk(fma2(pk(rcp_approx(d0), rcp_approx(d1)), pk(-2.0f, -2.0f), pk(1.0f, 1.0f)), t0, t1);
    (void)NEWTON;
#else
    float y0, y1;
    unpk(mul2(pk(x0, x1), pk(2.885390081777927f, 2.885390081777927f)), y0, y1);
    const float e0 = ex2_approx(-fabsf(y0)), e1 = ex2_approx(-fabsf(y1));
    const unsigned long long e = pk(e0, e1), one = pk(1.0f, 1.0f);
    const unsigned long long d = add2(e, one);
    const unsigned long long num = fma2(e, pk(-1.0f, -1.0f), one);
    float r0, r1;
    if (NEWTON) {
        // s = -1/d: s0 = -(c0 + c1 d + c2 d^2); s <- s + s (1 + d s) twice, the second step folded into the product with num
        unsigned long long sN = fma2(fma2(pk(-0.32322488f, -0.32322488f), d, pk(1.45451241f, 1.45451241f)), d, pk(-2.12117935f, -2.12117935f));
        sN = fma2(sN, fma2(d, sN, one), sN);
        const unsigned long long q = mul2(num, sN);
        unpk(fma2(q, fma2(d, sN, one), q), r0, r1);            // = -(1 - e) / (1 + e): only the magnitude is used
        t0 = __uint_as_float((__float_as_uint(r0) & 0x7FFFFFFFu) | (__float_as_uint(x0) & 0x80000000u));
        t1 = __uint_as_float((__float_as_uint(r1) & 0x7FFFFFFFu) | (__float_as_uint(x1) & 0x80000000u));
    } else {
        float d0, d1;
        unpk(d, d0, d1);
        unpk(mul2(num, pk(rcp_approx(d0), rcp_approx(d1))), r0, r1);
        t0 = __uint_as_float(__float_as_uint(r0) | (__float_as_uint(x0) & 0x80000000u));
        t1 = __uint_as_float(__float_as_uint(r1) | (__float_as_uint(x1) & 0x80000000u));
    }
#endif
}
// two float32 -> packed float16x2 (element 0 in the low half)
__device__ __forceinline__ uint32_t pack_h2(float lo, float hi) {
    uint32_t y;
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(y) : "f"(hi), "f"(lo));
    return y;
}
// x = hi + lo with hi = the top 11 significant bits (exact in float16 for |x| >= 2^-14, rounded to the float16 subnormal grid
// below: absolute error <= 2^-25) and lo = x - hi rounded to float16
__device__ __forceinline__ void split_h2(float x0, float x1, uint32_t& hi, uint32_t& lo) {
    const float h0 = __uint_as_float(__float_as_uint(x0) & 0xFFFFE000u), h1 = __uint_as_float(__float_as_uint(x1) & 0xFFFFE000u);
    hi = pack_h2(h0, h1);
    float l0, l1;
    unpk(fma2(pk(h0, h1), pk(-1.0f, -1.0f), pk(x0, x1)), l0, l1);
    lo = pack_h2(l0, l1);
}
__device__ __forceinline__ void split_h1(float x, __half& hi, __half& lo) {
    hi = __float2half_rn(x);
    lo = __float2half_rn(x - __half2float(hi));
}
__device__ __forceinline__ float4 lds128f(uint32_t saddr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
    return v;
}
__device__ __forceinline__ float ldg_stream(const float* p) {
    float v;
    asm("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ float4 ldg_stream4(const float4* p) {
    float4 v;
    asm("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ float ldg_pinned(const float* p) {
    float v;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
// Transposing butterfly: the warp-wide sums of v[0..7] in 9 shuffles.  Lane L returns the sum of v[sum8_index(L)].
__device__ __forceinline__ int sum8_index(int lane) { return ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1); }
__device__ __forceinline__ float warp_sum8(const float (&v)[8], int lane) {
    const bool h16 = lane & 16, h8 = lane & 8, h4 = lane & 4;
    float a[4], b[2], c;
#pragma unroll
    for (int i = 0; i < 4; ++i) a[i] = (h16 ? v[i + 4] : v[i]) + __shfl_xor_sync(0xffffffffu, h16 ? v[i] : v[i + 4], 16);
#pragma unroll
    for (int i = 0; i < 2; ++i) b[i] = (h8 ? a[i + 2] : a[i]) + __shfl_xor_sync(0xffffffffu, h8 ? a[i] : a[i + 2], 8);
    c = (h4 ? b[1] : b[0]) + __shfl_xor_sync(0xffffffffu, h4 ? b[0] : b[1], 4);
    c += __shfl_xor_sync(0xffffffffu, c, 2);
    c += __shfl_xor_sync(0xffffffffu, c, 1);
    return c;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// K-major, 128-byte-swizzled operand tile: rows of 128 B, 8-row atoms of 1024 B (SBO), descriptor version 1 (sm_100)
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) |
           ((uint64_t)2 << 61);
}
// kind::f16 instruction descriptor: D = f32, A = B = f16 (format 0), both K-major, M x N
__device__ __forceinline__ uint32_t umma_idesc_f16(int M, int N) {
    return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__host__ __device__ __forceinline__ uint32_t sw128_off(int row, int k /*0..63*/) {
    return (uint32_t)(row * 128 + ((((k >> 3) ^ (row & 7)) << 4) | ((k & 7) << 1)));
}

// 4 K steps of 16 over one 64-wide chunk, A from shared memory (descriptor) / from TMEM
__device__ __forceinline__ void issue_ss4(uint32_t d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc0) {
    umma_ss(d, a_desc, b_desc, idesc, acc0);
    umma_ss(d, a_desc + 2, b_desc + 2, idesc, 1);
    umma_ss(d, a_desc + 4, b_desc + 4, idesc, 1);
    umma_ss(d, a_desc + 6, b_desc + 6, idesc, 1);
}
__device__ __forceinline__ void issue_ts4(uint32_t d, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t acc0) {
    umma_ts(d, a_tmem, b_desc, idesc, acc0);
    umma_ts(d, a_tmem + 8, b_desc + 2, idesc, 1);
    umma_ts(d, a_tmem + 16, b_desc + 4, idesc, 1);
    umma_ts(d, a_tmem + 24, b_desc + 6, idesc, 1);
}

// observation stream -> float16 (hi[, lo]), tiled into the shared-memory image of each (M tile, K chunk, piece) stage
template <bool SPLIT>
__global__ void rollout_tc2_prep_kernel(const float* __restrict__ obsn, int T, int obs, int nkc, int n_mtiles, uint8_t* __restrict__ xnt) {
    constexpr int NP = SPLIT ? 2 : 1;
    const size_t total = (size_t)n_mtiles * nkc * TC_MT * TC_KC;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int k = (int)(i % TC_KC);
        const int row = (int)((i / TC_KC) % TC_MT);
        const int kc = (int)((i / (TC_KC * TC_MT)) % nkc);
        const int m = (int)(i / ((size_t)TC_KC * TC_MT * nkc));
        const int t = m * TC_MT + row, kk = kc * TC_KC + k;
        const float v = (kk < obs) ? ((t < T) ? obsn[(size_t)t * obs + kk] : 0.f) : ((kk == obs) ? 1.0f : 0.f);   // col `obs` = 1: bias
        uint8_t* stage = xnt + ((size_t)(m * nkc + kc) * NP) * TC_STAGE;
        __half hi, lo;
        split_h1(v, hi, lo);
        *(__half*)(stage + sw128_off(row, k)) = hi;
        if (SPLIT) *(__half*)(stage + TC_STAGE + sw128_off(row, k)) = lo;
    }
}

}  // namespace
