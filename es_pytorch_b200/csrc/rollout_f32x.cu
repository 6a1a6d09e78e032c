// rollout_f32x.cu -- fused perturb + MLP rollout + fitness in float32 on the CUDA cores at packed-FMA (fma.rn.f32x2) rate,
// for obs -> 64 -> 64 -> act (act <= 32) tanh MLPs.  Same contract as rollout_f32.cu (reference: src/core/policy.py:61-64,
// src/nn/nn.py:35-46, src/gym/gym_runner.py:50-54, src/gym/training_result.py:28); rollout_f32.cu stays the general-shape
// kernel (and the one that splits a single evaluation over the SMs).
//
// What changed against rollout_f32.cu (76 ms per K = 10 000 generation, FMA pipe 25 %, one LDS.128 per 3.5 FFMA):
//   * one CTA = one antithetic PAIR: layer 1 is V = Xn . eps1^T + eps_b1 once for both signs, z1+- = U +- sigma*V with
//     U = Xn . theta1^T + b1 computed once per generation (float64 accumulation, rounded once).  Layer 1 is 82 % of the
//     multiply-adds of an evaluation, so the pair costs 0.59 of two separate evaluations;
//   * register tiles of 8 time steps x 2 units per thread with the accumulators PAIRED ALONG K: acc[i][j] is a float32x2
//     holding the partial sums over even / odd k, so that both operands of fma.rn.f32x2 come straight out of one 128-bit
//     shared-memory load each (rows of Xn and rows of eps1 are both contiguous in k), no transposes, no duplicated operands;
//   * the shared-memory pipe, not the FMA pipe, is what a CUDA-core GEMM at FFMA2 rate runs out of first.  Measured with ncu
//     (profiles/r2_m_rollout_f32x_ncu_raw.csv): a 128-bit load costs 4 wavefronts when the lanes of a quarter warp read
//     different addresses and 2 when the whole warp reads one address.  Here a warp owns 8 time steps x 64 units: the 8
//     activation rows are read by all lanes at the same address (2 wavefronts each) and every lane reads its own 2 weight
//     rows (4 each): 24 wavefronts per 32 FFMA2 (= 16 FMA-pipe cycles) -- the same as the first version's 4 x 4 tiles with 8
//     rows x 4 units per warp (8 loads of ~3.3 wavefronts), and the two run equally fast: LSU data pipe 70 %, FMA pipe 47 %,
//     24.4 ms per K = 10 000 generation.  tools/bench_src/lds_bench.cu measures the load costs directly: 2.4 cycles for a
//     128-bit load with 1, 2 or 4 distinct addresses per warp, 4.0 with 8 or more.  By that model 8 x 4 tiles for layer 1 (two
//     teams of 8 warps splitting the K chunks, half-warp-broadcast rows, partial sums merged through shared memory) should cut
//     layer 1's LSU time by a third; built and measured: 25.6 ms, no gain (64 accumulator registers leave the compiler no room
//     to prefetch the next operands) -- reverted.
//   * eps1 is never converted or scaled: cp.async (4-byte granules: a slice has 4-byte alignment only) moves the next pair's
//     64 x obs block into shared memory while the last tile of the current pair is in its layers 2 / 3;
//   * the observation tiles are pre-tiled once per generation into the shared-memory image of every (tile, 16-column chunk)
//     stage and thread 0 streams them through a ring of stages, several chunks ahead, with one cp.async.bulk each.
//
// Thread mapping (512 threads = 16 warps): warp w owns time steps 8 w .. 8 w + 7 of the 128-step tile; lane l owns units
// l and l + 32 in layers 1 / 2 and unit l (< act) in layer 3.  Weight rows have a pitch of 16 bytes mod 128, so the 8 lanes
// of a quarter warp hit 8 different bank groups.
#include "common.cuh"

namespace {

typedef unsigned long long u64;

constexpr int FX_MT = 128;                          // time steps per tile
constexpr int FX_H = 64;                            // hidden width
constexpr int FX_KC = 16;                           // observation columns per stage
constexpr int FX_NST = 6;                           // stages in the ring
constexpr int FX_AHEAD = 4;                         // chunks in flight ahead of the one being consumed
constexpr int FX_XP = FX_KC;                        // stage row pitch (floats): rows are read by broadcast, no padding
constexpr int FX_STAGE_FLOATS = FX_MT * FX_XP;      // 2048 floats = 8 KB
constexpr int FX_HP = FX_H + 4;                     // row pitch of W2 / W3 (floats)
constexpr int FX_AP = FX_H;                         // row pitch of the activation tile H (read by broadcast)
constexpr int FX_CWARPS = 16;
constexpr int FX_CT = FX_CWARPS * 32;
constexpr int FX_THREADS = FX_CT;                 // (a 17th producer warp would cost the register file of 4 warps: 96 instead of 128 registers)
constexpr uint32_t FX_SPIN_LIMIT = 1u << 28;

struct FxParams {
    const float* table;
    const int64_t* idx;
    const float* theta;
    const float* xst;        // [n_tiles][nkc][FX_MT][FX_XP] stage images of the normalised observations
    const float* uperm;      // [n_tiles][16][FX_CT]: U in thread order (value i*2+j of thread tid)
    const float* rew;        // [T][act]
    const float* act_noise;  // [n_pairs][2][T][act] scaled action noise (mt_gauss.cu) or NULL
    double* fit_pos;
    double* fit_neg;
    float* behv_pos;
    float* behv_neg;
    int n_pairs, obs, act, T, nkc, n_tiles, fit_stride;
    float sigma, pos_scale;
    int w1, b1, w2, b2, w3, b3;
    long long table_len;
    int P;
    int* err;
    int n_eps;               // episodes per evaluation (act_noise [n_pairs][2][n_eps][T][act]); > 1 only in rollout_f32x_kernel<true>
};

struct FxSmem { uint32_t e1, xs, h, w2, w3, bias, posb, red, bars, total; int e1p, act4; };
__host__ __device__ inline FxSmem fx_layout(int obs, int act) {
    FxSmem L;
    const int nkc = (obs + FX_KC - 1) / FX_KC;
    L.e1p = nkc * FX_KC + 4;                         // (e1p * 4) mod 128 is 16 or 80: consecutive rows, different bank groups
    L.act4 = (act + 3) & ~3;
    uint32_t o = 0;
    L.e1 = o;   o += (uint32_t)FX_H * L.e1p * 4;
    L.xs = o;   o += (uint32_t)FX_NST * FX_STAGE_FLOATS * 4;
    L.h = o;    o += (uint32_t)FX_MT * FX_AP * 4;
    L.w2 = o;   o += 2u * FX_H * FX_HP * 4;
    L.w3 = o;   o += 2u * L.act4 * FX_HP * 4;
    L.bias = o; o += (2u * (FX_H + 32) + FX_H) * 4;   // [sign][b2 (64) | b3 (32)], then eps_b1 (64, unscaled)
    L.posb = o; o += (uint32_t)FX_MT * 4 * 4;
    L.red = o;  o += FX_CWARPS * 2 * 8 + 32;
    L.bars = o; o += 2 * FX_NST * 8;
    L.total = o;
    return L;
}

// ---- PTX wrappers ----------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t fx_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void fx_mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(fx_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fx_mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(fx_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fx_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(fx_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void fx_mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0, ok = 0;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(fx_smem_u32(bar)), "r"(parity) : "memory");
        if (!ok && ++spins > FX_SPIN_LIMIT) __trap();               // watchdog: trap instead of hanging the GPU
    } while (!ok);
}
__device__ __forceinline__ void fx_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(fx_smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(fx_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fx_cp_async4(float* dst_smem, const float* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(fx_smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void fx_cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ void fx_bar() { __syncthreads(); }
__device__ __forceinline__ u64 fx_fma2(u64 a, u64 b, u64 c) {
    u64 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ float fx_hsum(u64 v) {
    float a, b;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
    return a + b;
}
__device__ __forceinline__ double fx_warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// acc[i][j] += sum_k A[row i][k] * B[row j][k] over NK4 groups of four k.  A: 8 consecutive rows, the same for the whole warp
// (a_pitch4 apart, pitches in 16-byte units); B: this lane's two rows, 32 * b_pitch4 apart.  The two halves of every
// accumulator hold the even-k and the odd-k partial sums.
template <int NK4>
__device__ __forceinline__ void fx_tile_mma(const ulonglong2* __restrict__ A, int a_pitch4, const ulonglong2* __restrict__ B,
                                            int b_pitch4, u64 (&acc)[8][2]) {
#pragma unroll
    for (int k4 = 0; k4 < NK4; ++k4) {
        ulonglong2 a[8], b[2];
#pragma unroll
        for (int j = 0; j < 2; ++j) b[j] = B[j * 32 * b_pitch4 + k4];
#pragma unroll
        for (int i = 0; i < 8; ++i) a[i] = A[i * a_pitch4 + k4];
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                acc[i][j] = fx_fma2(a[i].x, b[j].x, acc[i][j]);
                acc[i][j] = fx_fma2(a[i].y, b[j].y, acc[i][j]);
            }
    }
}
// the warp-wide sums of v[0..7] in 9 shuffles (transposing butterfly): lane L returns the sum over the lanes of v[L / 4]
__device__ __forceinline__ float fx_warp_sum8(const float (&v)[8], int lane) {
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

// EPIS: p.n_eps > 1 episodes per evaluation sharing the forward pass; each adds its noise row to the layer-3 actions, its
// float32 reward goes into the float64 sums, and the last one drives the position integrator
template <bool EPIS>
__global__ void __launch_bounds__(FX_THREADS, 1) rollout_f32x_kernel(const __grid_constant__ FxParams p) {
    extern __shared__ __align__(128) uint8_t fx_smem[];
    const FxSmem L = fx_layout(p.obs, p.act);
    float* e1 = (float*)(fx_smem + L.e1);
    float* xs = (float*)(fx_smem + L.xs);
    float* H = (float*)(fx_smem + L.h);
    float* w2s = (float*)(fx_smem + L.w2);
    float* w3s = (float*)(fx_smem + L.w3);
    float* bias = (float*)(fx_smem + L.bias);
    float* posb = (float*)(fx_smem + L.posb);
    double* red = (double*)(fx_smem + L.red);
    float* redpos = (float*)(fx_smem + L.red + FX_CWARPS * 2 * 8);
    uint64_t* full = (uint64_t*)(fx_smem + L.bars);
    uint64_t* empty = full + FX_NST;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int my_pairs = (p.n_pairs - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const int NKC = p.nkc, NT = p.n_tiles, e1p = L.e1p, act4 = L.act4;

    if (tid == 0) {
        for (int s = 0; s < FX_NST; ++s) { fx_mbar_init(&full[s], 1); fx_mbar_init(&empty[s], FX_CWARPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // the padding columns of eps1 (multiplied by the zero padding of the observation stages) and the padding rows of W3 must
    // hold finite values
    for (int i = tid; i < FX_H * e1p; i += FX_THREADS) e1[i] = 0.f;
    for (int i = tid; i < 2 * act4 * FX_HP; i += FX_THREADS) w3s[i] = 0.f;
    for (int i = tid; i < 2 * (FX_H + 32) + FX_H; i += FX_THREADS) bias[i] = 0.f;
    float* eb1 = bias + 2 * (FX_H + 32);                        // the layer-1 bias part of the perturbation: V += eps_b1
    __syncthreads();

    // ===================== compute threads =====================
    const int r0 = warp * 8;                                    // this warp's rows of the tile: r0 .. r0 + 7
    const int n3 = min(lane, act4 - 1);                         // layer-3 unit of this lane (lanes >= act idle along)
    const float sg = p.sigma, ps = p.pos_scale;
    const bool want_pos = p.behv_pos != nullptr;
    const int e1p4 = e1p >> 2;

    // eps1 of a pair -> shared memory, asynchronously (4-byte granules: a slice start has 4-byte alignment only)
    auto stage_eps = [&](long long slice) {
        const float* __restrict__ src = p.table + slice + p.w1;
        const int total = FX_H * p.obs;
        int n = tid / p.obs, k = tid - n * p.obs;
        const int dn = FX_CT / p.obs, dk = FX_CT - dn * p.obs;
        for (int e = tid; e < total; e += FX_CT) {
            fx_cp_async4(e1 + n * e1p + k, src + e);
            n += dn; k += dk;
            if (k >= p.obs) { k -= p.obs; ++n; }
        }
    };
    // theta +- sigma*eps of layers 2 and 3 and the biases (the reference's two roundings: std * noise, then the sum)
    auto stage_w = [&](long long slice) {
        const float* __restrict__ eps = p.table + slice;
        for (int e = tid; e < FX_H * FX_H; e += FX_CT) {
            const float d = __fmul_rn(sg, __ldg(eps + p.w2 + e)), t = __ldg(p.theta + p.w2 + e);
            const int o = (e >> 6) * FX_HP + (e & 63);
            w2s[o] = __fadd_rn(t, d); w2s[FX_H * FX_HP + o] = __fadd_rn(t, -d);
        }
        for (int e = tid; e < p.act * FX_H; e += FX_CT) {
            const float d = __fmul_rn(sg, __ldg(eps + p.w3 + e)), t = __ldg(p.theta + p.w3 + e);
            const int o = (e >> 6) * FX_HP + (e & 63);
            w3s[o] = __fadd_rn(t, d); w3s[act4 * FX_HP + o] = __fadd_rn(t, -d);
        }
        if (tid < FX_H) {
            const float d = __fmul_rn(sg, __ldg(eps + p.b2 + tid)), t = __ldg(p.theta + p.b2 + tid);
            bias[tid] = __fadd_rn(t, d); bias[FX_H + 32 + tid] = __fadd_rn(t, -d);
        } else if (tid - FX_H < p.act) {
            const int j = tid - FX_H;
            const float d = __fmul_rn(sg, __ldg(eps + p.b3 + j)), t = __ldg(p.theta + p.b3 + j);
            bias[FX_H + j] = __fadd_rn(t, d); bias[FX_H + 32 + FX_H + j] = __fadd_rn(t, -d);
        } else if (tid >= 128 && tid < 128 + FX_H) {
            eb1[tid - 128] = __ldg(eps + p.b1 + tid - 128);
        }
    };

    // observation stages: the same sequence of n_tiles * nkc chunks for every pair, FX_AHEAD chunks ahead of the consumers.
    // Thread 0 issues chunk g + FX_AHEAD into the slot of chunk g + FX_AHEAD - FX_NST when the CTA starts chunk g: that slot was
    // released FX_NST - FX_AHEAD chunks ago, so the wait on its `empty` barrier is normally already satisfied.
    const int total_chunks = my_pairs * NT * NKC;
    const int chunks_per_pair = NT * NKC;
    int issued = 0;                                             // thread 0 only
    auto produce_to = [&](int upto) {
        for (; issued < upto && issued < total_chunks; ++issued) {
            const uint32_t slot = (uint32_t)(issued % FX_NST), use = (uint32_t)(issued / FX_NST);
            fx_mbar_wait(&empty[slot], (use & 1) ^ 1);
            fx_mbar_expect_tx(&full[slot], FX_STAGE_FLOATS * 4);
            fx_bulk_g2s(xs + slot * FX_STAGE_FLOATS, p.xst + (size_t)(issued % chunks_per_pair) * FX_STAGE_FLOATS, FX_STAGE_FLOATS * 4, &full[slot]);
        }
    };
    if (tid == 0) produce_to(FX_AHEAD);
    uint32_t stage = 0, phase = 0;
    int g = 0;                                                  // chunks consumed so far
    if (my_pairs > 0) {
        const long long slice = es_checked_slice(p.idx[blockIdx.x], p.P, p.table_len, p.err);
        stage_eps(slice);
        stage_w(slice);
    }
    for (int i = 0; i < my_pairs; ++i) {
        const int pair = blockIdx.x + i * gridDim.x;
        fx_cp_async_wait_all();
        fx_bar();                                               // eps1, W2/W3 and the biases of this pair are in place
        double fs0 = 0.0, fs1 = 0.0;                            // lanes 0, 4, .., 28: reward sums of one row of the warp over the tiles
        float pp0 = 0.f, pp1 = 0.f;                             // threads 0..2: position component tid of the + / - evaluation
        for (int m = 0; m < NT; ++m) {
            // ---- layer 1: V = Xn_tile . eps1^T + eps_b1 (both signs) ----
            float V[8][2];
            {
                u64 acc[8][2];
#pragma unroll
                for (int a = 0; a < 8; ++a) { acc[a][0] = 0ull; acc[a][1] = 0ull; }
                const ulonglong2* __restrict__ Bq = reinterpret_cast<const ulonglong2*>(e1) + lane * e1p4;
                for (int kc = 0; kc < NKC; ++kc, ++g) {
                    if (tid == 0) produce_to(g + 1 + FX_AHEAD);
                    fx_mbar_wait(&full[stage], phase);
                    const ulonglong2* __restrict__ Aq = reinterpret_cast<const ulonglong2*>(xs + stage * FX_STAGE_FLOATS) + r0 * (FX_XP / 4);
                    fx_tile_mma<FX_KC / 4>(Aq, FX_XP / 4, Bq + kc * (FX_KC / 4), e1p4, acc);
                    __syncwarp();
                    if (lane == 0) fx_mbar_arrive(&empty[stage]);
                    if (++stage == FX_NST) { stage = 0; phase ^= 1; }
                }
#pragma unroll
                for (int a = 0; a < 8; ++a)
#pragma unroll
                    for (int b = 0; b < 2; ++b) V[a][b] = fx_hsum(acc[a][b]) + eb1[lane + 32 * b];      // + the bias element of eps
            }
            const float* __restrict__ up = p.uperm + (size_t)m * 16 * FX_CT + tid;
            const int rows_valid = min(FX_MT, p.T - m * FX_MT);
#pragma unroll 1
            for (int sgn = 0; sgn < 2; ++sgn) {
                // ---- epi1: h1 = tanh(U +- sigma V) -> H ----
                const float s = sgn ? -sg : sg;
#pragma unroll
                for (int a = 0; a < 8; ++a)
#pragma unroll
                    for (int b = 0; b < 2; ++b)
                        H[(r0 + a) * FX_AP + lane + 32 * b] = tanhf(fmaf(s, V[a][b], __ldg(up + (a * 2 + b) * FX_CT)));
                fx_bar();
                if (sgn == 0 && m == NT - 1 && i + 1 < my_pairs)      // every warp is past its last read of eps1: fetch the next pair's
                    stage_eps(es_checked_slice(p.idx[pair + gridDim.x], p.P, p.table_len, p.err));
                // ---- layer 2 ----
                float D[8][2];
                {
                    u64 acc[8][2];
#pragma unroll
                    for (int a = 0; a < 8; ++a) { acc[a][0] = 0ull; acc[a][1] = 0ull; }
                    fx_tile_mma<FX_H / 4>(reinterpret_cast<const ulonglong2*>(H) + r0 * (FX_AP / 4), FX_AP / 4,
                                          reinterpret_cast<const ulonglong2*>(w2s + sgn * FX_H * FX_HP) + lane * (FX_HP / 4), FX_HP / 4, acc);
                    const float* b2 = bias + sgn * (FX_H + 32);
#pragma unroll
                    for (int a = 0; a < 8; ++a)
#pragma unroll
                        for (int b = 0; b < 2; ++b) D[a][b] = tanhf(fx_hsum(acc[a][b]) + b2[lane + 32 * b]);
                }
                fx_bar();                                           // every thread has read h1
#pragma unroll
                for (int a = 0; a < 8; ++a)
#pragma unroll
                    for (int b = 0; b < 2; ++b) H[(r0 + a) * FX_AP + lane + 32 * b] = D[a][b];
                fx_bar();
                // ---- layer 3 (lane = action unit), reward, position ----
                {
                    u64 acc3[8];
#pragma unroll
                    for (int a = 0; a < 8; ++a) acc3[a] = 0ull;
                    const ulonglong2* __restrict__ A3 = reinterpret_cast<const ulonglong2*>(H) + r0 * (FX_AP / 4);
                    const ulonglong2* __restrict__ B3 = reinterpret_cast<const ulonglong2*>(w3s + sgn * act4 * FX_HP) + n3 * (FX_HP / 4);
#pragma unroll 4
                    for (int k4 = 0; k4 < FX_H / 4; ++k4) {
                        const ulonglong2 b = B3[k4];
#pragma unroll
                        for (int a = 0; a < 8; ++a) {
                            const ulonglong2 x = A3[a * (FX_AP / 4) + k4];
                            acc3[a] = fx_fma2(x.x, b.x, acc3[a]);
                            acc3[a] = fx_fma2(x.y, b.y, acc3[a]);
                        }
                    }
                    const bool unit = lane < p.act;
                    const float b3 = bias[sgn * (FX_H + 32) + FX_H + n3];
                    const int tb = m * FX_MT + r0;                                     // time step of row 0 of this warp
                    if (EPIS) {
                        float av[8], cw[8], v[8];
#pragma unroll
                        for (int a = 0; a < 8; ++a) {
                            const bool live = unit && tb + a < p.T;
                            av[a] = tanhf(fx_hsum(acc3[a]) + b3);
                            cw[a] = live ? __ldg(p.rew + (size_t)(tb + a) * p.act + lane) : 0.f;
                        }
                        for (int e = 0; e < p.n_eps; ++e) {
                            const float* __restrict__ nz = p.act_noise + ((((size_t)pair * 2 + sgn) * p.n_eps + e) * p.T + tb) * p.act + lane;
#pragma unroll
                            for (int a = 0; a < 8; ++a) {
                                const bool live = unit && tb + a < p.T;
                                const float ae = live ? __fadd_rn(av[a], __ldg(nz + a * p.act)) : 0.f;
                                v[a] = ae * cw[a];
                                if (want_pos && e == p.n_eps - 1) {
#pragma unroll
                                    for (int jj = 0; jj < 3; ++jj)
                                        if (lane == jj % p.act) posb[(r0 + a) * 4 + jj] = ae;
                                }
                            }
                            const float r = fx_warp_sum8(v, lane);         // lanes 4 q .. 4 q + 3: episode e's reward of row q
                            if ((lane & 3) == 0) { if (sgn) fs1 += (double)r; else fs0 += (double)r; }
                        }
                    } else {
                    const float* __restrict__ nz = p.act_noise ? p.act_noise + (((size_t)pair * 2 + sgn) * p.T + tb) * p.act + lane : nullptr;
                    float v[8];
#pragma unroll
                    for (int a = 0; a < 8; ++a) {
                        float av = tanhf(fx_hsum(acc3[a]) + b3);
                        const bool live = unit && tb + a < p.T;
                        if (nz && live) av = __fadd_rn(av, __ldg(nz + a * p.act));     // a += randn * ac_std (nn.py:47-48)
                        v[a] = live ? av * __ldg(p.rew + (size_t)(tb + a) * p.act + lane) : 0.f;
                        if (want_pos) {
#pragma unroll
                            for (int jj = 0; jj < 3; ++jj)
                                if (lane == jj % p.act) posb[(r0 + a) * 4 + jj] = av;   // action component jj % act
                        }
                    }
                    const float r = fx_warp_sum8(v, lane);             // lanes 4 q .. 4 q + 3: the reward of row q
                    if ((lane & 3) == 0) { if (sgn) fs1 += (double)r; else fs0 += (double)r; }
                    }
                }
                fx_bar();                                           // H is free again; the position columns are visible
                if (want_pos && tid < 3) {
                    float pp = sgn ? pp1 : pp0;
                    for (int r = 0; r < rows_valid; ++r) pp = __fadd_rn(pp, __fmul_rn(ps, posb[r * 4 + tid]));   // step order
                    if (sgn) pp1 = pp; else pp0 = pp;
                }
            }
        }
        // ---- the pair's sums: rows -> warp -> CTA in fixed order ----
        const double w0 = fx_warp_sum_d(fs0), w1 = fx_warp_sum_d(fs1);
        if (lane == 0) { red[warp * 2 + 0] = w0; red[warp * 2 + 1] = w1; }
        if (want_pos && tid < 3) { redpos[tid] = pp0; redpos[4 + tid] = pp1; }
        fx_bar();
        if (tid == 0) {
            double fp = 0.0, fn = 0.0;
            for (int w = 0; w < FX_CWARPS; ++w) { fp += red[w * 2 + 0]; fn += red[w * 2 + 1]; }
            if (EPIS) { fp /= p.n_eps; fn /= p.n_eps; }               // obj.py: rews /= max(1, eps_per_policy)
            p.fit_pos[(size_t)pair * p.fit_stride] = fp;
            p.fit_neg[(size_t)pair * p.fit_stride] = fn;
            if (want_pos) {
                for (int j = 0; j < 3; ++j) { p.behv_pos[pair * 3 + j] = redpos[j]; p.behv_neg[pair * 3 + j] = redpos[4 + j]; }
            }
        }
        if (i + 1 < my_pairs) stage_w(es_checked_slice(p.idx[pair + gridDim.x], p.P, p.table_len, nullptr));
        fx_bar();                                                   // thread 0 has read `red` before anyone can write it again
    }
}

// observation stream -> stage images [tile][chunk][128 rows][16]: zero beyond T / obs
__global__ void rollout_f32x_prep_kernel(const float* __restrict__ obsn, int T, int obs, int nkc, int n_tiles, float* __restrict__ xst) {
    const size_t total = (size_t)n_tiles * nkc * FX_STAGE_FLOATS;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % FX_XP);
        const int r = (int)((i / FX_XP) % FX_MT);
        const int kc = (int)((i / FX_STAGE_FLOATS) % nkc);
        const int m = (int)(i / ((size_t)FX_STAGE_FLOATS * nkc));
        const int t = m * FX_MT + r, k = kc * FX_KC + c;
        xst[i] = (c < FX_KC && k < obs && t < T) ? obsn[(size_t)t * obs + k] : 0.f;
    }
}

// U[t][n] = b1[n] + sum_k Xn[t][k] * theta1[n][k], float64 accumulation (k ascending), rounded once; written in the thread
// order of the rollout kernel: uperm[(m * 16 + i * 2 + j) * 512 + tid] for row 8 (tid / 32) + i, unit tid % 32 + 32 j of tile m
constexpr int FX_UB_ROWS = 8, FX_UB_KT = 64;
__global__ void __launch_bounds__(256) rollout_f32x_ubase_kernel(const float* __restrict__ obsn, const float* __restrict__ theta,
                                                                  int w1, int b1, int T, int obs, float* __restrict__ uperm) {
    __shared__ float s_w[FX_UB_KT][FX_H + 1];
    __shared__ float s_x[FX_UB_ROWS][FX_UB_KT];
    const int n = threadIdx.x & 63, rg = threadIdx.x >> 6;
    const int t0 = blockIdx.x * FX_UB_ROWS;
    double acc[2];
    acc[0] = acc[1] = (double)__ldg(theta + b1 + n);
    for (int k0 = 0; k0 < obs; k0 += FX_UB_KT) {
        const int kn = min(FX_UB_KT, obs - k0);
        for (int i = threadIdx.x; i < FX_H * FX_UB_KT; i += 256) {
            const int nn = i / FX_UB_KT, kk = i - nn * FX_UB_KT;
            s_w[kk][nn] = (kk < kn) ? __ldg(theta + w1 + (size_t)nn * obs + k0 + kk) : 0.f;
        }
        for (int i = threadIdx.x; i < FX_UB_ROWS * FX_UB_KT; i += 256) {
            const int r = i / FX_UB_KT, kk = i - r * FX_UB_KT;
            const int t = t0 + r;
            s_x[r][kk] = (kk < kn && t < T) ? obsn[(size_t)t * obs + k0 + kk] : 0.f;
        }
        __syncthreads();
        for (int kk = 0; kk < kn; ++kk) {
            const double w = (double)s_w[kk][n];
            acc[0] = fma((double)s_x[rg * 2 + 0][kk], w, acc[0]);
            acc[1] = fma((double)s_x[rg * 2 + 1][kk], w, acc[1]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int t = t0 + rg * 2 + r;
        const int m = t / FX_MT, row = t % FX_MT;
        const int i = row & 7, j = n >> 5;
        const int tid = (row >> 3) * 32 + (n & 31);
        uperm[((size_t)m * 16 + i * 2 + j) * FX_CT + tid] = (t < T) ? (float)acc[r] : 0.f;
    }
}

}  // namespace

// Returns ES_OK after launching, or ES_ERR_UNSUPPORTED (no error text) when the shape is not covered: the caller falls
// back to the general kernel of rollout_f32.cu.
int es_impl_rollout_f32x(es_ctx* ctx, const float* table, int64_t table_len, const int64_t* idx, int n_pairs,
                         const float* theta, int P, float sigma, const int* layer_sizes, int n_layers, const float* obsn,
                         const float* rew_vec, int T, float pos_scale, double* fit_pos, double* fit_neg, int fit_stride,
                         float* behv_pos, float* behv_neg, const float* act_noise, int n_eps, cudaStream_t stream) {
    if (n_layers != 3 || layer_sizes[1] != FX_H || layer_sizes[2] != FX_H || layer_sizes[3] > 32 || layer_sizes[0] < 1)
        return ES_ERR_UNSUPPORTED;
    const FxSmem L = fx_layout(layer_sizes[0], layer_sizes[3]);
    if (L.total > 227 * 1024) return ES_ERR_UNSUPPORTED;
    FxParams p;
    memset(&p, 0, sizeof(p));
    p.table = table; p.idx = idx; p.theta = theta; p.rew = rew_vec; p.act_noise = act_noise;
    p.fit_pos = fit_pos; p.fit_neg = fit_neg; p.behv_pos = behv_pos; p.behv_neg = behv_neg;
    p.n_pairs = n_pairs; p.obs = layer_sizes[0]; p.act = layer_sizes[3]; p.T = T; p.fit_stride = fit_stride;
    p.nkc = es_div_up(p.obs, FX_KC);
    p.n_tiles = es_div_up(T, FX_MT);
    p.sigma = sigma; p.pos_scale = pos_scale;
    p.w1 = 0; p.b1 = p.obs * FX_H; p.w2 = p.b1 + FX_H; p.b2 = p.w2 + FX_H * FX_H; p.w3 = p.b2 + FX_H; p.b3 = p.w3 + FX_H * p.act;
    p.table_len = table_len; p.P = P; p.err = ctx->err_dev; p.n_eps = n_eps;

    const size_t xst_bytes = (size_t)p.n_tiles * p.nkc * FX_STAGE_FLOATS * sizeof(float);
    const size_t up_bytes = (size_t)p.n_tiles * 16 * FX_CT * sizeof(float);
    void* scratch = nullptr;
    int rc = es_ctx_scratch(ctx, xst_bytes + up_bytes, &scratch);
    if (rc) return rc;
    float* xst = (float*)scratch;
    float* uperm = (float*)((char*)scratch + xst_bytes);
    p.xst = xst; p.uperm = uperm;
    {
        const size_t total = (size_t)p.n_tiles * p.nkc * FX_STAGE_FLOATS;
        int blocks = es_div_up((int64_t)total, 256);
        if (blocks > ctx->sm_count * 8) blocks = ctx->sm_count * 8;
        rollout_f32x_prep_kernel<<<blocks, 256, 0, stream>>>(obsn, T, p.obs, p.nkc, p.n_tiles, xst);
        ES_LAUNCHED(ctx);
        rollout_f32x_ubase_kernel<<<p.n_tiles * FX_MT / FX_UB_ROWS, 256, 0, stream>>>(obsn, theta, p.w1, p.b1, T, p.obs, uperm);
        ES_LAUNCHED(ctx);
    }
    const int grid = n_pairs < ctx->sm_count ? n_pairs : ctx->sm_count;
    auto kernel = n_eps > 1 ? rollout_f32x_kernel<true> : rollout_f32x_kernel<false>;
    ES_CHECK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
    kernel<<<grid, FX_THREADS, L.total, stream>>>(p);
    ES_LAUNCHED(ctx);
    return ES_OK;
}
