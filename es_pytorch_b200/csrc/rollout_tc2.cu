// rollout_tc2.cu -- fused perturb + MLP rollout + fitness on the 5th-gen tensor cores, float16 operands, two precisions:
//
//   SPLIT = false (ES_ROLLOUT_TC):   one tcgen05.mma per product, tanh.approx            -> float16-grade fitness
//   SPLIT = true  (ES_ROLLOUT_TC3):  every operand is a float16 hi + lo pair (x = hi + lo to ~2^-22) and every product is
//                                    THREE MMAs  hi*hi + hi*lo + lo*hi  accumulated in float32 in TMEM (measured error of a
//                                    K=384 dot: 1.5e-6 relative, tools/bench_src/tc_micro.cu), the tanh is evaluated to
//                                    float32 accuracy ((1-e)/(1+e), e = 2^(-2|x| log2 e): max abs error 1.4e-7) and rewards
//                                    are summed in float64 -> float32-equivalent fitness (the reference's arithmetic is
//                                    float32: src/nn/nn.py:42-50, src/core/policy.py:61-64)
//
// Same contract as rollout_f32.cu (reference: src/core/policy.py:61-64, src/nn/nn.py:35-46, src/gym/gym_runner.py:50-54,
// src/gym/training_result.py:28) for obs -> 64 -> 64 -> act (act <= 32) tanh MLPs.
//
// One CTA = one antithetic pair at a time (persistent over pairs), episode time on the MMA M dimension, 128 steps per tile:
//   L1   V (128 x 64 f32, TMEM) = Xn_tile . eps1^T      eps1 UNSCALED, straight from a float16 shadow of the noise table;
//        z1+- = U +- sigma*V,  U = Xn . theta1^T + b1 computed once per generation in float64 -> float32 (ubase kernel), so one
//        MMA chain serves both signs and the unperturbed term carries no tensor-core rounding at all
//   epi1 h1+- = tanh(z1+-) -> float16 (hi[, lo]) -> TMEM (tcgen05.st): the activations never touch shared memory, they are the
//        A operand of the next layer's MMA straight from TMEM (tcgen05.mma [d], [a_tmem], b_desc: "TS" form)
//   L2   D2+- = h1+- . (theta2 +- sigma*eps2)^T,  epi2: h2+- = tanh(D2+- + b2+-) -> TMEM (over h1+-)
//   L3   D3+- = h2+- . (theta3 +- sigma*eps3)^T (N = 32),  epi3: a = tanh(D3 + b3), r_t = <a_t, c_t>, fitness += r_t
//
// Operand staging:
//   * Xn: pre-tiled once per generation into the exact shared-memory image of every (tile, K chunk[, piece]) stage
//     (rollout_tc2_prep_kernel) -> one 16 KB cp.async.bulk per stage into a ring;
//   * eps1 (82 % of a perturbation): the library keeps float16 shadows of the table (hi, and lo for SPLIT) in 8 copies shifted
//     by 0..7 elements; in copy idx % 8 every row of eps1 is 16-byte aligned, and ONE 3-D TMA tensor copy per K chunk
//     (dims {64 elements, origin in 16-byte units, 64 rows of stride obs*2 bytes}: overlapping strides, 128-byte swizzle)
//     lands the 64 x 64 block in the K-major swizzled layout the MMA descriptor expects.  No thread touches eps1.
//     (Shapes without 16-byte aligned rows, or no memory for the shadows: builder warps convert the float32 slice.)
//   * theta2/3 +- sigma*eps2/3 and the biases: builder warps compute them one pair ahead into an L2-resident image, a copier
//     warp moves the image into shared memory with two bulk copies when the previous pair's MMAs have retired.
//
// 28 warps (7 warpgroups), setmaxnreg moves registers from the data-movement warpgroups to the 16 epilogue warps:
//   warp 0 producer (Xn ring) | warp 1 L1 issuer + TMEM owner | warps 2-3 L2/L3 issuers
//   warps 4-19 epilogue (TMEM lane quarter = warp % 4) | warps 20-26 builders | warp 27 copier
// Epilogue organisation (what the 512 TMEM columns allow):
//   SPLIT=0: two groups of 8 warps on alternate tiles (column half = (warp-4)%8/4), 256 columns each; V is free again after
//            epi1, so the next L1 of a group runs under its own epi2/epi3; issuer warp g serves group g.
//   SPLIT=1: ONE group of 16 warps on every tile (column quarter = (warp-4)/4), the wide V double-buffered (2 x 128 columns) so
//            that L1 of tile g+1 runs under the epilogue of tile g; with two groups D2/D3 would have to alias V and every
//            group sat idle during its own L1 (31 % of the epilogue warps' time in the first version).  Issuer warp s serves
//            sign s.  In both modes the + sign runs one phase ahead of the - sign (epi1+ | L2+ under epi1- | L2- under epi2+
//            | L3+ under epi2- | L3- under epi3+ | epi3-), so the short L2/L3 MMAs are hidden behind epilogue work.
// TMEM (512 columns, 256 per epilogue group):
//   SPLIT=0 (per group, +256 for group 1): V 0-63 | h+ 64-95 | h- 96-127 | D2+ (D3+) 128-191 | D2- (D3-) 192-255
//   SPLIT=1: V buffer 0: 0-127, buffer 1: 128-255 (two partial sums each, see below) | h+hi 256-287 | h+lo 288-319 | h-hi 320-351 |
//            h-lo 352-383 | D2+ (D3+) 384-447 | D2- (D3-) 448-511
// SPLIT layer 1 issues HALF-as-many, twice-as-wide MMAs: eps1's hi and lo blocks of a K chunk are adjacent in shared memory, so
// x_hi . [eps_hi ; eps_lo]^T is ONE N = 128 instruction (columns 0-63: x_hi.eps_hi, 64-127: x_hi.eps_lo); x_lo . eps_hi (N = 64) adds
// into columns 0-63 and the epilogue reads V = cols[n] + cols[64 + n].  (The single L1 issuer warp was the split kernel's
// limiter at 12 small MMAs per K chunk: ~90 cycles of issue per 35 cycles of tensor work.)
#include <stdlib.h>
#include "tc_ptx.cuh"

namespace {

constexpr int T2_THREADS = 896;
constexpr int T2_W_PROD = 0, T2_W_L1 = 1, T2_W_L23 = 2, T2_EPI_WARP0 = 4, T2_GRP_WARPS = 8, T2_EPI_WARPS = 16,
              T2_BLD_WARP0 = 20, T2_BLD_WARPS = 7, T2_W_COPY = 27;
constexpr int T2_REG_MOVE = 48, T2_REG_BUILD = 48, T2_REG_EPI = 88;    // 128*48 + 256*48 + 512*88 = 63488 <= 28 warps x 72 x 32
constexpr int T2_H = 64, T2_MT = 128, T2_KC = 64, T2_ACT_PAD = 32;
constexpr int T2_STAGE = T2_MT * 128;          // 16 KB: 128 rows x 64 f16
constexpr int T2_B1_CHUNK = T2_H * 128;        // 8 KB: 64 rows x 64 f16
constexpr int T2_W3_BLOCK = T2_ACT_PAD * 128;  // 4 KB

struct T2Maps {
    CUtensorMap hi, lo;           // 3-D maps over the float16 shadows: dims {64 elements, origin (16-byte units), 64 rows}
};

struct T2Params {
    const float* table;
    const int64_t* idx;
    const float* theta;
    const uint8_t* xnt;           // [n_mtiles][nkc][pieces][16 KB stage image]
    const float* ubase;           // float4 [n_mtiles][2 halves][8 chunks][128 rows]
    const float* crt;             // reward vectors transposed per tile: [n_mtiles][32 cols][128 rows]
    const float* act_noise;       // [n_pairs][2][T][act] scaled action noise (mt_gauss.cu) or NULL
    uint8_t* images;              // [gridDim.x][2][image bytes]
    double* fit_pos;
    double* fit_neg;
    float* behv_pos;
    float* behv_neg;
    size_t shadow_stride;         // elements per shifted copy
    int use_tma;                  // eps1 by TMA from the shadows; 0: the builders convert the float32 slice
    int n_pairs, obs, act, T, nkc, n_mtiles, fit_stride;
    float sigma, pos_scale;
    int w1, b1, w2, b2, w3, b3;   // flat parameter offsets
    long long table_len;
    int P;
    int* err;
};

template <bool SPLIT> struct T2Cfg {
    static constexpr int NP = SPLIT ? 2 : 1;              // pieces per operand
    static constexpr int NST = SPLIT ? 4 : 8;             // observation stages in the ring
    static constexpr int NG = SPLIT ? 1 : 2;              // epilogue groups
    static constexpr int GW = T2_EPI_WARPS / NG;          // warps per group (barrier arrival counts)
    static constexpr int CW = 64 / (GW / 4);              // accumulator columns per epilogue warp (32 / 16)
    // TMEM columns.  !SPLIT: offsets inside a group's 256 columns.  SPLIT: absolute (one group), V buffer b at 128*b.
    static constexpr int V_STRIDE = SPLIT ? 128 : 256;    // V of tile g at V_STRIDE * (g & 1)
    static constexpr int G_STRIDE = SPLIT ? 0 : 256;      // group base of the H / D2 regions
    static constexpr int C_HP = SPLIT ? 256 : 64, C_HN = SPLIT ? 320 : 96;     // [+32: lo piece when SPLIT]
    static constexpr int C_D2P = SPLIT ? 384 : 128, C_D2N = SPLIT ? 448 : 192;
};

struct T2Smem { uint32_t b1, xst, w2, w3, bias, red, bars, total; };
template <bool SPLIT> __host__ __device__ inline T2Smem t2_layout(int nkc) {
    using C = T2Cfg<SPLIT>;
    T2Smem L;
    uint32_t o = 0;
    L.b1 = o;   o += (uint32_t)C::NP * nkc * T2_B1_CHUNK;         // [kc][piece][64 rows x 128 B]
    L.xst = o;  o += (uint32_t)C::NST * T2_STAGE;
    L.w2 = o;   o += 2u * C::NP * T2_B1_CHUNK;                    // [sign][piece][64 rows x 128 B]
    L.w3 = o;   o += 2u * C::NP * T2_W3_BLOCK;                    // [sign][piece][32 rows x 128 B]
    L.bias = o; o += 2 * 1024;                                    // double-buffered by pair parity
    L.red = o;  o += 2 * T2_EPI_WARPS * 64 + 64;                  // per-pair sums of the epilogue warps [parity][warp][8 doubles] + counters
    L.bars = o; o += 1024;
    L.total = o;
    return L;
}
// operand image in global scratch: [W2 | W3 | bias 1 KB | (B1 when the builders make it)]
struct T2Image { uint32_t w2, w3, bias, b1, total; };
template <bool SPLIT> __host__ __device__ inline T2Image t2_image(int nkc, int with_b1) {
    using C = T2Cfg<SPLIT>;
    T2Image I;
    uint32_t o = 0;
    I.w2 = o;   o += 2u * C::NP * T2_B1_CHUNK;
    I.w3 = o;   o += 2u * C::NP * T2_W3_BLOCK;
    I.bias = o; o += 1024;
    I.b1 = o;   o += with_b1 ? (uint32_t)C::NP * nkc * T2_B1_CHUNK : 0u;
    I.total = o;
    return I;
}

enum { B2_FULL = 0, B2_EMPTY = 8, B2_D1_FULL = 16, B2_V_FREE = 18, B2_H1P = 20, B2_H1N = 22, B2_D2P = 24, B2_D2N = 26,
       B2_H2P = 28, B2_H2N = 30, B2_D3P = 32, B2_D3N = 34, B2_EPS_TX = 36, B2_EPS_READY, B2_EPS_FREE, B2_W_READY, B2_W_FREE,
       B2_IMG_READY, B2_IMG_FREE = B2_IMG_READY + 2, B2_COUNT = B2_IMG_FREE + 2 };
static_assert(B2_COUNT * 8 + 16 <= 1024, "barrier block too small");

// NOISE: the action-noise variant (loads of the noise array in the layer-3 epilogue); a separate instantiation so that the
// registers it holds across the accumulator wait do not cost the noise-free kernel anything (measured: +6 % when shared)
// EPIS (with NOISE): n_eps > 1 episodes per evaluation, act_noise [n_pairs][2][n_eps][T][act]; the layer-3 epilogue keeps the
// noise-free actions of its columns and adds every episode's noise row to them (the last episode drives the position)
template <bool SPLIT, bool NOISE, bool EPIS>
__global__ void __launch_bounds__(T2_THREADS, 1) rollout_tc2_kernel(const __grid_constant__ T2Params p,
                                                                     const __grid_constant__ T2Maps maps, int n_eps) {
    using C = T2Cfg<SPLIT>;
    constexpr int NP = C::NP, NST = C::NST;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const T2Smem L = t2_layout<SPLIT>(p.nkc);
    uint64_t* bars = (uint64_t*)(smem + L.bars);
    uint32_t* tmem_slot = (uint32_t*)(smem + L.bars + B2_COUNT * 8);
    float* bias_all = (float*)(smem + L.bias);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int NMT = p.n_mtiles, NKC = p.nkc;
    const int my_pairs = (p.n_pairs - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

    // ---- one-time setup -----------------------------------------------------------------------------------------------
    if (tid == 0) {
        ((unsigned*)(smem + L.red + 2 * T2_EPI_WARPS * 64))[0] = 0;
        ((unsigned*)(smem + L.red + 2 * T2_EPI_WARPS * 64))[1] = 0;
        for (int s = 0; s < NST; ++s) { mbar_init(&bars[B2_FULL + s], 1); mbar_init(&bars[B2_EMPTY + s], 1); }
        for (int gq = 0; gq < 2; ++gq) {
            mbar_init(&bars[B2_D1_FULL + gq], 1); mbar_init(&bars[B2_V_FREE + gq], C::GW);
            mbar_init(&bars[B2_H1P + gq], C::GW); mbar_init(&bars[B2_H1N + gq], C::GW);
            mbar_init(&bars[B2_H2P + gq], C::GW); mbar_init(&bars[B2_H2N + gq], C::GW);
            mbar_init(&bars[B2_D2P + gq], 1); mbar_init(&bars[B2_D2N + gq], 1);
            mbar_init(&bars[B2_D3P + gq], 1); mbar_init(&bars[B2_D3N + gq], 1);
        }
        mbar_init(&bars[B2_EPS_TX], 1); mbar_init(&bars[B2_EPS_READY], 1); mbar_init(&bars[B2_EPS_FREE], 1);
        mbar_init(&bars[B2_W_READY], 1); mbar_init(&bars[B2_W_FREE], 2);
        for (int b = 0; b < 2; ++b) { mbar_init(&bars[B2_IMG_READY + b], T2_BLD_WARPS); mbar_init(&bars[B2_IMG_FREE + b], 1); }
        fence_barrier_init();
    }
    __syncthreads();
    if (warp == T2_W_L1) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp < T2_EPI_WARP0) {
        reg_dec<T2_REG_MOVE>();
        if (warp == T2_W_PROD) {
            // ===================== producer: observation stages =====================
            if (lane == 0) {
                uint32_t stage = 0, phase = 0;
                const int per_tile = NKC * NP;
                for (int i = 0; i < my_pairs; ++i)
                    for (int m = 0; m < NMT; ++m)
                        for (int s = 0; s < per_tile; ++s) {
                            mbar_wait(&bars[B2_EMPTY + stage], phase ^ 1);
                            mbar_expect_tx(&bars[B2_FULL + stage], T2_STAGE);
                            bulk_g2s(smem + L.xst + stage * T2_STAGE, p.xnt + ((size_t)m * per_tile + s) * T2_STAGE, T2_STAGE,
                                     &bars[B2_FULL + stage]);
                            if (++stage == NST) { stage = 0; phase ^= 1; }
                        }
            }
        } else if (warp == T2_W_L1) {
            // ===================== L1 MMA issuer (warp-uniform loop; one elected lane issues) =====================
            const uint32_t id_l1 = umma_idesc_f16(T2_MT, T2_H), id_l1w = umma_idesc_f16(T2_MT, 2 * T2_H);
            const uint64_t a_desc0 = umma_desc_sw128(smem_u32(smem + L.xst)), b_desc0 = umma_desc_sw128(smem_u32(smem + L.b1));
            uint32_t stage = 0, phase = 0, g = 0;
            for (int i = 0; i < my_pairs; ++i) {
                mbar_wait(&bars[B2_EPS_READY], i & 1);
                for (int m = 0; m < NMT; ++m, ++g) {
                    const uint32_t grp = g & 1, use = g >> 1;
                    mbar_wait(&bars[B2_V_FREE + grp], (use & 1) ^ 1);              // the group is done with this V (and what aliases it)
                    tc_fence_after();
                    const uint32_t d_v = tmem + grp * C::V_STRIDE;        // V buffer of this tile (grp = g & 1)
                    for (int kc = 0; kc < NKC; ++kc) {
                        const uint64_t bd = b_desc0 + (uint64_t)kc * ((NP * T2_B1_CHUNK) >> 4);       // [kc][piece] blocks
                        if (!SPLIT) {
                            mbar_wait(&bars[B2_FULL + stage], phase);
                            tc_fence_after();
                            const uint64_t ad = a_desc0 + (uint64_t)stage * (T2_STAGE >> 4);
                            if (elect_one()) {
                                issue_ss4(d_v, ad, bd, id_l1, kc != 0);                      // x . eps
                                umma_commit(&bars[B2_EMPTY + stage]);
                                if (kc == NKC - 1) umma_commit(&bars[B2_D1_FULL + grp]);
                            }
                            __syncwarp();
                            if (++stage == NST) { stage = 0; phase ^= 1; }
                        } else {
                            // the x_hi and x_lo stages of the chunk are adjacent ring slots (NST even): one issue region for both
                            const uint32_t st_hi = stage, st_lo = stage + 1;
                            mbar_wait(&bars[B2_FULL + st_hi], phase);
                            mbar_wait(&bars[B2_FULL + st_lo], phase);
                            tc_fence_after();
                            const uint64_t ah = a_desc0 + (uint64_t)st_hi * (T2_STAGE >> 4), al = a_desc0 + (uint64_t)st_lo * (T2_STAGE >> 4);
                            if (elect_one()) {
                                issue_ss4(d_v, ah, bd, id_l1w, kc != 0);                     // x_hi . [eps_hi ; eps_lo]  (N = 128)
                                umma_commit(&bars[B2_EMPTY + st_hi]);
                                issue_ss4(d_v, al, bd, id_l1, 1);                            // x_lo . eps_hi           (N = 64, columns 0-63)
                                umma_commit(&bars[B2_EMPTY + st_lo]);
                                if (kc == NKC - 1) umma_commit(&bars[B2_D1_FULL + grp]);
                            }
                            __syncwarp();
                            stage += 2;
                            if (stage == NST) { stage = 0; phase ^= 1; }
                        }
                    }
                }
                if (elect_one()) umma_commit(&bars[B2_EPS_FREE]);                   // the pair's last L1 is in flight
                __syncwarp();
            }
        } else {
            // ===================== L2 / L3 MMA issuers =====================
            // !SPLIT: issuer w serves epilogue group w (its alternate tiles, both signs, + first).  SPLIT: issuer w serves sign w of
            // every tile.  Order per tile and sign: wait H1 -> L2 -> commit D2, wait H2 -> L3 -> commit D3.
            const uint32_t iw = warp - T2_W_L23;
            const uint32_t eg = SPLIT ? 0 : iw;
            const uint32_t id_l2 = umma_idesc_f16(T2_MT, T2_H), id_l3 = umma_idesc_f16(T2_MT, T2_ACT_PAD);
            const uint64_t w2d = umma_desc_sw128(smem_u32(smem + L.w2)), w3d = umma_desc_sw128(smem_u32(smem + L.w3));
            constexpr uint64_t W2_BLK = T2_B1_CHUNK >> 4, W3_BLK = T2_W3_BLOCK >> 4;     // [sign][piece] blocks
            const uint32_t tb = tmem + eg * C::G_STRIDE;
            uint32_t k = 0;
            for (int i = 0; i < my_pairs; ++i) {
                mbar_wait(&bars[B2_W_READY], i & 1);
                tc_fence_after();
                for (uint32_t g = (uint32_t)i * NMT; g < (uint32_t)(i + 1) * NMT; ++g) {
                    if (!SPLIT && (g & 1) != eg) continue;
                    const uint32_t par = k & 1;
                    ++k;
#pragma unroll 1
                    for (int step = 0; step < (SPLIT ? 2 : 4); ++step) {
                        // !SPLIT: (L2+, L2-, L3+, L3-); SPLIT: (L2 s, L3 s) with s = iw
                        const int layer = SPLIT ? step : (step >> 1), sgn = SPLIT ? (int)iw : (step & 1);
                        const int hb = layer ? (sgn ? B2_H2N : B2_H2P) : (sgn ? B2_H1N : B2_H1P);
                        const int db = layer ? (sgn ? B2_D3N : B2_D3P) : (sgn ? B2_D2N : B2_D2P);
                        mbar_wait(&bars[hb + eg], par);
                        tc_fence_after();
                        if (elect_one()) {
                            const uint32_t a_hi = tb + (sgn ? C::C_HN : C::C_HP), a_lo = a_hi + 32;
                            const uint32_t d = tb + (sgn ? C::C_D2N : C::C_D2P);          // D3 aliases D2
                            const uint64_t bh = layer ? w3d + (uint64_t)(sgn * NP) * W3_BLK : w2d + (uint64_t)(sgn * NP) * W2_BLK;
                            const uint64_t bl = bh + (layer ? W3_BLK : W2_BLK);
                            const uint32_t id = layer ? id_l3 : id_l2;
                            issue_ts4(d, a_hi, bh, id, 0);                               // h_hi . w_hi
                            if (SPLIT) {
                                issue_ts4(d, a_hi, bl, id, 1);                           // h_hi . w_lo
                                issue_ts4(d, a_lo, bh, id, 1);                           // h_lo . w_hi
                            }
                            umma_commit(&bars[db + eg]);
                        }
                        __syncwarp();
                    }
                }
                if (elect_one()) umma_commit(&bars[B2_W_FREE]);                     // this issuer's L2/L3 of the pair are in flight
                __syncwarp();
            }
        }
    } else if (warp < T2_BLD_WARP0) {
        // ===================== epilogue warps =====================
        reg_inc<T2_REG_EPI>();
        constexpr int CW = C::CW, NB = CW / 8;                // accumulator columns per warp (32 / 16), batches of 8 columns
        const int ew = warp - T2_EPI_WARP0;                   // 0..15
        const uint32_t eg = SPLIT ? 0u : (uint32_t)(ew >> 3); // epilogue group
        const int q = warp & 3;                               // TMEM lane quarter
        const int cq = SPLIT ? (ew >> 2) : ((ew & 7) >> 2);   // column part of this warp: columns [cq*CW, cq*CW + CW)
        const int row = q * 32 + lane;
        const uint32_t lane_off = (uint32_t)(q * 32) << 16;
        const uint32_t tb = tmem + eg * C::G_STRIDE + lane_off;           // H / D2 regions of the group
        // action columns of this warp (layer 3): [a_lo, a_hi), at most 16, multiples of 4 (!SPLIT: two parts, SPLIT: four parts)
        const int a_per = SPLIT ? ((p.act <= 16) ? 4 : 8) : ((p.act <= 24) ? 8 : 16);
        const int a_lo = cq * a_per;
        const int a_hi = (cq == (SPLIT ? 3 : 1)) ? p.act : min(p.act, a_lo + a_per);
        const int nj = max(0, a_hi - a_lo);                   // warp-uniform
        const float sg = p.sigma;
        const bool want_pos = p.behv_pos != nullptr;
        double* red = (double*)(smem + L.red);                // [pair parity][16 warps][8]: per-pair sums of every epilogue warp
        unsigned* red_cnt = (unsigned*)(smem + L.red + 2 * T2_EPI_WARPS * 64);
        for (int i = 0; i < my_pairs; ++i) {
            const uint32_t b2p = smem_u32(bias_all + (i & 1) * 256) + cq * CW * 4, b2n = b2p + T2_H * 4;
            const uint32_t b3p = smem_u32(bias_all + (i & 1) * 256) + 2 * T2_H * 4 + a_lo * 4, b3n = b3p + T2_ACT_PAD * 4;
            // this thread's rows of the pair: compensated float32 sums (Kahan; the reference sums python floats, float64)
            float fps = 0.f, fpc = 0.f, fns = 0.f, fnc = 0.f;
            float pacc = 0.f;                                 // position sums: ONE register (transposing butterfly per tile)
            for (uint32_t g = (uint32_t)i * NMT; g < (uint32_t)(i + 1) * NMT; ++g) {
                if (!SPLIT && (g & 1) != eg) continue;
                const uint32_t vbuf = g & 1, par_v = (g >> 1) & 1;                 // V buffer of the tile and its use count parity
                const uint32_t par = SPLIT ? (g & 1) : par_v;                      // use count parity of the group's H / D2 / D3 barriers
                const int m = (int)(g - (uint32_t)i * NMT);
                const int t = m * T2_MT + row;
                const uint32_t tv_ = tmem + vbuf * C::V_STRIDE + lane_off + cq * CW;            // this warp's V columns
                const float4* __restrict__ up = reinterpret_cast<const float4*>(p.ubase) + ((size_t)m * 16 + cq * (CW / 4)) * T2_MT + row;
                if (EPIS && cq == 0) {
                    // the noise rows of every episode of both signs ([sign][episode] blocks of T * act floats) towards L2
                    const int t0 = m * T2_MT + q * 32;
                    const int rows = min(32, p.T - t0);
                    if (rows > 0) {
                        const size_t blk = (size_t)p.T * p.act * 4;
                        const char* nb = reinterpret_cast<const char*>(p.act_noise + (((size_t)(blockIdx.x + i * gridDim.x) * 2 * n_eps) * p.T + t0) * p.act);
                        const int bytes = rows * p.act * 4;
                        for (int k = 0; k < 2 * n_eps; ++k)
                            for (int o = lane * 128; o < bytes + 128; o += 32 * 128) prefetch_l2(nb + k * blk + min(o, bytes - 4));
                    }
                } else if (NOISE && p.act_noise && cq == 0) {
                    // action noise of this tile's rows (both signs) towards L2 now; it is read after layer 3 (one warp per lane quarter asks)
                    const int t0 = m * T2_MT + q * 32;
                    const int rows = min(32, p.T - t0);
                    if (rows > 0) {
                        const char* nb = reinterpret_cast<const char*>(p.act_noise + (((size_t)(blockIdx.x + i * gridDim.x) * 2) * p.T + t0) * p.act);
                        const int bytes = rows * p.act * 4;
                        for (int o = lane * 128; o < bytes + 128; o += 32 * 128) {
                            prefetch_l2(nb + min(o, bytes - 4));
                            prefetch_l2(nb + (size_t)p.T * p.act * 4 + min(o, bytes - 4));
                        }
                    }
                }
                mbar_wait(&bars[B2_D1_FULL + vbuf], par_v);
                tc_fence_after();
                // ---- epi1: h1+- = tanh(U +- sigma V), 8 columns at a time; the + sign first (its L2 MMA then runs while the - sign
                //      is computed); U and V are read again for the - sign (SPLIT: V = the two partial sums of the wide accumulator)
#pragma unroll
                for (int sgn = 0; sgn < 2; ++sgn) {
                    const unsigned long long s2 = sgn ? pk(-sg, -sg) : pk(sg, sg);
#pragma unroll
                    for (int c4 = 0; c4 < NB; ++c4) {
                        float4 ub[2];
#pragma unroll
                        for (int c = 0; c < 2; ++c) ub[c] = ldg_stream4(up + (c4 * 2 + c) * T2_MT);
                        uint32_t v[8];
                        tmem_ld8(tv_ + c4 * 8, v);
                        if (SPLIT) {
                            uint32_t v2[8];
                            tmem_ld8(tv_ + 64 + c4 * 8, v2);
                            tmem_ld_wait();
#pragma unroll
                            for (int e = 0; e < 4; ++e) {
                                float s0, s1;
                                unpk(add2(pk(__uint_as_float(v[2 * e]), __uint_as_float(v[2 * e + 1])),
                                          pk(__uint_as_float(v2[2 * e]), __uint_as_float(v2[2 * e + 1]))), s0, s1);
                                v[2 * e] = __float_as_uint(s0); v[2 * e + 1] = __float_as_uint(s1);
                            }
                        } else {
                            tmem_ld_wait();
                        }
                        uint32_t whi[4], wlo[4];
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const float4 u4 = ub[e >> 1];
                            const float u0 = (e & 1) ? u4.z : u4.x, u1 = (e & 1) ? u4.w : u4.y;
                            float z0, z1, t0, t1;
                            unpk(fma2(pk(__uint_as_float(v[2 * e]), __uint_as_float(v[2 * e + 1])), s2, pk(u0, u1)), z0, z1);
                            if (SPLIT) { tanh_acc2(z0, z1, t0, t1, (T2_NEWTON_MASK >> e) & 1); split_h2(t0, t1, whi[e], wlo[e]); }
                            else { whi[e] = pack_h2(tanh_fast(z0), tanh_fast(z1)); }
                        }
                        const uint32_t hc = tb + (sgn ? C::C_HN : C::C_HP) + cq * (CW / 2) + c4 * 4;
                        tmem_st4(hc, whi[0], whi[1], whi[2], whi[3]);
                        if (SPLIT) tmem_st4(hc + 32, wlo[0], wlo[1], wlo[2], wlo[3]);
                    }
                    tmem_st_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) {
                        if (sgn == 0) mbar_arrive(&bars[B2_H1P + eg]);
                        else { mbar_arrive(&bars[B2_V_FREE + vbuf]); mbar_arrive(&bars[B2_H1N + eg]); }   // V consumed
                    }
                }
                if (m < 2) mbar_wait(&bars[B2_W_READY], i & 1);                    // first tile of the pair: biases in place?
                // ---- epi2 (+ then -): h2 = tanh(D2 + b2), over h1 ----
#pragma unroll
                for (int sgn = 0; sgn < 2; ++sgn) {
                    mbar_wait(&bars[(sgn ? B2_D2N : B2_D2P) + eg], par);
                    tc_fence_after();
                    const uint32_t b2 = sgn ? b2n : b2p;
#pragma unroll
                    for (int c4 = 0; c4 < NB; ++c4) {
                        uint32_t d[8];
                        tmem_ld8(tb + (sgn ? C::C_D2N : C::C_D2P) + cq * CW + c4 * 8, d);
                        const float4 bb0 = lds128f(b2 + c4 * 32), bb1 = lds128f(b2 + c4 * 32 + 16);
                        tmem_ld_wait();
                        const float bs[8] = {bb0.x, bb0.y, bb0.z, bb0.w, bb1.x, bb1.y, bb1.z, bb1.w};
                        uint32_t whi[4], wlo[4];
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            float z0, z1, t0, t1;
                            unpk(add2(pk(__uint_as_float(d[2 * e]), __uint_as_float(d[2 * e + 1])), pk(bs[2 * e], bs[2 * e + 1])), z0, z1);
                            if (SPLIT) { tanh_acc2(z0, z1, t0, t1, (T2_NEWTON_MASK >> e) & 1); split_h2(t0, t1, whi[e], wlo[e]); }
                            else { whi[e] = pack_h2(tanh_fast(z0), tanh_fast(z1)); }
                        }
                        const uint32_t hc = tb + (sgn ? C::C_HN : C::C_HP) + cq * (CW / 2) + c4 * 4;
                        tmem_st4(hc, whi[0], whi[1], whi[2], whi[3]);
                        if (SPLIT) tmem_st4(hc + 32, wlo[0], wlo[1], wlo[2], wlo[3]);
                    }
                    tmem_st_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&bars[(sgn ? B2_H2N : B2_H2P) + eg]);
                }
                // ---- epi3 (+ then -): a = tanh(D3 + b3); reward and position ----
                const float* __restrict__ ccol = p.crt + ((size_t)m * T2_ACT_PAD + a_lo) * T2_MT + row;
                float cc[16];
#pragma unroll
                for (int jj = 0; jj < 16; ++jj) cc[jj] = (jj < nj) ? ldg_pinned(ccol + jj * T2_MT) : 0.f;
                // this row's action noise of the + evaluation, columns a_lo.. (the - evaluation: T * act further)
                const float* nzrow = (NOISE && p.act_noise && t < p.T)
                    ? p.act_noise + (((size_t)(blockIdx.x + i * gridDim.x) * 2) * p.T + t) * p.act + a_lo : nullptr;
                float tv[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                if (EPIS) {
#pragma unroll
                    for (int sgn = 0; sgn < 2; ++sgn) {
                        mbar_wait(&bars[(sgn ? B2_D3N : B2_D3P) + eg], par);
                        tc_fence_after();
                        // a = tanh(D3 + b3) of this warp's columns, noise-free (padded columns: tanh(0), zero reward coefficient)
                        float av[16];
#pragma unroll
                        for (int jj = 0; jj < 16; ++jj) av[jj] = 0.f;
                        if (nj > 0) {
                            const uint32_t b3 = sgn ? b3n : b3p;
#pragma unroll
                            for (int hf = 0; hf < 2; ++hf) {
                                if (hf * 8 < nj) {
                                    uint32_t d[8];
                                    tmem_ld8(tb + (sgn ? C::C_D2N : C::C_D2P) + a_lo + hf * 8, d);      // D3 aliases D2
                                    tmem_ld_wait();
#pragma unroll
                                    for (int g4 = 0; g4 < 2; ++g4) {
                                        const int gq = hf * 2 + g4;
                                        if (gq * 4 < nj) {
                                            const float4 bb = lds128f(b3 + gq * 16);
                                            const float z0 = __uint_as_float(d[g4 * 4 + 0]) + bb.x, z1 = __uint_as_float(d[g4 * 4 + 1]) + bb.y;
                                            const float z2 = __uint_as_float(d[g4 * 4 + 2]) + bb.z, z3 = __uint_as_float(d[g4 * 4 + 3]) + bb.w;
                                            float* a4 = av + gq * 4;
                                            if (SPLIT) { tanh_acc2(z0, z1, a4[0], a4[1], (T2_NEWTON_MASK >> 0) & 1); tanh_acc2(z2, z3, a4[2], a4[3], (T2_NEWTON_MASK >> 1) & 1); }
                                            else { a4[0] = tanh_fast(z0); a4[1] = tanh_fast(z1); a4[2] = tanh_fast(z2); a4[3] = tanh_fast(z3); }
                                        }
                                    }
                                }
                            }
                        }
                        tc_fence_before();
                        if (t < p.T && nj > 0) {
                            // episode e's noise row of this step and sign, columns a_lo..: obj.py's episode loop, one reward sum
                            const float* __restrict__ ns =
                                p.act_noise + ((((size_t)(blockIdx.x + i * gridDim.x) * 2 + sgn) * n_eps) * p.T + t) * p.act + a_lo;
                            float r = 0.f, q0 = 0.f, q1 = 0.f, q2 = 0.f;
                            for (int e = 0; e < n_eps; ++e) {
                                const float* __restrict__ ne = ns + (size_t)e * p.T * p.act;
                                float ae[16];
#pragma unroll
                                for (int jj = 0; jj < 16; ++jj) ae[jj] = av[jj] + ((jj < nj) ? ldg_pinned(ne + jj) : 0.f);
#pragma unroll
                                for (int jj = 0; jj < 16; ++jj) r = fmaf(ae[jj], cc[jj], r);
                                q0 = ae[0]; q1 = (p.act > 1) ? ae[1] : ae[0]; q2 = (p.act > 2) ? ae[2] : ae[0];
                            }
                            // Kahan step: (s, c) += r
                            if (sgn) { const float y = r - fnc, u = fns + y; fnc = (u - fns) - y; fns = u; tv[5] = q0; tv[6] = q1; tv[7] = q2; }
                            else     { const float y = r - fpc, u = fps + y; fpc = (u - fps) - y; fps = u; tv[2] = q0; tv[3] = q1; tv[4] = q2; }
                        }
                    }
                    if (want_pos && cq == 0) pacc += warp_sum8(tv, lane);
                    continue;
                }
                // the noise values of a sign are in flight before that sign's accumulator is waited for (the - sign's under the
                // + sign's arithmetic): read inside the tanh groups they cost several exposed memory latencies per tile
                constexpr int NZ = NOISE ? (SPLIT ? 8 : 16) : 1;
                float nz[2][NZ];
                if (NOISE) {
#pragma unroll
                    for (int jj = 0; jj < NZ; ++jj) nz[0][jj] = (nzrow && jj < nj) ? ldg_pinned(nzrow + jj) : 0.f;
                }
#pragma unroll
                for (int sgn = 0; sgn < 2; ++sgn) {
                    if (NOISE && sgn == 0) {
#pragma unroll
                        for (int jj = 0; jj < NZ; ++jj) nz[1][jj] = (nzrow && jj < nj) ? ldg_pinned(nzrow + (size_t)p.T * p.act + jj) : 0.f;
                    }
                    mbar_wait(&bars[(sgn ? B2_D3N : B2_D3P) + eg], par);
                    tc_fence_after();
                    float r = 0.f, q0 = 0.f, q1 = 0.f, q2 = 0.f;
                    if (nj > 0) {
                        const uint32_t b3 = sgn ? b3n : b3p;
#pragma unroll
                        for (int hf = 0; hf < 2; ++hf) {
                            if (hf * 8 < nj) {
                                uint32_t d[8];
                                tmem_ld8(tb + (sgn ? C::C_D2N : C::C_D2P) + a_lo + hf * 8, d);      // D3 aliases D2
                                tmem_ld_wait();
#pragma unroll
                                for (int g4 = 0; g4 < 2; ++g4) {
                                    const int gq = hf * 2 + g4;
                                    if (gq * 4 < nj) {
                                        // padded columns: zero weights, zero bias, zero reward coefficient -> tanh(0) * 0
                                        const float4 bb = lds128f(b3 + gq * 16);
                                        const float z0 = __uint_as_float(d[g4 * 4 + 0]) + bb.x, z1 = __uint_as_float(d[g4 * 4 + 1]) + bb.y;
                                        const float z2 = __uint_as_float(d[g4 * 4 + 2]) + bb.z, z3 = __uint_as_float(d[g4 * 4 + 3]) + bb.w;
                                        float a0, a1, a2, a3;
                                        if (SPLIT) { tanh_acc2(z0, z1, a0, a1, (T2_NEWTON_MASK >> 0) & 1); tanh_acc2(z2, z3, a2, a3, (T2_NEWTON_MASK >> 1) & 1); }
                                        else { a0 = tanh_fast(z0); a1 = tanh_fast(z1); a2 = tanh_fast(z2); a3 = tanh_fast(z3); }
                                        if (NOISE && gq * 4 < NZ) {        // a += rs.randn(act) * ac_std (src/nn/nn.py:47-48), drawn by mt_gauss.cu
                                            a0 += nz[sgn][(gq * 4 + 0) % NZ]; a1 += nz[sgn][(gq * 4 + 1) % NZ];
                                            a2 += nz[sgn][(gq * 4 + 2) % NZ]; a3 += nz[sgn][(gq * 4 + 3) % NZ];
                                        }
                                        r = fmaf(a0, cc[gq * 4 + 0], r);
                                        r = fmaf(a1, cc[gq * 4 + 1], r);
                                        r = fmaf(a2, cc[gq * 4 + 2], r);
                                        r = fmaf(a3, cc[gq * 4 + 3], r);
                                        if (gq == 0 && cq == 0) {          // position integrator: action components 0, 1 % act, 2 % act
                                            q0 = a0;
                                            q1 = (p.act > 1) ? a1 : a0;
                                            q2 = (p.act > 2) ? a2 : a0;
                                        }
                                    }
                                }
                            }
                        }
                    }
                    if (t < p.T) {
                        // Kahan step: (s, c) += r
                        if (sgn) { const float y = r - fnc, u = fns + y; fnc = (u - fns) - y; fns = u; tv[5] = q0; tv[6] = q1; tv[7] = q2; }
                        else     { const float y = r - fpc, u = fps + y; fpc = (u - fps) - y; fps = u; tv[2] = q0; tv[3] = q1; tv[4] = q2; }
                    }
                }
                tc_fence_before();
                if (want_pos && cq == 0) pacc += warp_sum8(tv, lane);
            }
            // ---- this warp's sums of the pair -> shared memory; the last of the 16 warps adds them in warp order and writes the pair's
            //      results (no global scratch, no device-wide fence: a CTA-scope release/acquire on a shared counter) ----
            const int pair = blockIdx.x + i * gridDim.x;
            const double fitp = warp_sum_d((double)fps - (double)fpc), fitn = warp_sum_d((double)fns - (double)fnc);
            double* mine = red + ((size_t)(i & 1) * T2_EPI_WARPS + ew) * 8;
            if (lane == 0) { mine[0] = fitp; mine[1] = fitn; }
            if (want_pos && (lane & 3) == 0) reinterpret_cast<float*>(mine + 2)[sum8_index(lane)] = pacc;
            __syncwarp();
            if (lane == 0) {
                __threadfence_block();
                // monotonic arrival counter per parity slot (pairs i, i+2, ... share one: no warp can be a whole pair ahead)
                if (atomicAdd(red_cnt + (i & 1), 1u) == (unsigned)(T2_EPI_WARPS * ((i >> 1) + 1) - 1)) {
                    __threadfence_block();
                    double fp = 0.0, fn = 0.0;
                    float tot[8];
#pragma unroll
                    for (int kk = 0; kk < 8; ++kk) tot[kk] = 0.f;
                    const volatile double* all = red + (size_t)(i & 1) * T2_EPI_WARPS * 8;
                    for (int w = 0; w < T2_EPI_WARPS; ++w) {
                        fp += all[w * 8 + 0]; fn += all[w * 8 + 1];
                        if (want_pos && (SPLIT ? (w >> 2) : ((w & 7) >> 2)) == 0) {
                            const volatile float* pf = reinterpret_cast<const volatile float*>(all + w * 8 + 2);
#pragma unroll
                            for (int kk = 2; kk < 8; ++kk) tot[kk] += pf[kk];
                        }
                    }
                    if (EPIS) { fp /= n_eps; fn /= n_eps; }                         // obj.py: rews /= max(1, eps_per_policy)
                    p.fit_pos[(size_t)pair * p.fit_stride] = fp;
                    p.fit_neg[(size_t)pair * p.fit_stride] = fn;
                    if (want_pos) {
                        p.behv_pos[pair * 3 + 0] = p.pos_scale * tot[2]; p.behv_pos[pair * 3 + 1] = p.pos_scale * tot[3];
                        p.behv_pos[pair * 3 + 2] = p.pos_scale * tot[4];
                        p.behv_neg[pair * 3 + 0] = p.pos_scale * tot[5]; p.behv_neg[pair * 3 + 1] = p.pos_scale * tot[6];
                        p.behv_neg[pair * 3 + 2] = p.pos_scale * tot[7];
                    }
                }
            }
        }
    } else {
      reg_dec<T2_REG_BUILD>();            // warps 20-27 (two whole warpgroups) execute the same instruction
      if (warp == T2_W_COPY) {
        // ===================== copier: eps1 by TMA from the shadows (or from the image), W2/W3/bias from the image =====================
        const T2Image I = t2_image<SPLIT>(NKC, !p.use_tma);
        const uint8_t* my_images = p.images + (size_t)blockIdx.x * 2 * I.total;
        const uint32_t w_bytes = 2u * NP * (T2_B1_CHUNK + T2_W3_BLOCK);
        for (int i = 0; i < my_pairs; ++i) {
            const uint32_t b = i & 1, u = i >> 1;
            const uint8_t* img = my_images + (size_t)b * I.total;
            const int pair = blockIdx.x + i * gridDim.x;
            const long long slice = es_checked_slice(p.idx[pair], p.P, p.table_len, p.err);
            mbar_wait(&bars[B2_IMG_READY + b], u & 1);                             // builders have finished image i
            if (i > 0) mbar_wait(&bars[B2_EPS_FREE], (i - 1) & 1);                 // previous pair's last L1 has retired
            if (lane == 0) {
                mbar_expect_tx(&bars[B2_EPS_TX], (uint32_t)(NP * NKC * T2_B1_CHUNK));
                if (p.use_tma) {
                    const long long at = slice + p.w1;
                    const int unit0 = (int)(((long long)(at & 7) * (long long)p.shadow_stride + (at - (at & 7))) >> 3);
#pragma unroll
                    for (int pc = 0; pc < NP; ++pc)
                        for (int kc = 0; kc < NKC; ++kc)
                            tma_load_3d(smem + L.b1 + (size_t)(kc * NP + pc) * T2_B1_CHUNK, pc ? &maps.lo : &maps.hi, 0, unit0 + 8 * kc, 0,
                                        &bars[B2_EPS_TX]);
                } else {
                    for (int c = 0; c < NP * NKC; ++c)
                        bulk_g2s(smem + L.b1 + (size_t)c * T2_B1_CHUNK, img + I.b1 + (size_t)c * T2_B1_CHUNK, T2_B1_CHUNK, &bars[B2_EPS_TX]);
                }
            }
            mbar_wait(&bars[B2_EPS_TX], i & 1);
            if (p.use_tma) {
                // the unit holding column `obs` received the first elements of the next row: it carries the bias element
                // eps_b1[n] (the observation tile has a constant 1 there) and zeros (obs % 8 == 0 on this path)
                const int kcb = p.obs >> 6, ub = (p.obs & 63) >> 3;
#pragma unroll
                for (int rr = 0; rr < 2; ++rr) {
                    const int n = 2 * lane + rr;
                    const float eb = ldg_stream(p.table + slice + p.b1 + n);
                    __half hi, lo;
                    split_h1(eb, hi, lo);
                    const uint32_t off = (uint32_t)(kcb * NP) * T2_B1_CHUNK + n * 128 + ((ub ^ (n & 7)) << 4);      // [kc][piece] blocks
                    *(uint4*)(smem + L.b1 + off) = make_uint4((uint32_t)__half_as_ushort(hi), 0, 0, 0);
                    if (SPLIT) *(uint4*)(smem + L.b1 + T2_B1_CHUNK + off) = make_uint4((uint32_t)__half_as_ushort(lo), 0, 0, 0);
                }
                fence_async_smem();
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars[B2_EPS_READY]);
            if (i > 0) mbar_wait(&bars[B2_W_FREE], (i - 1) & 1);                   // previous pair's last L3 has retired
            if (lane == 0) {
                mbar_expect_tx(&bars[B2_W_READY], w_bytes + 1024);
                bulk_g2s(smem + L.w2, img + I.w2, w_bytes, &bars[B2_W_READY]);     // W2 [sign][piece], W3 [sign][piece]: contiguous in both
                bulk_g2s((uint8_t*)bias_all + (i & 1) * 1024, img + I.bias, 1024, &bars[B2_W_READY]);
            }
            mbar_wait(&bars[B2_W_READY], i & 1);                                   // landed: the image slot may be rewritten
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars[B2_IMG_FREE + b]);
        }
      } else {
        // ===================== builder warps: W2+-, W3+-, biases (and eps1 without the shadows) one pair ahead =====================
        const int bw = warp - T2_BLD_WARP0, btid = tid - T2_BLD_WARP0 * 32;
        constexpr int BT = T2_BLD_WARPS * 32;
        const T2Image I = t2_image<SPLIT>(NKC, !p.use_tma);
        uint8_t* my_images = p.images + (size_t)blockIdx.x * 2 * I.total;
        const float sg = p.sigma;
        for (int j = 0; j < my_pairs; ++j) {
            const int pair = blockIdx.x + j * gridDim.x;
            mbar_wait(&bars[B2_IMG_FREE + (j & 1)], (((uint32_t)j >> 1) & 1) ^ 1);
            const long long slice = es_checked_slice(p.idx[pair], p.P, p.table_len, nullptr);
            const float* __restrict__ eps = p.table + slice;
            uint8_t* img = my_images + (size_t)(j & 1) * I.total;
            // W2+- / W3+-: element pairs (n, k), (n, k+1); theta +- sigma*eps with the reference's two roundings
            const int n2 = T2_H * T2_H / 2, n3 = T2_ACT_PAD * T2_H / 2;
            for (int e2 = btid; e2 < n2 + n3; e2 += BT) {
                const bool l3 = e2 >= n2;
                const int k2 = 2 * (l3 ? e2 - n2 : e2);
                const int n = k2 >> 6, kk = k2 & 63;
                const int off = (l3 ? p.w3 : p.w2) + k2;
                const bool live = !l3 || n < p.act;
                float wp0 = 0.f, wp1 = 0.f, wn0 = 0.f, wn1 = 0.f;
                if (live) {
                    const float d0 = __fmul_rn(sg, ldg_stream(eps + off)), d1 = __fmul_rn(sg, ldg_stream(eps + off + 1));
                    const float t0 = __ldg(p.theta + off), t1 = __ldg(p.theta + off + 1);
                    wp0 = __fadd_rn(t0, d0); wp1 = __fadd_rn(t1, d1); wn0 = __fadd_rn(t0, -d0); wn1 = __fadd_rn(t1, -d1);
                }
                const uint32_t blk = l3 ? T2_W3_BLOCK : T2_B1_CHUNK;
                uint8_t* base = img + (l3 ? I.w3 : I.w2) + sw128_off(n, kk);
                if (SPLIT) {
                    __half h0, l0, h1, l1;
                    split_h1(wp0, h0, l0); split_h1(wp1, h1, l1);
                    *(uint32_t*)(base + 0 * blk) = (uint32_t)__half_as_ushort(h0) | ((uint32_t)__half_as_ushort(h1) << 16);
                    *(uint32_t*)(base + 1 * blk) = (uint32_t)__half_as_ushort(l0) | ((uint32_t)__half_as_ushort(l1) << 16);
                    split_h1(wn0, h0, l0); split_h1(wn1, h1, l1);
                    *(uint32_t*)(base + 2 * blk) = (uint32_t)__half_as_ushort(h0) | ((uint32_t)__half_as_ushort(h1) << 16);
                    *(uint32_t*)(base + 3 * blk) = (uint32_t)__half_as_ushort(l0) | ((uint32_t)__half_as_ushort(l1) << 16);
                } else {
                    *(uint32_t*)(base + 0 * blk) = pack_h2(wp0, wp1);
                    *(uint32_t*)(base + 1 * blk) = pack_h2(wn0, wn1);
                }
            }
            {
                float* bias = (float*)(img + I.bias);
                if (btid < T2_H) {
                    const float d = __fmul_rn(sg, ldg_stream(eps + p.b2 + btid)), t = __ldg(p.theta + p.b2 + btid);
                    bias[btid] = __fadd_rn(t, d); bias[T2_H + btid] = __fadd_rn(t, -d);
                } else if (btid - T2_H < T2_ACT_PAD) {
                    const int j2 = btid - T2_H;
                    float vp = 0.f, vn = 0.f;
                    if (j2 < p.act) {
                        const float d = __fmul_rn(sg, ldg_stream(eps + p.b3 + j2)), t = __ldg(p.theta + p.b3 + j2);
                        vp = __fadd_rn(t, d); vn = __fadd_rn(t, -d);
                    }
                    bias[2 * T2_H + j2] = vp; bias[2 * T2_H + T2_ACT_PAD + j2] = vn;
                }
            }
            if (!p.use_tma) {
                // eps1 (unscaled) converted from the float32 slice: rows of 64, K padded to nkc*64, column `obs` = eps_b1
                const int Kp = NKC * T2_KC;
                for (int e2 = btid; e2 < T2_H * Kp / 2; e2 += BT) {
                    const int n = (2 * e2) / Kp, k = (2 * e2) - n * Kp;
                    float x0 = 0.f, x1 = 0.f;
                    if (k < p.obs) x0 = ldg_stream(eps + p.w1 + (size_t)n * p.obs + k); else if (k == p.obs) x0 = ldg_stream(eps + p.b1 + n);
                    if (k + 1 < p.obs) x1 = ldg_stream(eps + p.w1 + (size_t)n * p.obs + k + 1); else if (k + 1 == p.obs) x1 = ldg_stream(eps + p.b1 + n);
                    uint8_t* dst = img + I.b1 + (size_t)((k >> 6) * NP) * T2_B1_CHUNK + sw128_off(n, k & 63);     // [kc][piece] blocks
                    if (SPLIT) {
                        __half h0, l0, h1, l1;
                        split_h1(x0, h0, l0); split_h1(x1, h1, l1);
                        *(uint32_t*)dst = (uint32_t)__half_as_ushort(h0) | ((uint32_t)__half_as_ushort(h1) << 16);
                        *(uint32_t*)(dst + T2_B1_CHUNK) = (uint32_t)__half_as_ushort(l0) | ((uint32_t)__half_as_ushort(l1) << 16);
                    } else {
                        *(uint32_t*)dst = pack_h2(x0, x1);
                    }
                }
            }
            __threadfence();                                             // image visible device-wide (L2)
            asm volatile("fence.proxy.async;" ::: "memory");             // ... and to the async proxy that will copy it
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars[B2_IMG_READY + (j & 1)]);
            if (j + 1 < my_pairs) {                                      // L2 prefetch of the next pair's operands
                const long long nidx = es_checked_slice(p.idx[blockIdx.x + (j + 1) * gridDim.x], p.P, p.table_len, nullptr);
                const char* nxt = (const char*)(p.table + nidx);
                const int lines = (p.b3 + p.act) * 4 / 128 + 2;
                if (p.use_tma) {
                    const int skip = p.b1 * 4 / 128;                     // eps1 comes from the shadows
                    for (int l = skip + btid; l < lines; l += BT) prefetch_l2(nxt + (size_t)l * 128);
                } else {
                    for (int l = btid; l < lines; l += BT) prefetch_l2(nxt + (size_t)l * 128);
                }
            }
            (void)bw;
        }
      }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == T2_W_L1) tmem_dealloc(tmem, 512);
}

// U[t][n] = b1[n] + sum_k Xn[t][k] * theta1[n][k], accumulated in float64 (k ascending) and rounded once to float32.
// Output layout (float index): (((m*2 + h)*8 + c)*128 + row)*4 + e  for column n = 32h + 4c + e, t = 128m + row.
constexpr int T2_UB_ROWS = 8, T2_UB_KT = 64, T2_UB_RPT = T2_UB_ROWS / 4;
__global__ void __launch_bounds__(256) rollout_tc2_ubase_kernel(const float* __restrict__ obsn, const float* __restrict__ theta,
                                                                 int w1, int b1, int T, int obs, float* __restrict__ ubase) {
    __shared__ float s_w[T2_UB_KT][T2_H + 1];
    __shared__ float s_x[T2_UB_ROWS][T2_UB_KT];
    const int n = threadIdx.x & 63, rg = threadIdx.x >> 6;
    const int t0 = blockIdx.x * T2_UB_ROWS;
    double acc[T2_UB_RPT];
#pragma unroll
    for (int r = 0; r < T2_UB_RPT; ++r) acc[r] = (double)__ldg(theta + b1 + n);
    for (int k0 = 0; k0 < obs; k0 += T2_UB_KT) {
        const int kn = min(T2_UB_KT, obs - k0);
        for (int i = threadIdx.x; i < T2_H * T2_UB_KT; i += 256) {
            const int nn = i / T2_UB_KT, kk = i - nn * T2_UB_KT;
            s_w[kk][nn] = (kk < kn) ? __ldg(theta + w1 + (size_t)nn * obs + k0 + kk) : 0.f;
        }
        for (int i = threadIdx.x; i < T2_UB_ROWS * T2_UB_KT; i += 256) {
            const int r = i / T2_UB_KT, kk = i - r * T2_UB_KT;
            const int t = t0 + r;
            s_x[r][kk] = (kk < kn && t < T) ? obsn[(size_t)t * obs + k0 + kk] : 0.f;
        }
        __syncthreads();
        for (int kk = 0; kk < kn; ++kk) {
            const double w = (double)s_w[kk][n];
#pragma unroll
            for (int r = 0; r < T2_UB_RPT; ++r) acc[r] = fma((double)s_x[rg * T2_UB_RPT + r][kk], w, acc[r]);
        }
        __syncthreads();
    }
    const int h = n >> 5, c = (n & 31) >> 2, e = n & 3;
#pragma unroll
    for (int r = 0; r < T2_UB_RPT; ++r) {
        const int t = t0 + rg * T2_UB_RPT + r;
        const int m = t / T2_MT, row = t % T2_MT;
        ubase[(((size_t)(m * 2 + h) * 8 + c) * T2_MT + row) * 4 + e] = (t < T) ? (float)acc[r] : 0.f;
    }
}

// float16 shadows of the table: copy s, element j = f16(table[j + s]) (hi) / f16(table[j+s] - hi) (lo); zero beyond the end
__global__ void rollout_tc2_shadow_kernel(const float* __restrict__ table, int64_t len, size_t stride, __half* __restrict__ hi,
                                          __half* __restrict__ lo) {
    const size_t total = stride / 2;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int s = blockIdx.y;
        const int64_t j = (int64_t)(2 * i) + s;
        const float a = (j < len) ? __ldg(table + j) : 0.f, b = (j + 1 < len) ? __ldg(table + j + 1) : 0.f;
        __half ah, al, bh, bl;
        split_h1(a, ah, al); split_h1(b, bh, bl);
        *(__half2*)(hi + (size_t)s * stride + 2 * i) = __halves2half2(ah, bh);
        if (lo) *(__half2*)(lo + (size_t)s * stride + 2 * i) = __halves2half2(al, bl);
    }
}

// reward vectors transposed per tile: crt[(m*32 + j)*128 + row] = rew_vec[128m + row][j] (0 beyond T / act)
__global__ void rollout_tc2_crt_kernel(const float* __restrict__ rew_vec, int T, int act, int n_mtiles, float* __restrict__ crt) {
    const int total = n_mtiles * T2_ACT_PAD * T2_MT;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int row = i % T2_MT, j = (i / T2_MT) % T2_ACT_PAD, m = i / (T2_MT * T2_ACT_PAD);
        const int t = m * T2_MT + row;
        crt[i] = (t < T && j < act) ? rew_vec[(size_t)t * act + j] : 0.f;
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// 3-D map over a shadow allocation of 8 x stride float16: {64 elements, origin in 16-byte units (stride 16 B), 64 rows (stride
// obs*2 B)}; box {64, 1, 64} with the 128-byte swizzle = one K chunk of eps1 in the K-major operand layout
int t2_encode_map(CUtensorMap* map, void* base, size_t stride, int obs) {
    static EncodeTiledFn encode = nullptr;
    if (!encode) {
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", (void**)&encode, cudaEnableDefault, &qres) != cudaSuccess || !encode) {
            (void)cudaGetLastError();
            encode = nullptr;
            return -1;
        }
    }
    const cuuint64_t gdim[3] = {64, (cuuint64_t)stride /* = 8*stride/8 units */, 64};
    const cuuint64_t gstr[2] = {16, (cuuint64_t)obs * 2};
    const cuuint32_t box[3] = {64, 1, 64}, estr[3] = {1, 1, 1};
    return encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS ? 0 : -1;
}

template <bool SPLIT>
int t2_launch(es_ctx* ctx, T2Params& p, const T2Maps& maps, const float* obsn, const float* rew_vec, const float* theta, int T,
              int n_pairs, int n_eps, cudaStream_t stream) {
    const T2Smem L = t2_layout<SPLIT>(p.nkc);
    const size_t smem = (size_t)L.total + 1024;       // + alignment slack
    if (smem > 227 * 1024) {
        es_set_error("es_rollout_openloop(TC%s): obs_dim %d needs %zu bytes of shared memory (> 227 KB)", SPLIT ? "3" : "", p.obs, smem);
        return ES_ERR_UNSUPPORTED;
    }
    constexpr int NP = SPLIT ? 2 : 1;
    const size_t xnt_bytes = (size_t)p.n_mtiles * p.nkc * NP * T2_STAGE;
    const size_t ub_bytes = (size_t)p.n_mtiles * T2_MT * T2_H * sizeof(float);
    const size_t crt_bytes = (size_t)p.n_mtiles * T2_ACT_PAD * T2_MT * sizeof(float);
    const int grid = n_pairs < ctx->sm_count ? n_pairs : ctx->sm_count;
    const size_t img_bytes = (((size_t)grid * 2 * t2_image<SPLIT>(p.nkc, !p.use_tma).total) + 255) & ~(size_t)255;
    void* scratch = nullptr;
    int rc = es_ctx_scratch(ctx, xnt_bytes + ub_bytes + crt_bytes + img_bytes, &scratch);
    if (rc) return rc;
    char* at = (char*)scratch;
    uint8_t* xnt = (uint8_t*)at; at += xnt_bytes;
    float* ubase = (float*)at; at += ub_bytes;
    float* crt = (float*)at; at += crt_bytes;
    p.images = (uint8_t*)at;
    p.xnt = xnt; p.ubase = ubase; p.crt = crt;
    {
        const size_t total = (size_t)p.n_mtiles * p.nkc * T2_MT * T2_KC;
        int blocks = es_div_up((int64_t)total, 256);
        if (blocks > ctx->sm_count * 8) blocks = ctx->sm_count * 8;
        rollout_tc2_prep_kernel<SPLIT><<<blocks, 256, 0, stream>>>(obsn, T, p.obs, p.nkc, p.n_mtiles, xnt);
        ES_LAUNCHED(ctx);
        rollout_tc2_ubase_kernel<<<p.n_mtiles * T2_MT / T2_UB_ROWS, 256, 0, stream>>>(obsn, theta, p.w1, p.b1, T, p.obs, ubase);
        ES_LAUNCHED(ctx);
        rollout_tc2_crt_kernel<<<es_div_up(p.n_mtiles * T2_ACT_PAD * T2_MT, 256), 256, 0, stream>>>(rew_vec, T, p.act, p.n_mtiles, crt);
        ES_LAUNCHED(ctx);
    }
    auto kernel = !p.act_noise ? rollout_tc2_kernel<SPLIT, false, false>
                               : (n_eps > 1 ? rollout_tc2_kernel<SPLIT, true, true> : rollout_tc2_kernel<SPLIT, true, false>);
    ES_CHECK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kernel<<<grid, T2_THREADS, smem, stream>>>(p, maps, n_eps);
    ES_LAUNCHED(ctx);
    return ES_OK;
}

}  // namespace

void es_tc2_free_shadows(es_ctx* ctx) {
    if (ctx->sh16_hi) cudaFree(ctx->sh16_hi);
    if (ctx->sh16_lo) cudaFree(ctx->sh16_lo);
    if (ctx->sh16_maps) free(ctx->sh16_maps);
    ctx->sh16_hi = ctx->sh16_lo = nullptr;
    ctx->sh16_maps = nullptr;
    ctx->sh16_src = nullptr;
}

int es_impl_rollout_tc2(es_ctx* ctx, int split, const float* table, int64_t table_len, const int64_t* idx, int n_pairs,
                        const float* theta, int P, float sigma, const int* layer_sizes, int n_layers, const float* obsn,
                        const float* rew_vec, int T, float pos_scale, double* fit_pos, double* fit_neg, int fit_stride,
                        float* behv_pos, float* behv_neg, const float* act_noise, int n_eps, cudaStream_t stream) {
    if (n_layers != 3 || layer_sizes[1] != T2_H || layer_sizes[2] != T2_H || layer_sizes[3] > T2_ACT_PAD || layer_sizes[0] > 1023) {
        es_set_error("es_rollout_openloop(TC): the tensor-core path covers obs(<=1023)-64-64-act(<=32) tanh MLPs; "
                     "use ES_ROLLOUT_F32 for other shapes");
        return ES_ERR_UNSUPPORTED;
    }
    T2Params p;
    memset(&p, 0, sizeof(p));
    p.table = table; p.idx = idx; p.theta = theta; p.act_noise = act_noise;
    p.fit_pos = fit_pos; p.fit_neg = fit_neg; p.behv_pos = behv_pos; p.behv_neg = behv_neg;
    p.n_pairs = n_pairs; p.obs = layer_sizes[0]; p.act = layer_sizes[3]; p.T = T; p.fit_stride = fit_stride;
    p.sigma = sigma; p.pos_scale = pos_scale;
    p.nkc = es_div_up(p.obs + 1, T2_KC);                 // + the constant-1 column that carries the L1 bias
    p.n_mtiles = es_div_up(T, T2_MT);
    p.w1 = 0; p.b1 = p.obs * T2_H; p.w2 = p.b1 + T2_H; p.b2 = p.w2 + T2_H * T2_H; p.w3 = p.b2 + T2_H;
    p.b3 = p.w3 + T2_H * p.act;
    p.table_len = table_len; p.P = P; p.err = ctx->err_dev;

    // float16 shadows of the table (hi always, lo when a split rollout asks for it): 8 shifted copies each, built once per
    // (table pointer, length) and addressed through two TMA tensor maps.  Needs 16-byte aligned rows in every slice (obs % 8
    // == 0).  Without them (other shapes, no memory, no driver entry point) the builder warps convert the float32 slice.
    T2Maps maps;
    memset(&maps, 0, sizeof(maps));
    p.use_tma = 0;
    if (p.obs % 8 == 0 && !getenv("ES_TC_NO_SHADOW") && !ctx->sh16_failed) {
        const size_t stride = ((size_t)table_len + 64 * (size_t)p.obs + 79) & ~(size_t)7;       // room for the last slice's rows
        const bool fresh = ctx->sh16_src != table || ctx->sh16_len != table_len || ctx->sh16_stride != stride || ctx->sh16_obs != p.obs;
        if (fresh) es_tc2_free_shadows(ctx);
        bool ok = true;
        if (!ctx->sh16_hi) {
            ok = cudaMalloc(&ctx->sh16_hi, 8 * stride * sizeof(__half)) == cudaSuccess;
            if (ok) {
                rollout_tc2_shadow_kernel<<<dim3(ctx->sm_count * 8, 8), 256, 0, stream>>>(table, table_len, stride, (__half*)ctx->sh16_hi, nullptr);
                ES_LAUNCHED(ctx);
            }
        }
        if (ok && split && !ctx->sh16_lo) {
            ok = cudaMalloc(&ctx->sh16_lo, 8 * stride * sizeof(__half)) == cudaSuccess;
            if (ok) {
                // (recomputes hi: simpler than a second kernel, runs once per table)
                rollout_tc2_shadow_kernel<<<dim3(ctx->sm_count * 8, 8), 256, 0, stream>>>(table, table_len, stride, (__half*)ctx->sh16_hi,
                                                                                        (__half*)ctx->sh16_lo);
                ES_LAUNCHED(ctx);
            }
        }
        if (ok && !ctx->sh16_maps) {
            void* m = nullptr;
            ok = posix_memalign(&m, 64, sizeof(T2Maps)) == 0;
            if (ok) { memset(m, 0, sizeof(T2Maps)); ctx->sh16_maps = m; ctx->sh16_maps_lo = 0; }
            if (ok) ok = t2_encode_map(&((T2Maps*)ctx->sh16_maps)->hi, ctx->sh16_hi, stride, p.obs) == 0;
        }
        if (ok && split && !ctx->sh16_maps_lo) {
            ok = t2_encode_map(&((T2Maps*)ctx->sh16_maps)->lo, ctx->sh16_lo, stride, p.obs) == 0;
            if (ok) ctx->sh16_maps_lo = 1;
        }
        if (!ok) {
            (void)cudaGetLastError();
            es_tc2_free_shadows(ctx);
            ctx->sh16_failed = 1;
        } else {
            ctx->sh16_src = table; ctx->sh16_len = table_len; ctx->sh16_stride = stride; ctx->sh16_obs = p.obs;
            maps = *(T2Maps*)ctx->sh16_maps;
            p.use_tma = 1;
            p.shadow_stride = stride;
        }
    }
    return split ? t2_launch<true>(ctx, p, maps, obsn, rew_vec, theta, T, n_pairs, n_eps, stream)
                 : t2_launch<false>(ctx, p, maps, obsn, rew_vec, theta, T, n_pairs, n_eps, stream);
}
