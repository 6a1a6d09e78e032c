// rollout_tcw.cu -- fused perturb + MLP rollout + fitness on the tcgen05 tensor cores for WIDE policies:
// obs(<=1023) -> 2..4 hidden layers (each a multiple of 64 in [64, 256]) -> act(<=32) tanh MLPs, which covers the networks of
// every shipped training config (Hopper 15-256-256-3, HalfCheetah 17-256-256-256-6, Ant 28-128-256-256-128-8).  The
// obs-64-64-act shape stays with rollout_tc2.cu.  Same contract and the same two precisions as rollout_tc2.cu:
//   SPLIT = false (ES_ROLLOUT_TC):  float16 operands, one MMA per product, tanh.approx
//   SPLIT = true  (ES_ROLLOUT_TC3): float16 hi + lo operands, three MMAs per product (hi*hi + hi*lo + lo*hi) accumulated in
//                                   float32 in TMEM, accurate tanh, per-thread sums reduced to float64 fitness in a fixed order
//
// rollout_tc2's data movement does not carry over: there 82 % of the multiply-adds are layer 1, shared by both signs and all
// pairs through U +- sigma V.  Here 95-97 % are hidden x hidden products whose weights theta +- sigma*eps are unique to every
// pair and sign; one 256 x 256 layer is 128 KB of float16 per sign (256 KB as hi + lo), so no pair's weights fit on chip.
//
// One CTA = one antithetic pair at a time (persistent over pairs), 128 episode steps per MMA tile (M):
//   build   all warps write the pair's operand image into a per-CTA global scratch (L2): for every layer, sign and K chunk of
//           64, the N x 64 block of theta +- sigma*eps in the K-major 128-byte-swizzled layout of the MMA descriptor (pieces hi
//           [and lo]; N = the layer width, 32 for the output layer; the constant-1 column of the observation tile meets a zero
//           column); the biases theta +- sigma*eps go to shared memory and are added in float32 by the epilogue
//   stream  warp 0 moves the blocks, in the order they are consumed, through a ring of shared-memory slots: one bulk copy per
//           (layer, sign, K chunk); a layer-1 slot also carries the observation tile's chunk (rollout_tc2_prep_kernel's image)
//   MMA     warp 1: layer 1  D = X . W1^T with A from shared memory; hidden and output layers  D = h . W^T with the
//           activations h as the A operand in TMEM ("TS" form).  D = 128 lanes x N float32 columns in TMEM
//   epi     warps 2-17 (TMEM lane quarter = warp % 4, column quarter = (warp - 2) / 4): h = tanh(D + b) -> float16 (hi[, lo])
//           -> TMEM over the previous h; output layer: a = tanh(D + b) (+ action noise), r_t = <a_t, c_t> in float32 in column
//           order, fitness += r_t and the position integrator in float64 per thread
// TMEM (512 columns): D 0-255 | h hi 256-383 | h lo 384-511 (128 columns hold 256 float16 activations).  One (tile, sign) at a
// time runs through the layers; layer l+1's MMAs wait for layer l's epilogue (which frees D and fills h), so the tensor core
// and the epilogue warps alternate, while the ring keeps the copies of the next chunks in flight under both.
#include <stdlib.h>
#include "tc_ptx.cuh"

namespace {

constexpr int TW_THREADS = 576;                                  // 18 warps
constexpr int TW_W_PROD = 0, TW_W_MMA = 1, TW_EPI_WARP0 = 2, TW_EPI_WARPS = 16;
constexpr int TW_MAXL = 5;                                       // weight layers: 2..4 hidden + output
constexpr int TW_HMIN = 64, TW_HMAX = 256, TW_ACT_PAD = 32, TW_MAX_SLOTS = 8;
constexpr uint32_t TW_C_D = 0, TW_C_HHI = 256, TW_C_HLO = 384;   // TMEM columns
enum { TWB_FULL = 0, TWB_EMPTY = TW_MAX_SLOTS, TWB_DFULL = 2 * TW_MAX_SLOTS, TWB_EPI, TWB_COUNT };

struct TwParams {
    const float* table;
    const int64_t* idx;
    const float* theta;
    const uint8_t* xnt;           // [n_mtiles][nkc[0]][piece][16 KB stage image] (rollout_tc2_prep_kernel)
    const float* rew_vec;         // [T][act]
    const float* act_noise;       // [n_pairs][2][T][act] scaled action noise (mt_gauss.cu) or NULL
    uint8_t* images;              // [gridDim.x][img_bytes]
    double* fit_pos;
    double* fit_neg;
    float* behv_pos;
    float* behv_neg;
    int n_pairs, act, T, n_mtiles, fit_stride, nl;
    int in[TW_MAXL], out[TW_MAXL], N[TW_MAXL], nkc[TW_MAXL];     // N: MMA width (out, 32 for the output layer)
    int w_off[TW_MAXL], b_off[TW_MAXL];                          // flat parameter offsets
    uint32_t img_off[TW_MAXL];    // layer l's blocks in the image: [sign][kc][piece][N rows x 128 B]
    int bias_off[TW_MAXL];        // layer l's biases in shared memory (floats): [sign][N]
    uint32_t img_bytes, x_bytes, slot_bytes, s_bias, s_red, s_bars;
    int n_slots;
    float sigma, pos_scale;
    long long table_len;
    int P;
    int* err;
    int n_eps;                    // episodes per evaluation (act_noise [n_pairs][2][n_eps][T][act]); > 1 only with EPIS
};

// EPIS: p.n_eps > 1 episodes per evaluation sharing the forward pass; the output epilogue adds every episode's noise row to the
// noise-free actions, sums each episode's float32 reward into the float64 fitness, and integrates the last episode's position
template <bool SPLIT, bool EPIS>
__global__ void __launch_bounds__(TW_THREADS, 1) rollout_tcw_kernel(const __grid_constant__ TwParams p) {
    constexpr int NP = SPLIT ? 2 : 1;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = (uint64_t*)(smem + p.s_bars);
    uint32_t* tmem_slot = (uint32_t*)(bars + TWB_COUNT);
    float* bias_s = (float*)(smem + p.s_bias);
    double* red = (double*)(smem + p.s_red);                     // [epilogue warp][8]: the warps' sums of the pair

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int NL = p.nl, NMT = p.n_mtiles, NS = p.n_slots;
    const int my_pairs = (p.n_pairs - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

    if (tid == 0) {
        for (int s = 0; s < NS; ++s) { mbar_init(&bars[TWB_FULL + s], 1); mbar_init(&bars[TWB_EMPTY + s], 1); }
        mbar_init(&bars[TWB_DFULL], 1);
        mbar_init(&bars[TWB_EPI], TW_EPI_WARPS);
        fence_barrier_init();
    }
    __syncthreads();
    if (warp == TW_W_MMA) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    uint8_t* img = p.images + (size_t)blockIdx.x * p.img_bytes;

    uint32_t slot = 0, sphase = 0;       // ring position (producer, issuer)
    uint32_t u = 0;                      // (tile, sign, layer) units completed (issuer, epilogue)
    for (int i = 0; i < my_pairs; ++i) {
        const int pair = blockIdx.x + i * gridDim.x;
        // ===================== build: the pair's operand image (global scratch) and biases (shared memory) =====================
        {
            const float* __restrict__ eps = p.table + es_checked_slice(p.idx[pair], p.P, p.table_len, p.err);
            const float sg = p.sigma;
            for (int l = 0; l < NL; ++l) {
                const int in = p.in[l], out = p.out[l], N = p.N[l], Kp = p.nkc[l] * TC_KC;
                const uint32_t blk = (uint32_t)N * 128;
                const size_t sgn_stride = (size_t)p.nkc[l] * NP * blk;
                uint8_t* base = img + p.img_off[l];
                for (int e2 = tid; e2 < N * Kp / 2; e2 += TW_THREADS) {
                    const int n = (2 * e2) / Kp, k = 2 * e2 - n * Kp;
                    // theta +- sigma*eps with the reference's two roundings; zero beyond the layer (padding rows / columns)
                    float wp0 = 0.f, wp1 = 0.f, wn0 = 0.f, wn1 = 0.f;
                    if (n < out) {
                        const size_t off = (size_t)p.w_off[l] + (size_t)n * in + k;
                        if (k < in) {
                            const float d = __fmul_rn(sg, ldg_stream(eps + off)), t = __ldg(p.theta + off);
                            wp0 = __fadd_rn(t, d); wn0 = __fadd_rn(t, -d);
                        }
                        if (k + 1 < in) {
                            const float d = __fmul_rn(sg, ldg_stream(eps + off + 1)), t = __ldg(p.theta + off + 1);
                            wp1 = __fadd_rn(t, d); wn1 = __fadd_rn(t, -d);
                        }
                    }
                    uint8_t* dst = base + (size_t)((k >> 6) * NP) * blk + sw128_off(n, k & 63);
                    if (SPLIT) {
                        __half h0, l0, h1, l1;
                        split_h1(wp0, h0, l0); split_h1(wp1, h1, l1);
                        *(uint32_t*)dst = (uint32_t)__half_as_ushort(h0) | ((uint32_t)__half_as_ushort(h1) << 16);
                        *(uint32_t*)(dst + blk) = (uint32_t)__half_as_ushort(l0) | ((uint32_t)__half_as_ushort(l1) << 16);
                        split_h1(wn0, h0, l0); split_h1(wn1, h1, l1);
                        *(uint32_t*)(dst + sgn_stride) = (uint32_t)__half_as_ushort(h0) | ((uint32_t)__half_as_ushort(h1) << 16);
                        *(uint32_t*)(dst + sgn_stride + blk) = (uint32_t)__half_as_ushort(l0) | ((uint32_t)__half_as_ushort(l1) << 16);
                    } else {
                        *(uint32_t*)dst = pack_h2(wp0, wp1);
                        *(uint32_t*)(dst + sgn_stride) = pack_h2(wn0, wn1);
                    }
                }
                for (int n = tid; n < N; n += TW_THREADS) {
                    float vp = 0.f, vn = 0.f;
                    if (n < out) {
                        const float d = __fmul_rn(sg, ldg_stream(eps + p.b_off[l] + n)), t = __ldg(p.theta + p.b_off[l] + n);
                        vp = __fadd_rn(t, d); vn = __fadd_rn(t, -d);
                    }
                    bias_s[p.bias_off[l] + n] = vp;
                    bias_s[p.bias_off[l] + N + n] = vn;
                }
            }
            __threadfence();                                             // image visible device-wide (L2)
            asm volatile("fence.proxy.async;" ::: "memory");             // ... and to the async proxy that copies it
        }
        __syncthreads();

        if (warp == TW_W_PROD) {
            // ===================== producer: (observation chunk +) weight blocks, in consumption order =====================
            if (lane == 0) {
                for (int m = 0; m < NMT; ++m)
                    for (int s = 0; s < 2; ++s)
                        for (int l = 0; l < NL; ++l) {
                            const uint32_t wbytes = (uint32_t)NP * p.N[l] * 128;
                            for (int kc = 0; kc < p.nkc[l]; ++kc) {
                                mbar_wait(&bars[TWB_EMPTY + slot], sphase ^ 1);
                                uint8_t* dst = smem + (size_t)slot * p.slot_bytes;
                                mbar_expect_tx(&bars[TWB_FULL + slot], wbytes + (l == 0 ? p.x_bytes : 0u));
                                if (l == 0)
                                    bulk_g2s(dst, p.xnt + ((size_t)m * p.nkc[0] + kc) * p.x_bytes, p.x_bytes, &bars[TWB_FULL + slot]);
                                bulk_g2s(dst + p.x_bytes, img + p.img_off[l] + (size_t)(s * p.nkc[l] + kc) * wbytes, wbytes,
                                         &bars[TWB_FULL + slot]);
                                if (++slot == (uint32_t)NS) { slot = 0; sphase ^= 1; }
                            }
                        }
            }
            __syncwarp();
        } else if (warp == TW_W_MMA) {
            // ===================== MMA issuer (warp-uniform loop, one elected lane issues) =====================
            const uint32_t d = tmem + TW_C_D;
            for (int m = 0; m < NMT; ++m)
                for (int s = 0; s < 2; ++s)
                    for (int l = 0; l < NL; ++l, ++u) {
                        if (u > 0) mbar_wait(&bars[TWB_EPI], (u - 1) & 1);   // previous epilogue: D read, h written
                        tc_fence_after();
                        const uint32_t id = umma_idesc_f16(TC_MT, p.N[l]);
                        const uint32_t wblk = (uint32_t)p.N[l] * 128;
                        for (int kc = 0; kc < p.nkc[l]; ++kc) {
                            mbar_wait(&bars[TWB_FULL + slot], sphase);
                            tc_fence_after();
                            const uint32_t sb = smem_u32(smem + (size_t)slot * p.slot_bytes);
                            const uint64_t bh = umma_desc_sw128(sb + p.x_bytes), bl = umma_desc_sw128(sb + p.x_bytes + wblk);
                            if (elect_one()) {
                                if (l == 0) {
                                    const uint64_t ah = umma_desc_sw128(sb), al = umma_desc_sw128(sb + TC_STAGE);
                                    issue_ss4(d, ah, bh, id, kc != 0);                       // x_hi . w_hi
                                    if (SPLIT) {
                                        issue_ss4(d, ah, bl, id, 1);                         // x_hi . w_lo
                                        issue_ss4(d, al, bh, id, 1);                         // x_lo . w_hi
                                    }
                                } else {
                                    const uint32_t ah = tmem + TW_C_HHI + 32 * kc, al = tmem + TW_C_HLO + 32 * kc;
                                    issue_ts4(d, ah, bh, id, kc != 0);                       // h_hi . w_hi
                                    if (SPLIT) {
                                        issue_ts4(d, ah, bl, id, 1);                         // h_hi . w_lo
                                        issue_ts4(d, al, bh, id, 1);                         // h_lo . w_hi
                                    }
                                }
                                umma_commit(&bars[TWB_EMPTY + slot]);
                                if (kc == p.nkc[l] - 1) umma_commit(&bars[TWB_DFULL]);
                            }
                            __syncwarp();
                            if (++slot == (uint32_t)NS) { slot = 0; sphase ^= 1; }
                        }
                    }
        } else {
            // ===================== epilogue warps =====================
            const int ew = warp - TW_EPI_WARP0, q = warp & 3, cq = ew >> 2;
            const int row = q * 32 + lane;
            const uint32_t tl = tmem + ((uint32_t)(q * 32) << 16);
            const int act = p.act;
            double fit[2] = {0.0, 0.0}, pos[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
            for (int m = 0; m < NMT; ++m) {
                const int t = m * TC_MT + row;
                for (int s = 0; s < 2; ++s)
                    for (int l = 0; l < NL; ++l, ++u) {
                        mbar_wait(&bars[TWB_DFULL], u & 1);
                        tc_fence_after();
                        const float* bl = bias_s + p.bias_off[l] + s * p.N[l];
                        if (l + 1 < NL) {
                            // h = tanh(D + b) -> float16 (hi[, lo]) -> TMEM, 8 columns at a time
                            const int cw = p.N[l] >> 2, c_lo = cq * cw;
                            for (int c0 = c_lo; c0 < c_lo + cw; c0 += 8) {
                                uint32_t v[8];
                                tmem_ld8(tl + TW_C_D + c0, v);
                                const float4 b0 = *reinterpret_cast<const float4*>(bl + c0);
                                const float4 b1 = *reinterpret_cast<const float4*>(bl + c0 + 4);
                                tmem_ld_wait();
                                const float bs[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
                                uint32_t whi[4], wlo[4];
#pragma unroll
                                for (int e = 0; e < 4; ++e) {
                                    float z0, z1, t0, t1;
                                    unpk(add2(pk(__uint_as_float(v[2 * e]), __uint_as_float(v[2 * e + 1])), pk(bs[2 * e], bs[2 * e + 1])), z0, z1);
                                    if (SPLIT) { tanh_acc2(z0, z1, t0, t1, false); split_h2(t0, t1, whi[e], wlo[e]); }
                                    else { whi[e] = pack_h2(tanh_fast(z0), tanh_fast(z1)); }
                                }
                                tmem_st4(tl + TW_C_HHI + c0 / 2, whi[0], whi[1], whi[2], whi[3]);
                                if (SPLIT) tmem_st4(tl + TW_C_HLO + c0 / 2, wlo[0], wlo[1], wlo[2], wlo[3]);
                            }
                            tmem_st_wait();
                        } else if (cq * 8 < act) {
                            // output layer: this warp's 8 action columns (warp-uniform condition)
                            uint32_t v[8];
                            tmem_ld8(tl + TW_C_D + cq * 8, v);
                            const float4 b0 = *reinterpret_cast<const float4*>(bl + cq * 8);
                            const float4 b1 = *reinterpret_cast<const float4*>(bl + cq * 8 + 4);
                            tmem_ld_wait();
                            const float bs[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
                            float a[8];
#pragma unroll
                            for (int e = 0; e < 4; ++e) {
                                const float z0 = __uint_as_float(v[2 * e]) + bs[2 * e], z1 = __uint_as_float(v[2 * e + 1]) + bs[2 * e + 1];
                                if (SPLIT) tanh_acc2(z0, z1, a[2 * e], a[2 * e + 1], false);
                                else { a[2 * e] = tanh_fast(z0); a[2 * e + 1] = tanh_fast(z1); }
                            }
                            if (EPIS && t < p.T) {
                                const float* __restrict__ c = p.rew_vec + (size_t)t * act;
                                const float* __restrict__ ns = p.act_noise + ((((size_t)pair * 2 + s) * p.n_eps) * p.T + t) * act;
                                float cw[8], ae[8];
#pragma unroll
                                for (int e = 0; e < 8; ++e) cw[e] = (cq * 8 + e < act) ? __ldg(c + cq * 8 + e) : 0.f;
                                for (int ep = 0; ep < p.n_eps; ++ep) {
                                    const float* __restrict__ nz = ns + (size_t)ep * p.T * act;
                                    float r = 0.f;
#pragma unroll
                                    for (int e = 0; e < 8; ++e) {
                                        const int j = cq * 8 + e;
                                        ae[e] = a[e];
                                        if (j < act) {
                                            ae[e] = __fadd_rn(a[e], __ldg(nz + j));
                                            r = __fadd_rn(r, __fmul_rn(ae[e], cw[e]));
                                        }
                                    }
                                    fit[s] += (double)r;
                                }
                                if (cq == 0) {                                  // the last episode's position
                                    pos[3 * s + 0] += (double)ae[0];
                                    pos[3 * s + 1] += (double)(act > 1 ? ae[1] : ae[0]);
                                    pos[3 * s + 2] += (double)(act > 2 ? ae[2] : ae[0]);
                                }
                            } else if (!EPIS && t < p.T) {
                                const float* __restrict__ c = p.rew_vec + (size_t)t * act;
                                const float* __restrict__ nz =
                                    p.act_noise ? p.act_noise + (((size_t)pair * 2 + s) * p.T + t) * act : nullptr;
                                float r = 0.f;
#pragma unroll
                                for (int e = 0; e < 8; ++e) {
                                    const int j = cq * 8 + e;
                                    if (j < act) {
                                        if (nz) a[e] = __fadd_rn(a[e], __ldg(nz + j));   // a += rs.randn(act) * ac_std (src/nn/nn.py:47-48)
                                        r = __fadd_rn(r, __fmul_rn(a[e], __ldg(c + j)));
                                    }
                                }
                                fit[s] += (double)r;
                                if (cq == 0) {                                  // position integrator: components 0, 1 % act, 2 % act
                                    pos[3 * s + 0] += (double)a[0];
                                    pos[3 * s + 1] += (double)(act > 1 ? a[1] : a[0]);
                                    pos[3 * s + 2] += (double)(act > 2 ? a[2] : a[0]);
                                }
                            }
                        }
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&bars[TWB_EPI]);
                    }
            }
            // this warp's sums of the pair -> shared memory (butterfly: the same order on every run)
            if (EPIS) { fit[0] /= p.n_eps; fit[1] /= p.n_eps; }       // obj.py: rews /= max(1, eps_per_policy)
            double w8[8] = {fit[0], fit[1], pos[0], pos[1], pos[2], pos[3], pos[4], pos[5]};
#pragma unroll
            for (int k = 0; k < 8; ++k) w8[k] = warp_sum_d(w8[k]);
            if (lane == 0) {
#pragma unroll
                for (int k = 0; k < 8; ++k) red[ew * 8 + k] = w8[k];
            }
        }
        __syncthreads();
        if (tid == 0) {
            // the 16 warps' sums in warp order
            double tot[8] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
            for (int w = 0; w < TW_EPI_WARPS; ++w)
                for (int k = 0; k < 8; ++k) tot[k] += red[w * 8 + k];
            p.fit_pos[(size_t)pair * p.fit_stride] = tot[0];
            p.fit_neg[(size_t)pair * p.fit_stride] = tot[1];
            if (p.behv_pos) {
                for (int k = 0; k < 3; ++k) {
                    p.behv_pos[pair * 3 + k] = (float)((double)p.pos_scale * tot[2 + k]);
                    p.behv_neg[pair * 3 + k] = (float)((double)p.pos_scale * tot[5 + k]);
                }
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == TW_W_MMA) tmem_dealloc(tmem, 512);
}

template <bool SPLIT>
int tw_launch(es_ctx* ctx, TwParams& p, const float* obsn, int T, int n_pairs, cudaStream_t stream) {
    auto kernel = p.n_eps > 1 ? rollout_tcw_kernel<SPLIT, true> : rollout_tcw_kernel<SPLIT, false>;
    constexpr int NP = SPLIT ? 2 : 1;
    int nmax = 0, bias_floats = 0;
    uint32_t img = 0;
    for (int l = 0; l < p.nl; ++l) {
        p.img_off[l] = img;
        img += 2u * p.nkc[l] * NP * p.N[l] * 128;
        p.bias_off[l] = bias_floats;
        bias_floats += 2 * p.N[l];
        if (p.N[l] > nmax) nmax = p.N[l];
    }
    p.img_bytes = img;
    p.x_bytes = NP * TC_STAGE;
    p.slot_bytes = p.x_bytes + (uint32_t)NP * nmax * 128;
    const uint32_t fixed = (uint32_t)bias_floats * 4 + TW_EPI_WARPS * 64 + 256;
    const uint32_t budget = 227 * 1024 - 1024 - fixed;                  // (1024: alignment slack of the dynamic window)
    p.n_slots = (int)(budget / p.slot_bytes);
    if (p.n_slots > TW_MAX_SLOTS) p.n_slots = TW_MAX_SLOTS;
    if (p.n_slots < 2) {
        es_set_error("es_rollout_openloop(TC%s): a ring slot of %u bytes does not fit twice in shared memory", SPLIT ? "3" : "",
                     p.slot_bytes);
        return ES_ERR_UNSUPPORTED;
    }
    p.s_bias = (uint32_t)p.n_slots * p.slot_bytes;
    p.s_red = p.s_bias + (((uint32_t)bias_floats * 4 + 15) & ~15u);
    p.s_bars = p.s_red + TW_EPI_WARPS * 64;
    const size_t smem = (size_t)p.s_bars + 256 + 1024;

    const size_t xnt_bytes = (size_t)p.n_mtiles * p.nkc[0] * NP * TC_STAGE;
    const int grid = n_pairs < ctx->sm_count ? n_pairs : ctx->sm_count;
    void* scratch = nullptr;
    int rc = es_ctx_scratch(ctx, xnt_bytes + (size_t)grid * p.img_bytes, &scratch);
    if (rc) return rc;
    uint8_t* xnt = (uint8_t*)scratch;
    p.xnt = xnt;
    p.images = xnt + xnt_bytes;
    {
        const size_t total = (size_t)p.n_mtiles * p.nkc[0] * TC_MT * TC_KC;
        int blocks = es_div_up((int64_t)total, 256);
        if (blocks > ctx->sm_count * 8) blocks = ctx->sm_count * 8;
        rollout_tc2_prep_kernel<SPLIT><<<blocks, 256, 0, stream>>>(obsn, T, p.in[0], p.nkc[0], p.n_mtiles, xnt);
        ES_LAUNCHED(ctx);
    }
    ES_CHECK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kernel<<<grid, TW_THREADS, smem, stream>>>(p);
    ES_LAUNCHED(ctx);
    return ES_OK;
}

}  // namespace

int es_tcw_covers(const int* layer_sizes, int n_layers) {
    if (n_layers < 3 || n_layers > TW_MAXL) return 0;                   // 2..4 hidden layers
    if (layer_sizes[0] > 1023 || layer_sizes[n_layers] > TW_ACT_PAD) return 0;
    for (int l = 1; l < n_layers; ++l)
        if (layer_sizes[l] % 64 != 0 || layer_sizes[l] < TW_HMIN || layer_sizes[l] > TW_HMAX) return 0;
    return 1;
}

int es_impl_rollout_tcw(es_ctx* ctx, int split, const float* table, int64_t table_len, const int64_t* idx, int n_pairs,
                        const float* theta, int P, float sigma, const int* layer_sizes, int n_layers, const float* obsn,
                        const float* rew_vec, int T, float pos_scale, double* fit_pos, double* fit_neg, int fit_stride,
                        float* behv_pos, float* behv_neg, const float* act_noise, int n_eps, cudaStream_t stream) {
    if (!es_tcw_covers(layer_sizes, n_layers)) {
        es_set_error("es_rollout_openloop(TC): the wide tensor-core path covers obs(<=1023) -> 2..4 hidden layers (multiples of "
                     "64 in [64, 256]) -> act(<=32) tanh MLPs");
        return ES_ERR_UNSUPPORTED;
    }
    TwParams p;
    memset(&p, 0, sizeof(p));
    p.table = table; p.idx = idx; p.theta = theta; p.rew_vec = rew_vec; p.act_noise = act_noise;
    p.fit_pos = fit_pos; p.fit_neg = fit_neg; p.behv_pos = behv_pos; p.behv_neg = behv_neg;
    p.n_pairs = n_pairs; p.act = layer_sizes[n_layers]; p.T = T; p.n_mtiles = es_div_up(T, TC_MT); p.fit_stride = fit_stride;
    p.nl = n_layers;
    int off = 0;
    for (int l = 0; l < n_layers; ++l) {
        p.in[l] = layer_sizes[l];
        p.out[l] = layer_sizes[l + 1];
        p.N[l] = (l == n_layers - 1) ? TW_ACT_PAD : p.out[l];
        p.nkc[l] = (l == 0) ? es_div_up(p.in[0] + 1, TC_KC) : p.in[l] / TC_KC;   // layer 1: + the constant-1 column of the prep image
        p.w_off[l] = off; off += p.in[l] * p.out[l];
        p.b_off[l] = off; off += p.out[l];
    }
    p.sigma = sigma; p.pos_scale = pos_scale;
    p.table_len = table_len; p.P = P; p.err = ctx->err_dev; p.n_eps = n_eps;
    return split ? tw_launch<true>(ctx, p, obsn, T, n_pairs, stream) : tw_launch<false>(ctx, p, obsn, T, n_pairs, stream);
}
