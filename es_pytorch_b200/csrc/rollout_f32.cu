// rollout_f32.cu -- fused perturb + MLP rollout + fitness, float32 CUDA-core path.
//
// One CTA evaluates one perturbed policy (blockIdx.x = 2*pair + sign) over the whole
// open-loop episode:
//   W = theta +- sigma*table[idx : idx+P]      (src/core/policy.py:61-64; built straight into
//                                               shared memory, theta' never touches HBM)
//   a_t = tanh(W3 tanh(W2 tanh(W1 x_t + b1) + b2) + b3)   (src/nn/nn.py:35-36,46)
//   r_t = <a_t, c_t> float32;  fitness = sum_t r_t in float64, step order
//                                               (src/gym/training_result.py:28,62-64)
//   pos += pos_scale * a_t[0..2]                (synthetic env position integrator)
// This is the device-side precision reference for the tensor-core path and the general
// fallback (any layer sizes whose weights fit in shared memory).
//
// Shared-memory layout: weight rows are padded to a pitch with (pitch/4) odd so that the
// 128-bit reads of 32 different output rows at the same k hit 32 different bank groups;
// activations for a tile of RF_TM time steps ping-pong between two buffers.
#include <stdlib.h>
#include "common.cuh"

constexpr int RF_THREADS = 512;   // 16 warps: the dense tasks keep 8 of them busy, the others hide the load / staging latencies
constexpr int RF_WARPS = RF_THREADS / 32;
constexpr int RF_TM = 32;   // time steps per tile
constexpr int RF_RT = 8;    // time steps per thread (register tile)

struct RfDesc {
    int n_layers;
    int in[ES_MAX_LAYERS], out[ES_MAX_LAYERS];
    int in4[ES_MAX_LAYERS];      // in rounded up to a multiple of 4
    int pitch[ES_MAX_LAYERS];    // shared-memory row pitch of W_l (floats)
    int w_off[ES_MAX_LAYERS];    // offset of W_l / b_l in the flat parameter vector
    int b_off[ES_MAX_LAYERS];
    int sw_off[ES_MAX_LAYERS];   // offset of W_l / b_l in shared memory (floats)
    int sb_off[ES_MAX_LAYERS];
    int w_floats;                // total shared floats for weights + biases
    int xpitch;                  // activation buffer pitch (floats), multiple of 4
    int P;
    long long table_len;         // bounds of the noise table (NoiseTable.get's assert, noisetable.py:34)
    int* err;                    // ctx error word (es_checked_slice)
};

__device__ __forceinline__ void rf_dense(const float* __restrict__ Wsm, const float* __restrict__ bsm, int in4, int pitch,
                                         int out, const float* __restrict__ Xin, float* __restrict__ Xout, int xpitch) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_blocks = (out + 31) >> 5;
    const int tasks = n_blocks * (RF_TM / RF_RT);
    for (int task = warp; task < tasks; task += RF_WARPS) {
        const int nb = task % n_blocks, tg = task / n_blocks;
        const int n = nb * 32 + lane;
        const bool valid = n < out;
        const int nn = valid ? n : out - 1;
        float acc[RF_RT];
        const float bias = bsm[nn];
#pragma unroll
        for (int r = 0; r < RF_RT; ++r) acc[r] = bias;
        const float4* __restrict__ wrow = reinterpret_cast<const float4*>(Wsm + (size_t)nn * pitch);
        const float4* __restrict__ xrow = reinterpret_cast<const float4*>(Xin + (size_t)(tg * RF_RT) * xpitch);
        const int xp4 = xpitch >> 2;
        for (int k4 = 0; k4 < (in4 >> 2); ++k4) {
            const float4 w = wrow[k4];
#pragma unroll
            for (int r = 0; r < RF_RT; ++r) {
                const float4 x = xrow[r * xp4 + k4];
                acc[r] = fmaf(x.x, w.x, acc[r]);
                acc[r] = fmaf(x.y, w.y, acc[r]);
                acc[r] = fmaf(x.z, w.z, acc[r]);
                acc[r] = fmaf(x.w, w.w, acc[r]);
            }
        }
        if (valid) {
#pragma unroll
            for (int r = 0; r < RF_RT; ++r) Xout[(size_t)(tg * RF_RT + r) * xpitch + n] = tanhf(acc[r]);
        }
    }
}

// W = theta +- sigma*eps of one policy, rows padded to the layer's pitch (zero padding), biases behind the weights
__device__ __forceinline__ void rf_stage_weights(float* __restrict__ W, const float* __restrict__ eps,
                                                 const float* __restrict__ theta, float sigma, bool neg, const RfDesc& d) {
    for (int l = 0; l < d.n_layers; ++l) {
        const int in = d.in[l], cnt = d.in[l] * d.out[l];
        for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
            const int n = i / in, k = i - n * in;
            const float dlt = __fmul_rn(sigma, __ldg(eps + d.w_off[l] + i));     // std * noise
            const float t = __ldg(theta + d.w_off[l] + i);
            W[d.sw_off[l] + n * d.pitch[l] + k] = __fadd_rn(t, neg ? -dlt : dlt);
        }
        for (int i = threadIdx.x; i < d.out[l]; i += blockDim.x) {
            const float dlt = __fmul_rn(sigma, __ldg(eps + d.b_off[l] + i));
            W[d.sb_off[l] + i] = __fadd_rn(__ldg(theta + d.b_off[l] + i), neg ? -dlt : dlt);
        }
    }
}

// networks whose padded weights do not fit in shared memory (e.g. the 15-256-256-3 net of configs/simple_conf.json): the
// perturbed weights of every policy of the launch are staged in a global scratch (L2 resident) by this kernel first
__global__ void __launch_bounds__(RF_THREADS)
rollout_f32_stage_kernel(const float* __restrict__ table, const int64_t* __restrict__ idx, const float* __restrict__ theta,
                         float sigma, const __grid_constant__ RfDesc d, float* __restrict__ wglobal) {
    float* W = wglobal + (size_t)blockIdx.x * d.w_floats;
    for (int i = threadIdx.x; i < d.w_floats; i += RF_THREADS) W[i] = 0.f;
    __syncthreads();
    rf_stage_weights(W, table + es_checked_slice(idx[blockIdx.x >> 1], d.P, d.table_len, d.err), theta, sigma, blockIdx.x & 1, d);
}

// GW: weights in the global scratch filled by rollout_f32_stage_kernel instead of shared memory.
// EPIS: n_eps > 1 episodes per evaluation (act_noise [2*pair + sign][n_eps][T][act]); the forward pass is shared, every episode
// adds its own noise row (the actions in xin stay noise-free) and the last episode drives the position integrator
template <bool GW, bool EPIS>
__global__ void __launch_bounds__(RF_THREADS, 1)
rollout_f32_kernel(const float* __restrict__ table, const int64_t* __restrict__ idx, const float* __restrict__ theta,
                   float sigma, const __grid_constant__ RfDesc d, const float* __restrict__ obsn,
                   const float* __restrict__ rew_vec, int T, float pos_scale, double* __restrict__ fit_pos,
                   double* __restrict__ fit_neg, int fit_stride, float* __restrict__ behv_pos,
                   float* __restrict__ behv_neg, double* __restrict__ part, unsigned* __restrict__ tickets,
                   const float* __restrict__ wglobal, const float* __restrict__ act_noise, int n_eps) {
    extern __shared__ __align__(16) float smem[];
    float* Wsm = GW ? const_cast<float*>(wglobal) + (size_t)blockIdx.x * d.w_floats : smem;    // [w_floats]
    float* Xa = GW ? smem : smem + d.w_floats;          // [RF_TM][xpitch]
    float* Xb = Xa + RF_TM * d.xpitch;                  // [RF_TM][xpitch]
    float* s_rew = Xb + RF_TM * d.xpitch;               // [RF_TM]
    __shared__ double s_fit;
    __shared__ float s_pos[3];

    const int pair = blockIdx.x >> 1;
    const bool neg = blockIdx.x & 1;
    const float* __restrict__ eps = table + es_checked_slice(idx[pair], d.P, d.table_len, d.err);

    // ---- stage W = theta +- sigma*eps (zero the padding first) ----
    if (!GW) for (int i = threadIdx.x; i < d.w_floats; i += RF_THREADS) Wsm[i] = 0.f;
    for (int i = threadIdx.x; i < 2 * RF_TM * d.xpitch; i += RF_THREADS) Xa[i] = 0.f;
    if (threadIdx.x == 0) { s_fit = 0.0; s_pos[0] = s_pos[1] = s_pos[2] = 0.f; }
    __syncthreads();
    if (!GW) rf_stage_weights(Wsm, eps, theta, sigma, neg, d);
    __syncthreads();

    const int obs_dim = d.in[0];
    const int act_dim = d.out[d.n_layers - 1];
    // time split (gridDim.y > 1, used when there are fewer policies than SMs): the open-loop episode has no state, so
    // CTA y evaluates a contiguous range of time tiles; the partial sums are combined in tile order by the last CTA
    const int n_tiles = (T + RF_TM - 1) / RF_TM;
    const int tile_lo = (int)((long long)n_tiles * blockIdx.y / gridDim.y);
    const int tile_hi = (int)((long long)n_tiles * (blockIdx.y + 1) / gridDim.y);
    for (int t0 = tile_lo * RF_TM; t0 < min(T, tile_hi * RF_TM); t0 += RF_TM) {
        const int rows = min(RF_TM, T - t0);
        // observation tile -> Xa (rows beyond T are zero: computed and ignored)
        // (columns [obs_dim, in4) are re-zeroed every tile: later layers reuse this buffer)
        const int in40 = d.in4[0];
        for (int i = threadIdx.x; i < RF_TM * in40; i += RF_THREADS) {
            const int r = i / in40, k = i - r * in40;
            Xa[r * d.xpitch + k] = (r < rows && k < obs_dim) ? __ldg(obsn + (size_t)(t0 + r) * obs_dim + k) : 0.f;
        }
        __syncthreads();
        float* xin = Xa;
        float* xout = Xb;
        for (int l = 0; l < d.n_layers; ++l) {
            // the padding columns [out, in4_next) of xout must read as zero in the next layer
            if (l + 1 < d.n_layers && d.in4[l + 1] != d.out[l]) {
                const int padw = d.in4[l + 1] - d.out[l];
                for (int i = threadIdx.x; i < RF_TM * padw; i += RF_THREADS)
                    xout[(i / padw) * d.xpitch + d.out[l] + (i % padw)] = 0.f;
            }
            rf_dense(Wsm + d.sw_off[l], Wsm + d.sb_off[l], d.in4[l], d.pitch[l], d.out[l], xin, xout, d.xpitch);
            __syncthreads();
            float* tmp = xin; xin = xout; xout = tmp;
        }
        // xin now holds the actions [RF_TM][act_dim]
        if (EPIS) {
            // obj.py's episode loop: per step, the float32 reward of every episode's noisy action summed in float64 (the
            // reference's rews[t] += r before the division by E, done once at the end)
            __shared__ double s_rew_e[RF_TM];
            __shared__ float s_last[RF_TM][3];              // the last episode's noisy action components 0, 1 % act, 2 % act
            if (threadIdx.x < rows) {
                const int r = threadIdx.x;
                const float* a = xin + r * d.xpitch;
                const float* c = rew_vec + (size_t)(t0 + r) * act_dim;
                double racc = 0.0;
                for (int e = 0; e < n_eps; ++e) {
                    const float* __restrict__ nz = act_noise + (((size_t)blockIdx.x * n_eps + e) * T + t0 + r) * act_dim;
                    float acc = 0.f;
                    for (int j = 0; j < act_dim; ++j) acc = __fadd_rn(acc, __fmul_rn(__fadd_rn(a[j], __ldg(nz + j)), __ldg(c + j)));
                    racc += (double)acc;
                    if (e == n_eps - 1)
                        for (int k = 0; k < 3; ++k) s_last[r][k] = __fadd_rn(a[k % act_dim], __ldg(nz + k % act_dim));
                }
                s_rew_e[r] = racc;
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                double f = s_fit;
                float p0 = s_pos[0], p1 = s_pos[1], p2 = s_pos[2];
                for (int r = 0; r < rows; ++r) {
                    f += s_rew_e[r];
                    p0 = __fadd_rn(p0, __fmul_rn(pos_scale, s_last[r][0]));
                    p1 = __fadd_rn(p1, __fmul_rn(pos_scale, s_last[r][1]));
                    p2 = __fadd_rn(p2, __fmul_rn(pos_scale, s_last[r][2]));
                }
                s_fit = f; s_pos[0] = p0; s_pos[1] = p1; s_pos[2] = p2;
            }
            __syncthreads();
            continue;
        }
        if (act_noise) {
            // a += rs.randn(act) * ac_std (src/nn/nn.py:47-48): the scaled gaussians of this evaluation, drawn in stream order
            // by mt_gauss.cu; reward and position see the noisy action (the env receives it, gym_runner.py:53)
            const float* __restrict__ nz = act_noise + ((size_t)blockIdx.x * T + t0) * act_dim;
            for (int i = threadIdx.x; i < rows * act_dim; i += RF_THREADS) {
                const int r = i / act_dim, j = i - r * act_dim;
                xin[r * d.xpitch + j] = __fadd_rn(xin[r * d.xpitch + j], __ldg(nz + i));
            }
            __syncthreads();
        }
        if (threadIdx.x < rows) {
            const int r = threadIdx.x;
            const float* a = xin + r * d.xpitch;
            const float* c = rew_vec + (size_t)(t0 + r) * act_dim;
            float acc = 0.f;
            for (int j = 0; j < act_dim; ++j) acc = __fadd_rn(acc, __fmul_rn(a[j], __ldg(c + j)));
            s_rew[r] = acc;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            double f = s_fit;
            float p0 = s_pos[0], p1 = s_pos[1], p2 = s_pos[2];
            for (int r = 0; r < rows; ++r) {
                f += (double)s_rew[r];
                const float* a = xin + r * d.xpitch;
                p0 = __fadd_rn(p0, __fmul_rn(pos_scale, a[0 % act_dim]));
                p1 = __fadd_rn(p1, __fmul_rn(pos_scale, a[1 % act_dim]));
                p2 = __fadd_rn(p2, __fmul_rn(pos_scale, a[2 % act_dim]));
            }
            s_fit = f; s_pos[0] = p0; s_pos[1] = p1; s_pos[2] = p2;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        double f = s_fit;
        float p0 = s_pos[0], p1 = s_pos[1], p2 = s_pos[2];
        bool writer = true;
        if (gridDim.y > 1) {
            double* mine = part + ((size_t)blockIdx.x * gridDim.y + blockIdx.y) * 4;
            __stcg(mine + 0, f); __stcg(mine + 1, (double)p0); __stcg(mine + 2, (double)p1); __stcg(mine + 3, (double)p2);
            __threadfence();
            writer = atomicAdd(tickets + blockIdx.x, 1u) == gridDim.y - 1;
            if (writer) {
                __threadfence();
                tickets[blockIdx.x] = 0;                                 // self-resetting
                f = 0.0; p0 = p1 = p2 = 0.f;
                for (unsigned y = 0; y < gridDim.y; ++y) {
                    const double* q = part + ((size_t)blockIdx.x * gridDim.y + y) * 4;
                    f += __ldcg(q + 0);
                    p0 = __fadd_rn(p0, (float)__ldcg(q + 1)); p1 = __fadd_rn(p1, (float)__ldcg(q + 2));
                    p2 = __fadd_rn(p2, (float)__ldcg(q + 3));
                }
            }
        }
        if (writer) {
            if (EPIS) f /= n_eps;                                        // obj.py: rews /= max(1, eps_per_policy)
            (neg ? fit_neg : fit_pos)[(size_t)pair * fit_stride] = f;
            float* b = neg ? behv_neg : behv_pos;
            if (b) { b[pair * 3 + 0] = p0; b[pair * 3 + 1] = p1; b[pair * 3 + 2] = p2; }
        }
    }
}

static int rf_round4(int x) { return (x + 3) & ~3; }

int es_impl_rollout_f32(es_ctx* ctx, const float* table, int64_t table_len, const int64_t* idx, int n_pairs,
                        const float* theta, int P, float sigma, const int* layer_sizes, int n_layers, const float* obsn,
                        const float* rew_vec, int T, float pos_scale, double* fit_pos, double* fit_neg, int fit_stride,
                        float* behv_pos, float* behv_neg, const float* act_noise, int n_eps, cudaStream_t stream) {
    // obs-64-64-act networks with enough pairs to fill the GPU: the packed-FMA kernel of rollout_f32x.cu (one CTA per pair);
    // fewer pairs than half the SMs (single evaluations, es.step's noiseless evaluation) stay here, where the episode's time
    // tiles are split over the idle SMs.  ES_F32_GENERAL=1 forces this kernel (tests compare the two).
    if (2 * n_pairs >= ctx->sm_count && !getenv("ES_F32_GENERAL")) {
        const int rc = es_impl_rollout_f32x(ctx, table, table_len, idx, n_pairs, theta, P, sigma, layer_sizes, n_layers, obsn, rew_vec,
                                            T, pos_scale, fit_pos, fit_neg, fit_stride, behv_pos, behv_neg, act_noise, n_eps, stream);
        if (rc != ES_ERR_UNSUPPORTED) return rc;
    }
    RfDesc d;
    memset(&d, 0, sizeof(d));
    d.n_layers = n_layers;
    d.P = P;
    d.table_len = table_len;
    d.err = ctx->err_dev;
    int off = 0, soff = 0, xmax = 0;
    for (int l = 0; l < n_layers; ++l) {
        d.in[l] = layer_sizes[l];
        d.out[l] = layer_sizes[l + 1];
        d.in4[l] = rf_round4(d.in[l]);
        d.pitch[l] = ((d.in4[l] >> 2) & 1) ? d.in4[l] : d.in4[l] + 4;   // (pitch/4) odd -> conflict-free float4 rows
        d.w_off[l] = off; off += d.in[l] * d.out[l];
        d.b_off[l] = off; off += d.out[l];
        d.sw_off[l] = soff; soff += d.out[l] * d.pitch[l];
        if (d.in4[l] > xmax) xmax = d.in4[l];
        if (rf_round4(d.out[l]) > xmax) xmax = rf_round4(d.out[l]);
    }
    for (int l = 0; l < n_layers; ++l) { d.sb_off[l] = soff; soff += rf_round4(d.out[l]); }
    d.w_floats = rf_round4(soff);
    d.xpitch = xmax;
    const size_t act_smem = (2 * (size_t)RF_TM * d.xpitch + RF_TM) * sizeof(float);
    const size_t smem_w = (size_t)d.w_floats * sizeof(float) + act_smem;
    const bool gw = smem_w > 227 * 1024;              // weights do not fit beside the activation tiles: global scratch
    if (act_smem > 227 * 1024) {
        es_set_error("es_rollout_openloop(F32): layer width needs %zu bytes of shared memory for the activation tiles (> 227 KB)",
                     act_smem);
        return ES_ERR_UNSUPPORTED;
    }
    ES_REQUIRE(n_pairs <= (1 << 30), "es_rollout_openloop: too many pairs");
    const int n_tiles = (T + RF_TM - 1) / RF_TM;
    // policies per launch: everything at once with the weights in shared memory; chunks of <= 256 MB of staged weights else
    int chunk = n_pairs;
    if (gw) {
        const size_t per_pair = 2 * (size_t)d.w_floats * sizeof(float);
        chunk = (int)((256u << 20) / per_pair);
        if (chunk < 1) chunk = 1;
        if (chunk > n_pairs) chunk = n_pairs;
    }
    for (int p0 = 0; p0 < n_pairs; p0 += chunk) {
        const int np = (n_pairs - p0 < chunk) ? n_pairs - p0 : chunk;
        // fewer policies than SMs (single evaluations of the per-perturbation compatibility path, es.step's noiseless
        // evaluation): split the episode's time tiles over the idle SMs
        int n_splits = 1;
        if (2 * np < ctx->sm_count) {
            n_splits = ctx->sm_count / (2 * np);
            if (n_splits > n_tiles) n_splits = n_tiles;
            if (n_splits < 1) n_splits = 1;
        }
        const size_t part_bytes = (n_splits > 1) ? ((size_t)2 * np * n_splits * 4 * sizeof(double) + 255) & ~(size_t)255 : 0;
        const size_t w_bytes = gw ? (size_t)2 * np * d.w_floats * sizeof(float) : 0;
        double* part = nullptr;
        unsigned* tickets = nullptr;
        float* wglobal = nullptr;
        if (part_bytes + w_bytes) {
            void* scratch = nullptr;
            int rc = es_ctx_scratch(ctx, part_bytes + w_bytes, &scratch);
            if (rc) return rc;
            part = part_bytes ? (double*)scratch : nullptr;
            wglobal = gw ? (float*)((char*)scratch + part_bytes) : nullptr;
            if (n_splits > 1) {
                rc = es_ctx_counters(ctx, 4096, &tickets);
                if (rc) return rc;
            }
        }
        double* fp = fit_pos + (size_t)p0 * fit_stride;
        double* fn = fit_neg + (size_t)p0 * fit_stride;
        float* bp = behv_pos ? behv_pos + (size_t)p0 * 3 : nullptr;
        float* bn = behv_neg ? behv_neg + (size_t)p0 * 3 : nullptr;
        const float* an = act_noise ? act_noise + (size_t)p0 * 2 * n_eps * T * layer_sizes[n_layers] : nullptr;
        if (gw) {
            rollout_f32_stage_kernel<<<2 * np, RF_THREADS, 0, stream>>>(table, idx + p0, theta, sigma, d, wglobal);
            ES_LAUNCHED(ctx);
        }
        const dim3 grid(2 * np, n_splits);
        const size_t smem = gw ? act_smem : smem_w;
        const float* wg = gw ? wglobal : nullptr;
        auto kernel = gw ? (n_eps > 1 ? rollout_f32_kernel<true, true> : rollout_f32_kernel<true, false>)
                         : (n_eps > 1 ? rollout_f32_kernel<false, true> : rollout_f32_kernel<false, false>);
        ES_CHECK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kernel<<<grid, RF_THREADS, smem, stream>>>(table, idx + p0, theta, sigma, d, obsn, rew_vec, T, pos_scale, fp, fn, fit_stride, bp,
                                                   bn, part, tickets, wg, an, n_eps);
        ES_LAUNCHED(ctx);
    }
    return ES_OK;
}
