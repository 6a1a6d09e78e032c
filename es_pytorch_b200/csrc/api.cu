// api.cu -- extern "C" surface of libes_b200.so (declared in include/es_b200.h):
// argument validation, context/scratch management, dispatch to the kernels.
#include <stdarg.h>
#include <stdlib.h>
#include "common.cuh"

static thread_local char g_err[512] = "";

void es_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int es_ctx_scratch(es_ctx* ctx, size_t bytes, void** out) {
    if (bytes > ctx->scratch_bytes) {
        // growing is rare (first call per shape); it synchronises the device, which is
        // fine outside the steady state.
        if (ctx->scratch) ES_CHECK_CUDA(cudaFree(ctx->scratch));
        ctx->scratch = nullptr;
        ctx->scratch_bytes = 0;
        size_t want = bytes + (bytes >> 2) + 4096;
        cudaError_t e = cudaMalloc(&ctx->scratch, want);
        if (e != cudaSuccess) {
            es_set_error("scratch cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
            return ES_ERR_NOMEM;
        }
        ctx->scratch_bytes = want;
    }
    *out = ctx->scratch;
    return ES_OK;
}

int es_ctx_counters(es_ctx* ctx, size_t n, unsigned** out) {
    if (n > ctx->n_counters) {
        if (ctx->counters) ES_CHECK_CUDA(cudaFree(ctx->counters));
        ctx->counters = nullptr;
        ctx->n_counters = 0;
        size_t want = n * 2 + 64;
        cudaError_t e = cudaMalloc((void**)&ctx->counters, want * sizeof(unsigned));
        if (e != cudaSuccess) {
            es_set_error("counter cudaMalloc failed: %s", cudaGetErrorString(e));
            return ES_ERR_NOMEM;
        }
        ES_CHECK_CUDA(cudaMemset(ctx->counters, 0, want * sizeof(unsigned)));
        ctx->n_counters = want;
    }
    *out = ctx->counters;
    return ES_OK;
}

extern "C" {

int es_abi_version(void) { return 1; }

const char* es_last_error(void) { return g_err; }

int es_ctx_create(int device, es_ctx** out) {
    ES_REQUIRE(out != nullptr, "es_ctx_create: out is NULL");
    int n = 0;
    ES_CHECK_CUDA(cudaGetDeviceCount(&n));
    ES_REQUIRE(device >= 0 && device < n, "es_ctx_create: device %d out of range (%d devices)", device, n);
    ES_CHECK_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    ES_CHECK_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        es_set_error("es_ctx_create: device %d is sm_%d%d; this library is built for sm_100a only", device,
                     prop.major, prop.minor);
        return ES_ERR_UNSUPPORTED;
    }
    es_ctx* c = (es_ctx*)calloc(1, sizeof(es_ctx));
    if (!c) return ES_ERR_NOMEM;
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    {   // mapped error word for kernel-side argument checks (see es_checked_slice)
        int* h = nullptr;
        if (cudaHostAlloc((void**)&h, sizeof(int), cudaHostAllocMapped) == cudaSuccess) {
            *h = 0;
            int* d = nullptr;
            if (cudaHostGetDevicePointer((void**)&d, h, 0) == cudaSuccess) { c->err_host = h; c->err_dev = d; }
            else cudaFreeHost(h);
        }
        (void)cudaGetLastError();
    }
    *out = c;
    return ES_OK;
}

int es_ctx_destroy(es_ctx* ctx) {
    if (!ctx) return ES_OK;
    cudaSetDevice(ctx->device);
    if (ctx->scratch) cudaFree(ctx->scratch);
    if (ctx->counters) cudaFree(ctx->counters);
    es_tc2_free_shadows(ctx);
    if (ctx->err_host) cudaFreeHost((void*)ctx->err_host);
    free(ctx);
    return ES_OK;
}

int es_noise_table_changed(es_ctx* ctx) {
    if (!ctx) return ES_ERR_INVALID;
    ctx->sh16_src = nullptr;            // the shadows (if any) are rebuilt by the next tensor-core rollout
    ctx->sh16_len = 0;
    return ES_OK;
}

static int es_async_error(es_ctx* ctx, const char* where) {
    if (ctx->err_host && *ctx->err_host) {
        const int code = *ctx->err_host;
        *ctx->err_host = 0;
        if (code == ES_ASYNC_BAD_INDEX)
            es_set_error("%s: a previous kernel was given a noise index outside the table (index < 0 or index + n_params >= "
                         "table length; the reference asserts this in NoiseTable.get, src/core/noisetable.py:34): the "
                         "results of that call are invalid", where);
        else if (code == ES_ASYNC_RNG_OVERFLOW)
            es_set_error("%s: es_draw_noisy consumed more MT19937 words than its jump-ahead pass had generated (a > 12 sigma "
                         "event of the polar method's acceptance count, or a bug): the draws of that call are invalid; set "
                         "ES_MT_JUMP=0 to use the sequential kernel", where);
        else
            es_set_error("%s: a previous kernel reported error %d", where, code);
        return ES_ERR_INVALID;
    }
    return ES_OK;
}

int es_check_async(es_ctx* ctx) {
    if (!ctx) { es_set_error("es_check_async: ctx is NULL"); return ES_ERR_INVALID; }
    return es_async_error(ctx, "es_check_async");
}

int64_t es_launch_count(const es_ctx* ctx) { return ctx ? ctx->launches : -1; }
int es_sm_count(const es_ctx* ctx) { return ctx ? ctx->sm_count : -1; }

#define ES_ENTER(ctx)                                                        \
    ES_REQUIRE((ctx) != nullptr, "%s: ctx is NULL", __func__);               \
    ES_CHECK_CUDA(cudaSetDevice((ctx)->device));                             \
    do { int _a = es_async_error((ctx), __func__); if (_a) return _a; } while (0)

int es_draw_indices(es_ctx* ctx, uint32_t* mt_key, int32_t* mt_pos, int n_streams, int n_per_stream,
                    uint64_t upper_bound, int extra_words, int64_t* idx_out, uint32_t* extra_out, void* stream) {
    ES_ENTER(ctx);
    ES_REQUIRE(mt_key && mt_pos && idx_out, "es_draw_indices: NULL pointer");
    ES_REQUIRE(n_streams >= 0 && n_per_stream >= 0, "es_draw_indices: negative count");
    ES_REQUIRE(extra_words >= 0 && extra_words <= 7, "es_draw_indices: extra_words must be in [0,7]");
    // NoiseTable.sample_idx raises ValueError when upper_bound <= 0 (noisetable.py:39)
    ES_REQUIRE(upper_bound >= 1, "es_draw_indices: upper_bound must be >= 1 (network too large for noise table)");
    if (upper_bound - 1 >= 0xFFFFFFFFull) {
        es_set_error("es_draw_indices: ranges >= 2^32 use numpy's 64-bit draw path, not implemented");
        return ES_ERR_UNSUPPORTED;
    }
    if (n_streams == 0 || n_per_stream == 0) return ES_OK;
    return es_impl_draw_indices(ctx, mt_key, mt_pos, n_streams, n_per_stream, upper_bound, extra_words, idx_out,
                                extra_out, (cudaStream_t)stream);
}

int es_mt_skip(es_ctx* ctx, uint32_t* mt_key, int32_t* mt_pos, int n_streams, int n_words, void* stream) {
    ES_ENTER(ctx);
    ES_REQUIRE(mt_key && mt_pos, "es_mt_skip: NULL pointer");
    ES_REQUIRE(n_streams >= 0 && n_words >= 0, "es_mt_skip: negative count");
    if (n_streams == 0 || n_words == 0) return ES_OK;
    return es_impl_mt_skip(ctx, mt_key, mt_pos, n_streams, n_words, (cudaStream_t)stream);
}

int es_perturb(es_ctx* ctx, const float* theta, const float* table, int64_t table_len, const int64_t* idx, int n_idx,
               int P, float sigma, float* out_pos, float* out_neg, void* stream) {
    ES_ENTER(ctx);
    ES_REQUIRE(theta && table && idx && out_pos, "es_perturb: NULL pointer");
    ES_REQUIRE(n_idx >= 0 && P > 0 && table_len > P, "es_perturb: bad sizes");
    if (n_idx == 0) return ES_OK;
    return es_impl_perturb(ctx, theta, table, table_len, idx, n_idx, P, sigma, out_pos, out_neg, (cudaStream_t)stream);
}

int es_normalise_obs(es_ctx* ctx, const float* obs, const double* mean, const double* std, double clip, int rows,
                     int obs_dim, float* out, void* stream) {
    ES_ENTER(ctx);
    ES_REQUIRE(obs && mean && std && out, "es_normalise_obs: NULL pointer");
    ES_REQUIRE(rows >= 0 && obs_dim > 0, "es_normalise_obs: bad sizes");
    if (rows == 0) return ES_OK;
    return es_impl_normalise_obs(ctx, obs, mean, std, clip, rows, obs_dim, out, (cudaStream_t)stream);
}

int es_obs_colsum(es_ctx* ctx, const float* obs, int rows, int obs_dim, float* sum_out, float* sumsq_out, void* stream) {
    ES_ENTER(ctx);
    ES_REQUIRE(obs && sum_out && sumsq_out, "es_obs_colsum: NULL pointer");
    ES_REQUIRE(rows >= 0 && obs_dim > 0, "es_obs_colsum: bad sizes");
    return es_impl_obs_colsum(ctx, obs, rows, obs_dim, sum_out, sumsq_out, (cudaStream_t)stream);
}

int es_obstat_accumulate(es_ctx* ctx, double* sum, double* sumsq, const float* s, const float* ssq, int obs_dim,
                         int n_rollouts, void* stream) {
    ES_ENTER(ctx);
    ES_REQUIRE(sum && sumsq && s && ssq, "es_obstat_accumulate: NULL pointer");
    ES_REQUIRE(obs_dim > 0 && n_rollouts >= 0, "es_obstat_accumulate: bad sizes");
    if (n_rollouts == 0) return ES_OK;
    return es_impl_obstat_accumulate(ctx, sum, sumsq, s, ssq, obs_dim, n_rollouts, (cudaStream_t)stream);
}

int es_obstat_accumulate_coins(es_ctx* ctx, double* sum, double* sumsq, double* count_io, const float* s,
                               const float* ssq, int obs_dim, int rows_per_rollout, const uint32_t* coin_words,
                               int n_coins, double chance, void* stream) {
    ES_ENTER(ctx);
    ES_REQUIRE(sum && sumsq && count_io && s && ssq && (coin_words || n_coins == 0),
               "es_obstat_accumulate_coins: NULL pointer");
    ES_REQUIRE(obs_dim > 0 && n_coins >= 0 && rows_per_rollout >= 0, "es_obstat_accumulate_coins: bad sizes");
    return es_impl_obstat_accumulate_coins(ctx, sum, sumsq, count_io, s, ssq, obs_dim, rows_per_rollout, coin_words,
                                           n_coins, chance, (cudaStream_t)stream);
}

// es_rollout_openloop_noisy (n_episodes = 1) and es_rollout_openloop_episodes: validation and dispatch
static int rollout_openloop(es_ctx* ctx, const float* table, int64_t table_len, const int64_t* idx, int n_pairs,
                            const float* theta, int P, float sigma, const int* layer_sizes, int n_layers, const float* obsn,
                            const float* rew_vec, int T, float pos_scale, double* fit_pos, double* fit_neg, int fit_stride,
                            float* behv_pos, float* behv_neg, const float* act_noise, int n_eps, int mode, cudaStream_t stream) {
    ES_REQUIRE(table && idx && theta && layer_sizes && obsn && rew_vec && fit_pos && fit_neg,
               "es_rollout_openloop: NULL pointer");
    ES_REQUIRE(n_layers >= 1 && n_layers <= ES_MAX_LAYERS, "es_rollout_openloop: n_layers must be in [1,%d]",
               ES_MAX_LAYERS);
    ES_REQUIRE(n_pairs >= 0 && T >= 1 && fit_stride >= 1, "es_rollout_openloop: bad sizes");
    ES_REQUIRE((behv_pos == nullptr) == (behv_neg == nullptr), "es_rollout_openloop: behv_pos/behv_neg must both be set or NULL");
    int64_t count = 0;
    for (int l = 0; l < n_layers; ++l) {
        ES_REQUIRE(layer_sizes[l] > 0 && layer_sizes[l + 1] > 0, "es_rollout_openloop: layer size <= 0");
        count += (int64_t)layer_sizes[l] * layer_sizes[l + 1] + layer_sizes[l + 1];
    }
    ES_REQUIRE(count == P, "es_rollout_openloop: layer sizes give %lld params, P=%d", (long long)count, P);
    ES_REQUIRE(table_len > P, "es_rollout_openloop: table smaller than the network");
    ES_REQUIRE(n_eps >= 1, "es_rollout_openloop_episodes: n_episodes must be >= 1, got %d", n_eps);
    if (!act_noise) n_eps = 1;          // noise-free episodes are all the same episode: their average is its reward, exactly
    ES_REQUIRE(n_eps == 1 || (int64_t)n_eps * T * layer_sizes[n_layers] <= 0x7FFFFFFF,
               "es_rollout_openloop_episodes: n_episodes * T * act_dim = %lld exceeds INT_MAX (es_draw_noisy's normals_per_eval)",
               (long long)n_eps * T * layer_sizes[n_layers]);
    if (n_pairs == 0) return ES_OK;
    if (mode == ES_ROLLOUT_F32)
        return es_impl_rollout_f32(ctx, table, table_len, idx, n_pairs, theta, P, sigma, layer_sizes, n_layers, obsn,
                                   rew_vec, T, pos_scale, fit_pos, fit_neg, fit_stride, behv_pos, behv_neg,
                                   act_noise, n_eps, stream);
    if (mode == ES_ROLLOUT_TC || mode == ES_ROLLOUT_TC3) {
        // obs-64-64-act: rollout_tc2.cu (layer 1 shared by both signs through U +- sigma V); 2..4 hidden layers of 64..256
        // (multiples of 64): rollout_tcw.cu (per-pair weight images streamed through shared memory)
        const bool h64 = n_layers == 3 && layer_sizes[1] == 64 && layer_sizes[2] == 64;
        if (!h64 && es_tcw_covers(layer_sizes, n_layers))
            return es_impl_rollout_tcw(ctx, mode == ES_ROLLOUT_TC3, table, table_len, idx, n_pairs, theta, P, sigma, layer_sizes,
                                       n_layers, obsn, rew_vec, T, pos_scale, fit_pos, fit_neg, fit_stride, behv_pos, behv_neg,
                                       act_noise, n_eps, stream);
        if (!h64) {
            es_set_error("es_rollout_openloop(TC): the tensor-core path covers tanh MLPs obs(<=1023) -> 2..4 hidden layers "
                         "(each a multiple of 64 in [64, 256]) -> act(<=32); use ES_ROLLOUT_F32 for other shapes");
            return ES_ERR_UNSUPPORTED;
        }
        return es_impl_rollout_tc2(ctx, mode == ES_ROLLOUT_TC3, table, table_len, idx, n_pairs, theta, P, sigma, layer_sizes, n_layers,
                                   obsn, rew_vec, T, pos_scale, fit_pos, fit_neg, fit_stride, behv_pos, behv_neg,
                                   act_noise, n_eps, stream);
    }
    es_set_error("es_rollout_openloop: unknown mode %d", mode);
    return ES_ERR_INVALID;
}

int es_rollout_openloop_noisy(es_ctx* ctx, const float* table, int64_t table_len, const int64_t* idx, int n_pairs,
                              const float* theta, int P, float sigma, const int* layer_sizes, int n_layers, const float* obsn,
                              const float* rew_vec, int T, float pos_scale, double* fit_pos, double* fit_neg, int fit_stride,
                              float* behv_pos, float* behv_neg, const float* act_noise, int mode, void* stream) {
    ES_ENTER(ctx);
    return rollout_openloop(ctx, table, table_len, idx, n_pairs, theta, P, sigma, layer_sizes, n_layers, obsn, rew_vec, T, pos_scale,
                            fit_pos, fit_neg, fit_stride, behv_pos, behv_neg, act_noise, 1, mode, (cudaStream_t)stream);
}

int es_rollout_openloop_episodes(es_ctx* ctx, const float* table, int64_t table_len, const int64_t* idx, int n_pairs,
                                 const float* theta, int P, float sigma, const int* layer_sizes, int n_layers, const float* obsn,
                                 const float* rew_vec, int T, float pos_scale, double* fit_pos, double* fit_neg, int fit_stride,
                                 float* behv_pos, float* behv_neg, const float* act_noise, int n_episodes, int mode, void* stream) {
    ES_ENTER(ctx);
    return rollout_openloop(ctx, table, table_len, idx, n_pairs, theta, P, sigma, layer_sizes, n_layers, obsn, rew_vec, T, pos_scale,
                            fit_pos, fit_neg, fit_stride, behv_pos, behv_neg, act_noise, n_episodes, mode, (cudaStream_t)stream);
}

int es_rollout_openloop(es_ctx* ctx, const float* table, int64_t table_len, const int64_t* idx, int n_pairs,
                        const float* theta, int P, float sigma, const int* layer_sizes, int n_layers, const float* obsn,
                        const float* rew_vec, int T, float pos_scale, double* fit_pos, double* fit_neg, int fit_stride,
                        float* behv_pos, float* behv_neg, int mode, void* stream) {
    return es_rollout_openloop_noisy(ctx, table, table_len, idx, n_pairs, theta, P, sigma, layer_sizes, n_layers, obsn, rew_vec, T,
                                     pos_scale, fit_pos, fit_neg, fit_stride, behv_pos, behv_neg, nullptr, mode, stream);
}

int es_rollout_closedloop(es_ctx* ctx, const float* table, int64_t table_len, const int64_t* idx, int n_pairs, const float* theta,
                          int P, float sigma, const int* layer_sizes, int n_layers, const double* ob_mean, const double* ob_std,
                          double ob_clip, const float* obs0, const float* env_a, int band, const float* env_b, const float* rew_vec,
                          int T, float pos_scale, const uint32_t* coin_words, double save_obs_chance, double* fit_pos,
                          double* fit_neg, int fit_stride, float* behv_pos, float* behv_neg, double* ob_sum, double* ob_sumsq,
                          double* ob_count, void* stream) {
    ES_ENTER(ctx);
    ES_REQUIRE(table && idx && theta && layer_sizes && ob_mean && ob_std && obs0 && env_a && env_b && rew_vec && fit_pos && fit_neg,
               "es_rollout_closedloop: NULL pointer");
    if (n_layers != 3) {
        es_set_error("es_rollout_closedloop: two hidden layers (n_layers == 3) supported, got %d", n_layers);
        return ES_ERR_UNSUPPORTED;
    }
    ES_REQUIRE(n_pairs >= 0 && T >= 1 && fit_stride >= 1 && band >= 1, "es_rollout_closedloop: bad sizes");
    ES_REQUIRE((behv_pos == nullptr) == (behv_neg == nullptr), "es_rollout_closedloop: behv_pos/behv_neg must both be set or NULL");
    ES_REQUIRE((ob_sum == nullptr) == (ob_sumsq == nullptr) && (ob_sum == nullptr) == (ob_count == nullptr),
               "es_rollout_closedloop: ob_sum/ob_sumsq/ob_count must all be set or NULL");
    int64_t count = 0;
    for (int l = 0; l < n_layers; ++l) {
        ES_REQUIRE(layer_sizes[l] > 0 && layer_sizes[l + 1] > 0, "es_rollout_closedloop: layer size <= 0");
        count += (int64_t)layer_sizes[l] * layer_sizes[l + 1] + layer_sizes[l + 1];
    }
    ES_REQUIRE(count == P, "es_rollout_closedloop: layer sizes give %lld params, P=%d", (long long)count, P);
    ES_REQUIRE(table_len > P, "es_rollout_closedloop: table smaller than the network");
    ES_REQUIRE(band <= layer_sizes[0], "es_rollout_closedloop: band wider than the observation");
    if (n_pairs == 0) return ES_OK;
    return es_impl_rollout_closed(ctx, table, table_len, idx, n_pairs, theta, P, sigma, layer_sizes, ob_mean, ob_std, ob_clip, obs0,
                                  env_a, band, env_b, rew_vec, T, pos_scale, coin_words, save_obs_chance, fit_pos, fit_neg, fit_stride,
                                  behv_pos, behv_neg, ob_sum, ob_sumsq, ob_count, (cudaStream_t)stream);
}

int es_draw_noisy(es_ctx* ctx, uint32_t* mt_key, int32_t* mt_pos, int32_t* has_gauss, double* gauss, int n_streams,
                  int n_per_stream, uint64_t upper_bound, int coins_per_eval, int normals_per_eval, double scale,
                  int64_t* idx_out, uint32_t* coin_out, float* noise_out, void* stream) {
    ES_ENTER(ctx);
    ES_REQUIRE(mt_key && mt_pos && has_gauss && gauss && idx_out && noise_out, "es_draw_noisy: NULL pointer");
    ES_REQUIRE(n_streams >= 0 && n_per_stream >= 0 && normals_per_eval >= 0, "es_draw_noisy: negative count");
    ES_REQUIRE(coins_per_eval >= 0 && coins_per_eval <= 8, "es_draw_noisy: coins_per_eval must be in [0,8]");
    ES_REQUIRE(coins_per_eval == 0 || coin_out, "es_draw_noisy: coin_out is NULL");
    // NoiseTable.sample_idx raises ValueError when upper_bound <= 0 (noisetable.py:39)
    ES_REQUIRE(upper_bound >= 1, "es_draw_noisy: upper_bound must be >= 1 (network too large for noise table)");
    if (upper_bound - 1 >= 0xFFFFFFFFull) {
        es_set_error("es_draw_noisy: ranges >= 2^32 use numpy's 64-bit draw path, not implemented");
        return ES_ERR_UNSUPPORTED;
    }
    if (n_streams == 0 || n_per_stream == 0) return ES_OK;
    return es_impl_draw_noisy(ctx, mt_key, mt_pos, has_gauss, gauss, n_streams, n_per_stream, upper_bound, coins_per_eval,
                              normals_per_eval, scale, idx_out, coin_out, noise_out, (cudaStream_t)stream);
}

int es_novelty(es_ctx* ctx, const float* behv, int n, const double* archive, int A, int k, double* out, int out_stride,
               void* stream) {
    ES_ENTER(ctx);
    ES_REQUIRE(behv && archive && out, "es_novelty: NULL pointer");
    ES_REQUIRE(n >= 0 && A >= 1 && k >= 1 && out_stride >= 1, "es_novelty: bad sizes");
    ES_REQUIRE((k < A ? k : A) <= 64, "es_novelty: min(k, archive size) > 64 not supported");
    if (n == 0) return ES_OK;
    return es_impl_novelty(ctx, behv, n, archive, A, k, out, out_stride, (cudaStream_t)stream);
}

int es_centered_rank(es_ctx* ctx, const double* fpos, const double* fneg, int K, int n_obj, float w0, float w1,
                     int k_begin, int k_count, float* weights_out, int32_t* ranks_out, void* stream) {
    ES_ENTER(ctx);
    ES_REQUIRE(fpos && fneg && weights_out, "es_centered_rank: NULL pointer");
    // MultiObjectiveRanker asserts exactly two columns (rankers.py:114)
    ES_REQUIRE(n_obj == 1 || n_obj == 2, "es_centered_rank: n_obj must be 1 or 2");
    ES_REQUIRE(K >= 1 && k_begin >= 0 && k_count >= 0 && k_begin + k_count <= K, "es_centered_rank: bad shard");
    if (k_count == 0) return ES_OK;
    return es_impl_rank_transform(ctx, fpos, fneg, K, n_obj, ES_RANK_CENTERED, (double)w0, (double)w1, 0, k_begin, k_count,
                                  nullptr, weights_out, nullptr, ranks_out, nullptr, nullptr, nullptr,
                                  (cudaStream_t)stream);
}

int es_rank_transform(es_ctx* ctx, const double* fpos, const double* fneg, int K, int n_obj, int kind, double w0,
                      double w1, int elite_n, int k_begin, int k_count, const int64_t* noise_idx, float* weights_out,
                      double* weights64_out, int32_t* ranks_out, double* elite_vals_out, int32_t* elite_fit_out,
                      int64_t* elite_idx_out, void* stream) {
    ES_ENTER(ctx);
    ES_REQUIRE(fpos && fneg && weights_out, "es_rank_transform: NULL pointer");
    ES_REQUIRE(kind >= ES_RANK_CENTERED && kind <= ES_RANK_MAX_NORMALIZED, "es_rank_transform: unknown kind");
    ES_REQUIRE(n_obj == 1 || n_obj == 2, "es_rank_transform: n_obj must be 1 or 2");   // rankers.py:114
    ES_REQUIRE(K >= 1 && k_begin >= 0 && k_count >= 0 && k_begin + k_count <= K, "es_rank_transform: bad shard");
    ES_REQUIRE(elite_n >= 0 && elite_n <= 2 * K, "es_rank_transform: elite_n out of range");
    if (elite_n > 0) {
        // EliteRanker(MultiObjectiveRanker) would need a second ranking of the blended values: not provided
        if (n_obj != 1) { es_set_error("es_rank_transform: elite selection needs a single objective"); return ES_ERR_UNSUPPORTED; }
        ES_REQUIRE(!elite_idx_out || noise_idx, "es_rank_transform: elite_idx_out needs noise_idx");
    }
    if (k_count == 0) return ES_OK;
    return es_impl_rank_transform(ctx, fpos, fneg, K, n_obj, kind, w0, w1, elite_n, k_begin, k_count, noise_idx,
                                  weights_out, weights64_out, ranks_out, elite_vals_out, elite_fit_out, elite_idx_out,
                                  (cudaStream_t)stream);
}

int es_grad_reconstruct(es_ctx* ctx, const float* table, int64_t table_len, const int64_t* idx, const float* weights,
                        int n_idx, int P, float* out, void* stream) {
    ES_ENTER(ctx);
    ES_REQUIRE(table && out, "es_grad_reconstruct: NULL pointer");
    ES_REQUIRE(n_idx >= 0 && P > 0 && table_len > P, "es_grad_reconstruct: bad sizes");
    ES_REQUIRE(n_idx == 0 || (idx && weights), "es_grad_reconstruct: NULL idx/weights");
    if (n_idx == 0) {
        ES_CHECK_CUDA(cudaMemsetAsync(out, 0, (size_t)P * sizeof(float), (cudaStream_t)stream));
        return ES_OK;
    }
    return es_impl_grad_reconstruct(ctx, table, table_len, idx, weights, n_idx, P, out, (cudaStream_t)stream);
}

int es_adam_step(es_ctx* ctx, float* theta, float* m, float* v, const float* gsum, float n_ranked, float l2coeff,
                 float neg_a, float beta1, float one_minus_beta1, float beta2, float one_minus_beta2, float epsilon,
                 int P, void* stream) {
    ES_ENTER(ctx);
    ES_REQUIRE(theta && m && v && gsum && P > 0, "es_adam_step: bad arguments");
    return es_impl_adam(ctx, theta, m, v, gsum, n_ranked, l2coeff, neg_a, beta1, one_minus_beta1, beta2,
                        one_minus_beta2, epsilon, P, (cudaStream_t)stream);
}

int es_sgd_step(es_ctx* ctx, float* theta, float* v, const float* gsum, float n_ranked, float l2coeff, float neg_lr,
                float momentum, float one_minus_momentum, int P, void* stream) {
    ES_ENTER(ctx);
    ES_REQUIRE(theta && v && gsum && P > 0, "es_sgd_step: bad arguments");
    return es_impl_sgd(ctx, theta, v, gsum, n_ranked, l2coeff, neg_lr, momentum, one_minus_momentum, P,
                       (cudaStream_t)stream);
}

int es_simple_step(es_ctx* ctx, float* theta, const float* gsum, float n_ranked, float l2coeff, float lr, int P,
                   void* stream) {
    ES_ENTER(ctx);
    ES_REQUIRE(theta && gsum && P > 0, "es_simple_step: bad arguments");
    return es_impl_simple(ctx, theta, gsum, n_ranked, l2coeff, lr, P, (cudaStream_t)stream);
}

}  // extern "C"
