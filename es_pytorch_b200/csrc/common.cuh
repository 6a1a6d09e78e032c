// common.cuh -- shared host/device helpers for libes_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include "../../include/es_b200.h"

#ifndef __CUDA_ARCH_LIST__
#endif

struct es_ctx {
    int device;
    int sm_count;
    int64_t launches;
    // scratch owned by the ctx (grown on demand, never shrunk)
    void* scratch;          // generic scratch (reconstruct partials, rank keys, ...)
    size_t scratch_bytes;
    unsigned* counters;     // small zero-initialised counter array (last-block detection)
    size_t n_counters;
    // float16 shadows for rollout_tc2.cu: hi = f16(table), lo = f16(table - hi) (split rollout only), 8 shifted copies each,
    // plus the two TMA tensor maps over them (host copy, 64-byte aligned)
    const float* sh16_src;
    int64_t sh16_len;
    void* sh16_hi;
    void* sh16_lo;
    void* sh16_maps;
    int sh16_maps_lo;
    size_t sh16_stride;
    int sh16_obs;
    int sh16_failed;
    // asynchronous kernel-side argument errors: a mapped, page-locked host word the kernels set when a noise index is
    // out of range (the reference asserts `len > i + size`, src/core/noisetable.py:34); surfaced by es_check_async and
    // by the next entry point
    volatile int* err_host;
    int* err_dev;
    int mj_lists_ready;     // mt_gauss.cu: the set-bit lists of the jump polynomials have been built on this device
};

#define ES_ASYNC_BAD_INDEX 1
#define ES_ASYNC_RNG_OVERFLOW 2      // es_draw_noisy (jump-ahead path): the stream consumed more words than were generated ahead

void es_set_error(const char* fmt, ...);

#define ES_CHECK_CUDA(expr)                                                              \
    do {                                                                                 \
        cudaError_t _e = (expr);                                                         \
        if (_e != cudaSuccess) {                                                         \
            es_set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #expr,              \
                         cudaGetErrorString(_e));                                        \
            return ES_ERR_CUDA;                                                          \
        }                                                                                \
    } while (0)

#define ES_REQUIRE(cond, ...)                                                            \
    do {                                                                                 \
        if (!(cond)) {                                                                   \
            es_set_error(__VA_ARGS__);                                                   \
            return ES_ERR_INVALID;                                                       \
        }                                                                                \
    } while (0)

// after a kernel launch: count it and surface launch-configuration errors
#define ES_LAUNCHED(ctx)                                                                 \
    do {                                                                                 \
        (ctx)->launches++;                                                               \
        ES_CHECK_CUDA(cudaGetLastError());                                               \
    } while (0)

int es_ctx_scratch(es_ctx* ctx, size_t bytes, void** out);
int es_ctx_counters(es_ctx* ctx, size_t n, unsigned** out);

static inline int es_div_up(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// ---- entry points implemented one per .cu file (called from api.cu) -------------------------
int es_impl_draw_indices(es_ctx*, uint32_t*, int32_t*, int, int, uint64_t, int, int64_t*, uint32_t*, cudaStream_t);
int es_impl_mt_skip(es_ctx*, uint32_t*, int32_t*, int, int, cudaStream_t);
int es_impl_perturb(es_ctx*, const float*, const float*, int64_t, const int64_t*, int, int, float, float*, float*,
                    cudaStream_t);
int es_impl_normalise_obs(es_ctx*, const float*, const double*, const double*, double, int, int, float*, cudaStream_t);
int es_impl_obs_colsum(es_ctx*, const float*, int, int, float*, float*, cudaStream_t);
int es_impl_obstat_accumulate(es_ctx*, double*, double*, const float*, const float*, int, int, cudaStream_t);
int es_impl_obstat_accumulate_coins(es_ctx*, double*, double*, double*, const float*, const float*, int, int,
                                    const uint32_t*, int, double, cudaStream_t);
int es_impl_draw_noisy(es_ctx*, uint32_t*, int32_t*, int32_t*, double*, int, int, uint64_t, int, int, double, int64_t*, uint32_t*,
                       float*, cudaStream_t);
// (the trailing const float*, int of the rollouts: scaled action noise [n_pairs][2][n_eps][T][act], or NULL, and the number
// of episodes per evaluation n_eps; n_eps > 1 only with noise)
int es_impl_rollout_f32(es_ctx*, const float*, int64_t, const int64_t*, int, const float*, int, float, const int*, int,
                        const float*, const float*, int, float, double*, double*, int, float*, float*, const float*, int,
                        cudaStream_t);
int es_impl_rollout_f32x(es_ctx*, const float*, int64_t, const int64_t*, int, const float*, int, float, const int*, int,
                         const float*, const float*, int, float, double*, double*, int, float*, float*, const float*, int,
                         cudaStream_t);
int es_impl_rollout_tc2(es_ctx*, int split, const float*, int64_t, const int64_t*, int, const float*, int, float, const int*,
                        int, const float*, const float*, int, float, double*, double*, int, float*, float*, const float*, int,
                        cudaStream_t);
void es_tc2_free_shadows(es_ctx* ctx);
int es_impl_rollout_tcw(es_ctx*, int split, const float*, int64_t, const int64_t*, int, const float*, int, float, const int*,
                        int, const float*, const float*, int, float, double*, double*, int, float*, float*, const float*, int,
                        cudaStream_t);
int es_tcw_covers(const int* layer_sizes, int n_layers);      // shapes of rollout_tcw.cu
int es_impl_rollout_closed(es_ctx*, const float*, int64_t, const int64_t*, int, const float*, int, float, const int*, const double*,
                           const double*, double, const float*, const float*, int, const float*, const float*, int, float,
                           const uint32_t*, double, double*, double*, int, float*, float*, double*, double*, double*, cudaStream_t);
int es_impl_novelty(es_ctx*, const float*, int, const double*, int, int, double*, int, cudaStream_t);
int es_impl_rank_transform(es_ctx*, const double*, const double*, int, int, int, double, double, int, int, int,
                           const int64_t*, float*, double*, int32_t*, double*, int32_t*, int64_t*, cudaStream_t);
int es_impl_grad_reconstruct(es_ctx*, const float*, int64_t, const int64_t*, const float*, int, int, float*,
                             cudaStream_t);
int es_impl_adam(es_ctx*, float*, float*, float*, const float*, float, float, float, float, float, float, float, float,
                 int, cudaStream_t);
int es_impl_sgd(es_ctx*, float*, float*, const float*, float, float, float, float, float, int, cudaStream_t);
int es_impl_simple(es_ctx*, float*, const float*, float, float, float, int, cudaStream_t);

#ifdef __CUDACC__
// start of the noise slice of one perturbation, checked like NoiseTable.get (src/core/noisetable.py:34:
// `assert len(self) > i + size`).  An out-of-range index is reported through the ctx's mapped error word and replaced
// by 0 (a valid address): the launch's results are garbage and the caller is told so by the next entry point /
// es_check_async.
__device__ __forceinline__ long long es_checked_slice(long long i, int P, long long table_len, int* err) {
    if (i < 0 || i + (long long)P >= table_len) {
        if (err) *(volatile int*)err = ES_ASYNC_BAD_INDEX;
        return 0;
    }
    return i;
}
__device__ __forceinline__ float es_warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int es_warp_sum_i(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
#endif
