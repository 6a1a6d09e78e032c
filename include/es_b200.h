/* es_b200.h -- C ABI of libes_b200.so: the B200 (sm_100a) OpenAI-ES generation step.
 *
 * The reference (sash-a/es_pytorch) is pure Python; its boundary for this path is
 * the Python API of src.core / src.nn / src.utils.  Each entry point below replaces
 * the arithmetic of one reference function (cited as file:line into the reference
 * checkout); the Python mirror in es_pytorch_b200/ binds them with ctypes.
 *
 * Conventions
 *   - every pointer marked "dev" is a device pointer owned by the caller (a torch
 *     tensor's storage); the library never frees or retains it past the call;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *     all work is enqueued asynchronously on it, nothing synchronises the device;
 *   - return value: 0 = ok, negative = error (ES_ERR_*); es_last_error() returns a
 *     thread-local message for the last failing call;
 *   - one es_ctx per device and per host thread; the ctx owns scratch buffers only.
 */
#ifndef ES_B200_H
#define ES_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ES_OK                 0
#define ES_ERR_INVALID       -1   /* bad argument                                   */
#define ES_ERR_CUDA          -2   /* a CUDA runtime call failed                     */
#define ES_ERR_UNSUPPORTED   -3   /* shape / mode not implemented by this build     */
#define ES_ERR_NOMEM         -4

#define ES_MAX_LAYERS         8
#define ES_MT_N             624   /* MT19937 state words                            */

typedef struct es_ctx es_ctx;

/* ---- context ------------------------------------------------------------------ */
int         es_ctx_create(int device, es_ctx** out);
int         es_ctx_destroy(es_ctx* ctx);
const char* es_last_error(void);
int         es_abi_version(void);
/* Kernel-side argument errors are asynchronous: a kernel that is handed a noise index outside the table (index < 0 or
 * index + n_params >= table_len -- NoiseTable.get asserts `len(self) > i + size`, src/core/noisetable.py:34) flags it in
 * a mapped host word, substitutes index 0 and carries on; the results of that launch are invalid.  es_check_async
 * returns ES_ERR_INVALID (once) if any kernel launched through this ctx and completed so far has flagged an error;
 * call it after synchronising the stream.  Every entry point performs the same check on entry.                    */
int         es_check_async(es_ctx* ctx);
/* kernels launched through this ctx since creation (bench.py's "gpu_launches"). */
int64_t     es_launch_count(const es_ctx* ctx);
int         es_sm_count(const es_ctx* ctx);

/* ---- a2: draw noise indices ------------------------------------------------------
 * Replaces NoiseTable.sample_idx, src/core/noisetable.py:37-40, as called n times per
 * rank from es.test_params, src/core/es.py:67-68: numpy's legacy
 * RandomState.randint(0, upper_bound) = MT19937 + masked rejection, bit-exact.
 * One independent stream per virtual MPI rank (src/utils/utils.py:63-65).  After each
 * accepted index the next `extra_words` raw 32-bit outputs of the same stream are
 * consumed and returned (4 = the two rs.random() save_obs coins of one antithetic
 * pair, simple_example.py:38 / obj.py:54; 0 = index-only).
 *   mt_key  dev uint32 [n_streams][624]  in/out  (RandomState.get_state()[1])
 *   mt_pos  dev int32  [n_streams]       in/out  (get_state()[2], 0..624)
 *   idx_out dev int64  [n_streams*n_per_stream]  rank-major (es.py:89-95 order)
 *   extra_out dev uint32 [n_streams*n_per_stream][extra_words] or NULL            */
int es_draw_indices(es_ctx* ctx, uint32_t* mt_key, int32_t* mt_pos, int n_streams, int n_per_stream,
                    uint64_t upper_bound, int extra_words, int64_t* idx_out, uint32_t* extra_out,
                    void* stream);

/* Advance every stream by n_words 32-bit outputs without using them: the save_obs coin (rs.random() = 2 words) that the
 * scripts' fit_fn draws at the start of EVERY evaluation, including the noiseless one of es.step (src/core/es.py:48,
 * simple_example.py:38, obj.py:54) whose rollout is computed separately.                                              */
int es_mt_skip(es_ctx* ctx, uint32_t* mt_key, int32_t* mt_pos, int n_streams, int n_words, void* stream);

/* ---- a3: materialise theta +- sigma*eps -------------------------------------------
 * Replaces Policy.pheno's arithmetic, src/core/policy.py:61-64 (two separately
 * rounded float32 ops, no FMA).  out_neg may be NULL.  Used by the per-perturbation
 * compatibility path and by parity tests; the fused rollout never writes theta' out.
 *   out_pos/out_neg dev float [n_idx][P]                                            */
int es_perturb(es_ctx* ctx, const float* theta, const float* table, int64_t table_len, const int64_t* idx,
               int n_idx, int P, float sigma, float* out_pos, float* out_neg, void* stream);

/* ---- a4: observation normalisation -------------------------------------------------
 * clamp((o - mean) / std, +-clip) in float64, then float32: src/nn/nn.py:45.
 *   obs dev float [rows][obs_dim]; mean/std dev double [obs_dim]; out dev float      */
int es_normalise_obs(es_ctx* ctx, const float* obs, const double* mean, const double* std, double clip,
                     int rows, int obs_dim, float* out, void* stream);

/* ---- a3+a4+a5: fused perturb + batched MLP rollout + fitness ------------------------
 * For every antithetic pair k: W+- = theta +- sigma*table[idx[k] : idx[k]+P]
 * (policy.py:61-64), T steps of the FeedForward forward (Linear+tanh after every
 * layer, src/nn/nn.py:35-36,46) on the pre-normalised open-loop observation stream,
 * reward r_t = <a_t, rew_vec[t]> (float32), fitness = sum_t r_t accumulated in
 * float64 in step order (python sum(rews), src/gym/training_result.py:28,62-64), and
 * the synthetic env's position integrator pos += pos_scale * a_t[0..2].
 *   layer_sizes  host int [n_layers+1]  (obs_dim, hidden..., act_dim)
 *   obsn   dev float [T][obs_dim]   rew_vec dev float [T][act_dim]
 *   fit_pos/fit_neg dev double [n_pairs*fit_stride]  (element k*fit_stride)
 *   behv_pos/behv_neg dev float [n_pairs][3] or NULL (final x,y,z)
 *   mode: ES_ROLLOUT_F32 = float32 CUDA-core path (parity reference on device),
 *         ES_ROLLOUT_TC  = tcgen05 tensor-core path, float16 operands, tanh.approx (fast; fitness within ~1e-3 of the
 *                          population spread of the float32 result, see DESIGN.md)
 *         ES_ROLLOUT_TC3 = tcgen05 tensor-core path at float32-equivalent accuracy: every operand is split into
 *                          float16 hi + lo parts and every product is three MMAs (hi*hi + hi*lo + lo*hi), float32
 *                          accumulation in TMEM, accurate tanh, float64 fitness sums (see DESIGN.md)
 *         The tensor-core modes cover tanh MLPs with obs_dim <= 1023, act_dim <= 32 and either two hidden layers of 64
 *         (rollout_tc2.cu) or 2 to 4 hidden layers, each a multiple of 64 in [64, 256] (rollout_tcw.cu: the networks of
 *         the shipped configs); other shapes return ES_ERR_UNSUPPORTED.                                              */
#define ES_ROLLOUT_F32 0
#define ES_ROLLOUT_TC  1
#define ES_ROLLOUT_TC3 2
int es_rollout_openloop(es_ctx* ctx, const float* table, int64_t table_len, const int64_t* idx, int n_pairs,
                        const float* theta, int P, float sigma, const int* layer_sizes, int n_layers,
                        const float* obsn, const float* rew_vec, int T, float pos_scale,
                        double* fit_pos, double* fit_neg, int fit_stride, float* behv_pos, float* behv_neg,
                        int mode, void* stream);

/* The same with action noise: act_noise dev float [n_pairs][2 (+,-)][T][act_dim] (or NULL = es_rollout_openloop) is added to
 * the action of every step before the env sees it -- FeedForward.forward's `a += rs.randn(*a.shape) * self._action_std`
 * (src/nn/nn.py:47-48); reward and position are computed from the noisy action (src/gym/gym_runner.py:52-53).  The array is
 * what es_draw_noisy wrote for the same pairs.                                                                        */
int es_rollout_openloop_noisy(es_ctx* ctx, const float* table, int64_t table_len, const int64_t* idx, int n_pairs,
                              const float* theta, int P, float sigma, const int* layer_sizes, int n_layers,
                              const float* obsn, const float* rew_vec, int T, float pos_scale,
                              double* fit_pos, double* fit_neg, int fit_stride, float* behv_pos, float* behv_neg,
                              const float* act_noise, int mode, void* stream);

/* The same with n_episodes >= 1 episodes per evaluation (obj.py's r_fn: `for _ in range(max(1, eps_per_policy))` runs the
 * policy E times, adds the per-step rewards in a float64 array and divides it by E; behaviour = the last episode's).  On the
 * open-loop env the E episodes share their forward pass and differ only in the action noise:
 *   act_noise dev float [n_pairs][2 (+,-)][n_episodes][T][act_dim] (es_draw_noisy with normals_per_eval = n_episodes*T*act_dim)
 *   fitness   = (sum over steps and episodes of the float32 reward of episode e's noisy action, in float64) / n_episodes
 *   behv      = the final position of episode n_episodes - 1
 * With act_noise == NULL every episode is the noise-free one and the call is es_rollout_openloop (exact: the reference's
 * per-step average of E equal float32 rewards is that reward).  n_episodes * T * act_dim must not exceed INT_MAX
 * (ES_ERR_INVALID), the noise offsets are 64-bit.  n_episodes == 1 is es_rollout_openloop_noisy.                       */
int es_rollout_openloop_episodes(es_ctx* ctx, const float* table, int64_t table_len, const int64_t* idx, int n_pairs,
                                 const float* theta, int P, float sigma, const int* layer_sizes, int n_layers,
                                 const float* obsn, const float* rew_vec, int T, float pos_scale,
                                 double* fit_pos, double* fit_neg, int fit_stride, float* behv_pos, float* behv_neg,
                                 const float* act_noise, int n_episodes, int mode, void* stream);

/* ---- a3 + a4 + a5 on the CLOSED-LOOP synthetic env (SURVEY.md section 8d's optional variant; never part of the headline) --
 * obs_{t+1} = tanh(A obs_t + B a_t): the observation depends on the policy's own actions, so the episode runs step by step
 * with one pair's perturbed weights resident on chip (rollout_closed.cu).  Replaces the same reference loop as
 * es_rollout_openloop -- Policy.pheno (src/core/policy.py:61-64), FeedForward.forward incl. the observation normalisation
 * clip((ob - mean) / std) (src/nn/nn.py:42-50), run_model's reward / position / saved observations
 * (src/gym/gym_runner.py:33-67) -- plus the ObStat increments of the evaluations whose save_obs coin fell
 * (src/core/es.py:73-74, src/gym/training_result.py:17-21).
 *   layer_sizes host int [4] (obs, h1, h2, act): two hidden layers <= 64 units, obs <= 384, act <= 64
 *   ob_mean/ob_std dev double [obs]      obs0 dev float [obs]
 *   env_a dev float [band][obs] (A's diagonals, transposed: env_a[d][i] multiplies obs[(i + d - band/2) mod obs])
 *   env_b dev float [act][obs] (B transposed)   rew_vec dev float [T][act]
 *   coin_words dev uint32 [n_pairs][2 (+,-)][2] (the save_obs coin of every evaluation as drawn by es_draw_indices) or NULL
 *   ob_sum/ob_sumsq dev double [obs], ob_count dev double [2] (rows, rollouts): incremented atomically; or all NULL   */
int es_rollout_closedloop(es_ctx* ctx, const float* table, int64_t table_len, const int64_t* idx, int n_pairs,
                          const float* theta, int P, float sigma, const int* layer_sizes, int n_layers,
                          const double* ob_mean, const double* ob_std, double ob_clip,
                          const float* obs0, const float* env_a, int band, const float* env_b, const float* rew_vec, int T,
                          float pos_scale, const uint32_t* coin_words, double save_obs_chance,
                          double* fit_pos, double* fit_neg, int fit_stride, float* behv_pos, float* behv_neg,
                          double* ob_sum, double* ob_sumsq, double* ob_count, void* stream);

/* ---- a2 + a4 with action noise: all draws of a generation in stream order ---------------------------------------------
 * When FeedForward._action_std != 0 every step of every rollout draws rs.randn(act_dim) from the SAME RandomState that
 * draws the noise indices and the save_obs coins (src/nn/nn.py:47-48, src/core/es.py:66-72, simple_example.py:37-40).  Per
 * stream and pair, in the reference's order: randint (as es_draw_indices); then for the + and the - evaluation:
 * coins_per_eval doubles (2 words each), then normals_per_eval (= steps x act_dim) legacy polar-method gaussians
 * (numpy legacy_gauss, including the cached second value across calls).  The word stream is reproduced exactly (indices,
 * coin words, final key / position / has_gauss bit-exact; the cached gaussian to <= 1 ulp of float64, log() being CUDA's).
 *   has_gauss dev int32 [n_streams], gauss dev double [n_streams]   in/out  (RandomState.get_state()[3], [4])
 *   coin_out  dev uint32 [n_streams*n_per_stream][4*coins_per_eval]  (+ coins then - coins) or NULL when coins_per_eval == 0
 *   noise_out dev float [n_streams*n_per_stream][2][normals_per_eval] = float32(gaussian * scale), scale = ac_std          */
int es_draw_noisy(es_ctx* ctx, uint32_t* mt_key, int32_t* mt_pos, int32_t* has_gauss, double* gauss, int n_streams,
                  int n_per_stream, uint64_t upper_bound, int coins_per_eval, int normals_per_eval, double scale,
                  int64_t* idx_out, uint32_t* coin_out, float* noise_out, void* stream);

/* The tensor-core rollouts keep float16 shadows of the noise table (8 shifted copies of f16(table), 2 bytes x 8 x table_len
 * of HBM; ES_ROLLOUT_TC3 a second set for the low-order parts), built on first use and keyed by the table's device pointer,
 * its length and the policy's obs_dim.  The reference never writes to its table after NoiseTable.create_shared
 * (src/core/noisetable.py:66-91); a caller that does overwrite it in place must say so.  Table values must be finite and
 * below 65504 in magnitude (float16 range) for the tensor-core modes.                                               */
int es_noise_table_changed(es_ctx* ctx);

/* ---- a13: novelty ---------------------------------------------------------------------
 * mean of the k smallest euclidean distances (float64) between behv[e][0..1] and the
 * archive rows: src/utils/novelty.py:16-18, src/gym/training_result.py:82-97.
 *   behv dev float [n][3]; archive dev double [A][2]; out dev double, element e*out_stride */
int es_novelty(es_ctx* ctx, const float* behv, int n, const double* archive, int A, int k, double* out,
               int out_stride, void* stream);

/* ---- a8/a9: centered rank -> antithetic weights -------------------------------------------
 * Replaces Ranker.rank with CenteredRanker (src/utils/rankers.py:9-17,37-58) and, for
 * n_obj == 2, MultiObjectiveRanker (rankers.py:106-120): ranks over all 2K fitnesses
 * (pos then neg), y = float32(rank)/(2K-1) - 0.5, blend y0*w0 + y1*w1, weight[k] =
 * y[k] - y[K+k].  Ranks are integer-exact; ties broken by position (stable).  Only the
 * weights of pairs [k_begin, k_begin+k_count) are produced (a GPU's shard) but ranks
 * are global over all K pairs.
 *   fpos/fneg dev double [K][n_obj]; weights_out dev float [k_count]
 *   ranks_out dev int32 [n_obj][2][k_count] or NULL (debug/parity: rank of pos/neg)   */
int es_centered_rank(es_ctx* ctx, const double* fpos, const double* fneg, int K, int n_obj, float w0, float w1,
                     int k_begin, int k_count, float* weights_out, int32_t* ranks_out, void* stream);

/* ---- f4: the other fitness shapings of src/utils/rankers.py:61-103 ----------------------------
 * Same ranking as es_centered_rank, then per fitness (n = 2K, r = rank):
 *   ES_RANK_CENTERED         y = float32(r)/(n-1) - 0.5                         (rankers.py:53-58)
 *   ES_RANK_DOUBLE_POSITIVE  centered, then y *= 2 where y > 0                  (rankers.py:61-65)
 *   ES_RANK_SEMI_CENTERED    y = ((1/n)*square(float32(r) + 0.29*n))/n - 0.5    (rankers.py:78-83), float32
 *   ES_RANK_MAX_NORMALIZED   float64: y = x + (-mn if mn > 0 else mn); y /= max(y); y = 2*y - 1 (rankers.py:68-75);
 *                            fitnesses must be finite
 * n_obj == 2: MultiObjectiveRanker blend y0*w0 + y1*w1 in the kind's dtype (rankers.py:106-120).
 * elite_n == 0: weight[k] = y[k] - y[K+k] (Ranker._post_rank, rankers.py:42-44).
 * elite_n  > 0: EliteRanker(inner, pct) with elite_n = max(1, int(2K*pct)) (rankers.py:86-103): only the elite_n
 *   largest y are kept, nothing is subtracted and each elite keeps the noise index of its pair regardless of its
 *   sign (as the reference does): weight[k] = [y+ elite]*y+ + [y- elite]*y-;  n_fits_ranked = elite_n.  The compact
 *   lists the reference returns are written in ascending rank order (np.argpartition's order is unspecified):
 *   elite_vals_out double [elite_n] = ranked[elite], elite_fit_out int32 [elite_n] = index into concat(pos, neg),
 *   elite_idx_out int64 [elite_n] = noise_idx[fit % K]; only entries whose pair lies in the shard are written.
 *   Single objective only (ES_ERR_UNSUPPORTED otherwise).
 *   weights_out dev float [k_count]; weights64_out dev double [k_count] or NULL = the same weight before the cast to
 *   float32 (MAX_NORMALIZED is a float64 shaping); noise_idx dev int64 [K] or NULL; ranks_out as es_centered_rank. */
enum { ES_RANK_CENTERED = 0, ES_RANK_DOUBLE_POSITIVE = 1, ES_RANK_SEMI_CENTERED = 2, ES_RANK_MAX_NORMALIZED = 3 };
int es_rank_transform(es_ctx* ctx, const double* fpos, const double* fneg, int K, int n_obj, int kind, double w0,
                      double w1, int elite_n, int k_begin, int k_count, const int64_t* noise_idx, float* weights_out,
                      double* weights64_out, int32_t* ranks_out, double* elite_vals_out, int32_t* elite_fit_out,
                      int64_t* elite_idx_out, void* stream);

/* ---- a10: gradient reconstruction ---------------------------------------------------------
 * out[p] = sum_k weights[k] * table[idx[k] + p], p in [0,P): scale_noise/batch_noise,
 * src/utils/utils.py:14-39.  HBM-bound: reads n_idx*P*4 bytes of the table once.
 * Deterministic (fixed summation order for a given shape).                            */
int es_grad_reconstruct(es_ctx* ctx, const float* table, int64_t table_len, const int64_t* idx,
                        const float* weights, int n_idx, int P, float* out, void* stream);

/* ---- a11/a12: gradient scaling + optimizer step ----------------------------------------------
 * g = l2coeff*theta - gsum/n_ranked (src/core/es.py:100-101), then the optimizer step
 * and theta += step (src/core/policy.py:73-74), all float32 with every operation
 * rounded separately (numpy 1.18 casting of src/nn/optimizers.py:28-61).
 * Adam: neg_a = float32(-lr*sqrt(1-b2^t)/(1-b1^t)) computed by the caller in float64.   */
int es_adam_step(es_ctx* ctx, float* theta, float* m, float* v, const float* gsum, float n_ranked, float l2coeff,
                 float neg_a, float beta1, float one_minus_beta1, float beta2, float one_minus_beta2,
                 float epsilon, int P, void* stream);
int es_sgd_step(es_ctx* ctx, float* theta, float* v, const float* gsum, float n_ranked, float l2coeff,
                float neg_lr, float momentum, float one_minus_momentum, int P, void* stream);
int es_simple_step(es_ctx* ctx, float* theta, const float* gsum, float n_ranked, float l2coeff, float lr, int P,
                   void* stream);

/* ---- a14: observation statistics (open-loop stream) ---------------------------------------------
 * column sums of obs and obs^2 over rows, float32 sequential in row order
 * (TrainingResult.ob_sum_sq_cnt, src/gym/training_result.py:17-21).
 *   obs dev float [rows][obs_dim]; sum_out/sumsq_out dev float [obs_dim]               */
int es_obs_colsum(es_ctx* ctx, const float* obs, int rows, int obs_dim, float* sum_out, float* sumsq_out,
                  void* stream);

/* gen_obstat.inc(sum, sumsq, cnt) repeated for the n_rollouts rollouts that saved their
 * observations (ObStat.inc, src/nn/obstat.py:19-22, called per evaluation from
 * src/core/es.py:73-74): sum += (double)s, sumsq += (double)ssq, n_rollouts times in
 * order (float64 repeated addition is not n*s).  In the open-loop env every saved
 * rollout contributes the same (s, ssq).
 *   sum/sumsq dev double [obs_dim] in/out; s/ssq dev float [obs_dim]                    */
int es_obstat_accumulate(es_ctx* ctx, double* sum, double* sumsq, const float* s, const float* ssq, int obs_dim,
                         int n_rollouts, void* stream);
/* Same, with the number of saving rollouts decided on the device from the save_obs coins
 * drawn by es_draw_indices: rollout e saves iff double(coin_words[2e], coin_words[2e+1])
 * < chance (numpy legacy random_sample: (a>>5, b>>6) -> 53-bit double; the coin is
 * simple_example.py:38 / obj.py:54).  count_io[0] += rows_per_rollout per saving rollout
 * (ObStat.count, obstat.py:22); count_io[1] = number of saving rollouts (out).
 *   coin_words dev uint32 [n_coins][2]; count_io dev double [2]                          */
int es_obstat_accumulate_coins(es_ctx* ctx, double* sum, double* sumsq, double* count_io, const float* s,
                               const float* ssq, int obs_dim, int rows_per_rollout, const uint32_t* coin_words,
                               int n_coins, double chance, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ES_B200_H */
