"""obj.py's fit_fn with several episodes per evaluation (``cfg.general.eps_per_policy``, obj.py:53-61), restated on top of the
primitives of ``oracle/es_oracle.py``: the save_obs coin, then ``max(1, eps_per_policy)`` calls of run_model with the same
stream, the per-step rewards added into a float64 array of length ``max_steps`` with ``+=``, divided by the episode count with
``/=`` and summed with ``sum``; behaviour, observations and the step index are the last episode's.

``es_test_params`` / ``generation`` / ``es_step`` mirror the functions of the same names in the oracle (es.py:38-81 for R
virtual ranks, centered ranking, the noiseless evaluation of es.py:48) with that fit_fn.  Used by tests/test_episodes_host.py
and tests/test_gpu_episodes.py."""
from typing import List, Optional, Sequence

import numpy as np

from oracle import es_oracle as orc


def run_episodes(env, layers, obmean, obstd, ob_clip: float, max_steps: int, eps_per_policy: int, batched: bool = False,
                 ac_std: float = 0.0, rs: Optional[np.random.RandomState] = None):
    """obj.py:55-60: (rews list of length max_steps, last episode's behv, last episode's obs, last episode's step)."""
    rews = np.zeros(max_steps)
    for _ in range(max(1, eps_per_policy)):
        rew, behv, obs, steps = orc.run_model(env, layers, obmean, obstd, ob_clip, max_steps, batched, ac_std, rs)
        rews[:len(rew)] += np.array(rew)
    rews /= max(1, eps_per_policy)
    return rews.tolist(), behv, obs, steps


def es_test_params(table: np.ndarray, flat: np.ndarray, std: float, dims, env, rank_seeds: Sequence[int], n_per_rank: int,
                   obmean, obstd, ob_clip: float, max_steps: int, eps_per_policy: int, coins_per_eval: int = 0,
                   save_obs_chance: float = 0.0, batched: bool = True,
                   rank_states: Optional[List[np.random.RandomState]] = None, ac_std: float = 0.0):
    """es.py:54-81 with obj.py's fit_fn, one objective.  Returns (pos[K,1], neg[K,1], inds[K], steps, obstat), rank-major."""
    P = len(flat)
    gen_obstat = orc.ObStatOracle((env.obs_dim,), 0)
    rows_per_rank, steps_total = [], 0
    for r, seed in enumerate(rank_seeds):
        rs = rank_states[r] if rank_states is not None else np.random.RandomState(seed)
        rows = []
        for _ in range(n_per_rank):
            idx = orc.sample_idx(len(table), rs, P)
            noise = orc.table_get(table, idx, P)
            res = []
            for sign in (1.0, -1.0):
                save_obs = False
                for _c in range(coins_per_eval):
                    save_obs = rs.random() < save_obs_chance
                layers = orc.unflatten(orc.pheno_params(flat, std, noise if sign > 0 else -noise), dims)
                rews, behv, obs, step = run_episodes(env, layers, obmean, obstd, ob_clip, max_steps, eps_per_policy, batched,
                                                     ac_std, rs)
                res.append(orc.reward_result(rews))
                steps_total += step
                o = obs if save_obs else np.array([np.zeros((env.obs_dim,))])
                gen_obstat.inc(*orc.ob_sum_sq_cnt(o))
            rows.append(res[0] + res[1] + [idx])
        rows_per_rank.append(np.array(rows, dtype=np.float64).reshape(n_per_rank, 3))
    results = orc.share_results(rows_per_rank)
    return results[:, 0:1], results[:, 1:2], results[:, -1], steps_total, gen_obstat


def generation(table, flat, optim, std, dims, env, rank_seeds, n_per_rank, obmean, obstd, ob_clip, max_steps, batch_size,
               l2coeff, eps_per_policy, coins_per_eval=0, rank_states=None, batched=True, save_obs_chance=0.0, ac_std=0.0):
    """One generation (es.py:38-47) with obj.py's fit_fn and the centered ranker; mutates ``flat``."""
    pos, neg, inds, steps, obstat = es_test_params(table, flat, std, dims, env, rank_seeds, n_per_rank, obmean, obstd, ob_clip,
                                                   max_steps, eps_per_policy, coins_per_eval=coins_per_eval,
                                                   save_obs_chance=save_obs_chance, batched=batched, rank_states=rank_states,
                                                   ac_std=ac_std)
    w, n_ranked = orc.centered_ranker(pos, neg)
    orc.approx_grad(flat, optim, w, inds, n_ranked, table, batch_size, l2coeff)
    return dict(pos=pos, neg=neg, inds=inds, steps=steps, weights=w, n_ranked=n_ranked, obstat=obstat)


def es_step(table, flat, optim, std, dims, env, rank_states, n_per_rank, obmean, obstd, ob_clip, max_steps, batch_size, l2coeff,
            eps_per_policy, coins_per_eval=1, save_obs_chance=0.0, batched=True, ac_std=0.0):
    """es.step (es.py:38-51): the generation, then every rank's noiseless evaluation ``fit_fn(policy.pheno(zeros), False)`` of the
    updated parameters -- its coin(s), then E episodes without action noise (use_ac_noise=False: nothing drawn).  Returns the
    generation's dict plus ``noiseless`` (the result list of rank 0)."""
    out = generation(table, flat, optim, std, dims, env, [None] * len(rank_states), n_per_rank, obmean, obstd, ob_clip, max_steps,
                     batch_size, l2coeff, eps_per_policy, coins_per_eval=coins_per_eval, rank_states=rank_states, batched=batched,
                     save_obs_chance=save_obs_chance, ac_std=ac_std)
    noiseless = None
    for rs in rank_states:
        for _c in range(coins_per_eval):
            rs.random()
        layers = orc.unflatten(orc.pheno_params(flat, std, None), dims)
        rews, _, _, _ = run_episodes(env, layers, obmean, obstd, ob_clip, max_steps, eps_per_policy, batched)
        noiseless = orc.reward_result(rews) if noiseless is None else noiseless
    out['noiseless'] = noiseless
    return out
