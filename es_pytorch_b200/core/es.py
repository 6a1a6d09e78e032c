"""One ES generation (mirror of src/core/es.py): ``step``, ``test_params``,
``_share_results``, ``approx_grad`` with the reference signatures and return layouts.

Two evaluation paths behind ``test_params``:
  * ``fit_fn`` is a ``BatchedRollout``  -> the whole rank's pairs are drawn, perturbed,
    rolled out and scored by the fused device pipeline (``DeviceGeneration.evaluate``);
  * any other callable -> the reference's per-perturbation loop (es.py:67-74); each
    ``policy.pheno`` / ``run_model`` call still runs its arithmetic on the device.
``approx_grad`` always runs rank-weights -> reconstruction -> optimizer on the device, each
process summing only its own shard of pairs followed by one allreduce.
"""
from __future__ import annotations

from typing import Callable, List, Tuple

import numpy as np
import torch

from .. import devcache, dist
from ..engine import get_engine
from ..generation import DeviceGeneration
from ..gym.training_result import TrainingResult
from ..nn.obstat import ObStat
from ..utils.rankers import CenteredRanker, Ranker
from ..utils.reporters import Reporter, StdoutReporter
from .noisetable import NoiseTable
from .policy import Policy


def step(cfg, comm, policy: Policy, nt: NoiseTable, env, fit_fn: Callable, rs: np.random.RandomState = None,
         ranker: Ranker = None, reporter: Reporter = None) -> Tuple[TrainingResult, ObStat]:
    """Runs a single generation of ES (es.py:23-51); returns the noiseless result and the
    generation's observation statistics."""
    rs = np.random.RandomState() if rs is None else rs
    ranker = CenteredRanker() if ranker is None else ranker
    reporter = StdoutReporter(comm) if reporter is None else reporter
    assert cfg.general.policies_per_gen % comm.size == 0 and (cfg.general.policies_per_gen / comm.size) % 2 == 0
    eps_per_proc = int((cfg.general.policies_per_gen / comm.size) / 2)

    gen_obstat = ObStat(env.observation_space.shape, 0)
    if _can_fuse_step(comm, policy, fit_fn, ranker):
        return _step_fused(cfg, comm, eps_per_proc, policy, nt, gen_obstat, fit_fn, rs, ranker, reporter)
    pos_res, neg_res, inds, steps = test_params(comm, eps_per_proc, policy, nt, gen_obstat, fit_fn, rs)

    reporter.print(f'n dupes: {len(inds) - len(set(inds))}')

    ranker.rank(pos_res, neg_res, inds)
    approx_grad(policy, ranker, nt, policy.flat_params, cfg.general.batch_size, cfg.policy.l2coeff)
    noiseless_result = fit_fn(policy.pheno(np.zeros(len(policy))), False)
    reporter.log_gen(ranker.fits, noiseless_result, policy, steps)

    return noiseless_result, gen_obstat


TRACE = None      # dev: set to a dict to collect perf_counter marks of _step_fused's host phases (tools/dev_step_breakdown.py)


def _mark(name, _clock=__import__('time').perf_counter):
    if TRACE is not None:
        TRACE.setdefault(name, []).append(_clock())


def _silent(reporter) -> bool:
    """True for reporters that discard messages (the O(K) host-side message formatting can be skipped)."""
    from ..utils.reporters import ReporterSet
    return type(reporter) is Reporter or (type(reporter) is ReporterSet and not reporter.reporters)


def _queue_common_downloads(eng, gen, fpos, fneg):
    """Fitness, RNG streams and obs statistics towards pinned host memory with as few copies as possible: the two fitness
    halves are one buffer on a single GPU, the streams and the statistics are one buffer each."""
    if gen.comm.size == 1:
        h_fit = eng.download_async(gen.fit_local, 'fit')             # [pos | neg][K][n_obj]
        h_pos, h_neg = h_fit[0], h_fit[1]
    else:
        h_pos, h_neg = eng.download_async(fpos, 'fpos'), eng.download_async(fneg, 'fneg')
    h_state = eng.download_async(gen.mt_state, 'mtstate')
    R = gen.n_streams
    nk = R * gen.mt_key.shape[1]
    h_key, h_mtpos = h_state[:nk].view(R, -1), h_state[nk:nk + R]
    gen._h_gauss = (h_state[nk + R:nk + 2 * R], h_state[nk + 2 * R:].view(torch.float64))    # valid after the synchronisation
    h_stats = eng.download_async(gen._gen_stats, 'gstats') if gen.extra_words else None
    return h_pos, h_neg, h_key, h_mtpos, h_stats


def _host_gauss(gen):
    """(has_gauss, cached gaussian) host copies of the last _queue_common_downloads, when the generation drew action noise."""
    if gen.ac_std == 0.0:
        return None
    return gen._h_gauss[0].numpy().copy(), gen._h_gauss[1].numpy().copy()


def _obstat_from(h_stats, obs_dim):
    a = h_stats.numpy()
    return a[:obs_dim].copy(), a[obs_dim:2 * obs_dim].copy(), float(a[2 * obs_dim])


def _can_fuse_step(comm, policy: Policy, fit_fn, ranker: Ranker) -> bool:
    """``step`` can keep the whole generation on the device (one synchronisation) when the evaluation is a
    ``BatchedRollout`` of a tanh MLP and the ranker is a float32 shaping without elite selection (the others return host
    arrays of a different dtype / length: they take the call-by-call route)."""
    from .._lib import ES_RANK_MAX_NORMALIZED
    if not getattr(fit_fn, 'is_batched_rollout', False) or not policy._module.is_tanh_mlp():
        return False
    if comm.size != dist.world().size:                       # a communicator this package does not drive
        return False
    try:
        kind, _, _, elite_n = ranker._spec(fit_fn.n_obj, 2)
    except Exception:
        return False
    return elite_n == 0 and kind != ES_RANK_MAX_NORMALIZED and type(ranker).rank is Ranker.rank


def _step_fused(cfg, comm, n: int, policy: Policy, nt: NoiseTable, gen_obstat: ObStat, fit_fn, rs, ranker: Ranker,
                reporter: Reporter):
    """es.py:38-51 with every stage queued on the device back to back -- draw, rollouts, rank, reconstruction, optimizer
    step, noiseless evaluation of the new theta -- and ONE synchronisation before the host-side bookkeeping.  Same
    results and side effects as the call-by-call route (test_params -> Ranker.rank -> approx_grad -> fit_fn)."""
    streams = fit_fn.rank_streams if fit_fn.rank_streams is not None else [rs]
    _mark('t0')
    gen = _device_generation(fit_fn, policy, nt, streams)
    _mark('t1_prepared')
    eng = gen.eng
    gen.l2coeff, gen.ranker = float(cfg.policy.l2coeff), ranker
    fpos, fneg = gen.evaluate(n)
    _mark('t2_evaluate_queued')
    gen.update(fpos, fneg, all_weights=True)
    gen.l2coeff, gen.ranker = 0.0, None                    # approx_grad passes its own l2coeff on the other route
    fit0, behv0 = gen.noiseless_eval()
    gen.skip_eval_coins(1)                                 # the fit_fn's rs.random() of the noiseless call (es.py:48)
    h_pos, h_neg, h_key, h_mtpos, h_stats = _queue_common_downloads(eng, gen, fpos, fneg)
    w_all, idx_all = gen.weights, gen.idx
    if gen.comm.size > 1:
        # what Ranker.rank / _share_results hand to every rank: all K weights and noise indices.  Both are already here: the
        # indices travelled with the fitness rows (one allgather, as in es.py:89-95) and every process finalised all K weights
        w_all, idx_all = gen.weights_all, gen.idx_all
    h_idx = eng.download_async(idx_all, 'idx')
    h_w = eng.download_async(w_all, ('ranked', id(ranker)))
    h_theta = eng.download_async(gen.theta, ('theta', id(policy)))
    h_fit0, h_behv0 = eng.download_async(fit0, 'nlfit'), eng.download_async(behv0, 'nlbehv')
    _mark('t3_all_queued')
    eng.sync()
    _mark('t4_synced')
    version = gen.version
    valid = lambda g=gen, v=version: g.version == v
    pos = devcache.attach(h_pos.numpy().reshape(gen.K, gen.n_obj).copy(), fpos, valid)
    neg = devcache.attach(h_neg.numpy().reshape(gen.K, gen.n_obj).copy(), fneg, valid)
    inds = devcache.attach(h_idx.numpy().astype(np.float64), idx_all, valid)
    gen.store_states(streams, h_key.numpy().copy(), h_mtpos.numpy().copy(), _host_gauss(gen))
    if h_stats is not None:
        gen_obstat.inc(*_obstat_from(h_stats, gen.obs_dim))
    steps = 2 * gen.K * (fit_fn.max_steps - 1)
    if not _silent(reporter):
        reporter.print(f'n dupes: {len(inds) - len(set(inds))}')
    # what Ranker.rank leaves behind (rankers.py:37-50)
    ranker._pre_rank(pos, neg, inds)
    w = w_all
    ranker.ranked_fits_dev = w
    res = h_w.numpy().copy()
    if not ranker._squeezes() and pos.ndim == 2:
        res = res.reshape(-1, 1)
    ranker.ranked_fits = devcache.attach(res, w, lambda r=ranker, t=w: r.ranked_fits_dev is t)
    # what approx_grad and policy.pheno(zeros) leave behind: flat_params and the module carry the new theta
    policy.flat_params[...] = h_theta.numpy()
    policy.set_nn_params(torch.from_numpy(policy.flat_params.copy()))
    noiseless_result = fit_fn.result_from_device(float(h_fit0.numpy()[0]), h_behv0.numpy()[0].astype(np.float64))
    reporter.log_gen(ranker.fits, noiseless_result, policy, steps)
    _mark('t5_done')
    return noiseless_result, gen_obstat


def _device_generation(fit_fn, policy: Policy, nt: NoiseTable, streams) -> DeviceGeneration:
    eng = get_engine()
    gen = fit_fn._gen
    theta = policy.theta_dev(eng)
    if (gen is None or gen.theta is not theta or gen.n_streams != len(streams) or gen.table is not nt.device_table(eng)
            or gen.coins_per_eval != int(fit_fn.coins_per_eval) or gen.rollout_mode != fit_fn.rollout_mode
            or (gen.archive is None) != (fit_fn.archive is None)
            or gen.eps_per_policy != getattr(fit_fn, 'eps_per_policy', 1)):
        env = fit_fn.env
        obs_dev, rew_dev = env.device_arrays(eng)
        T = fit_fn.max_steps
        archive = None if fit_fn.archive is None else eng.to_device(fit_fn.archive, torch.float64)
        gen = DeviceGeneration(nt.device_table(eng), theta, policy._module.layer_sizes(), obs_dev[:T + 1].contiguous(),
                               rew_dev[:T].contiguous(), streams, policy.std, 0.0, policy.optim,
                               ob_clip=policy._module.ob_clip, pos_scale=env.pos_scale,
                               coins_per_eval=fit_fn.coins_per_eval, save_obs_chance=fit_fn.save_obs_chance,
                               archive=archive, nov_k=fit_fn.nov_k, rollout_mode=fit_fn.rollout_mode, engine=eng,
                               ac_std=float(getattr(policy._module, '_action_std', 0.0) or 0.0),
                               closed=env.device_closed(eng) if getattr(env, 'is_synthetic_closedloop', False) else None,
                               eps_per_policy=getattr(fit_fn, 'eps_per_policy', 1))
        fit_fn._gen = gen
    else:
        gen.load_states(streams)
        if getattr(fit_fn, 'stream_env_from_host', False):
            # the env's observation / reward streams are this generation's inputs: copy them from the host again
            env = fit_fn.env
            pinned = bool(getattr(env, 'host_pinned', False))
            eng.upload_async(gen.obs_stream, env.obs_stream[:gen.T + 1], ('obs', id(gen)), src_pinned=pinned)
            eng.upload_async(gen.rew_vec, env.rew_vec[:gen.T], ('rew', id(gen)), src_pinned=pinned)
    fit_fn._streams_in_use = streams                    # BatchedRollout.__call__ draws the noiseless call's coin from them
    gen.sigma = float(policy.std)                       # scripts decay the noise std between generations
    ac_std = float(getattr(policy._module, '_action_std', 0.0) or 0.0)       # obj.py:81 decays it between generations
    if ac_std != gen.ac_std:
        gen.ac_std = ac_std
        gen._host_states = None                         # the gaussian cache starts / stops travelling: upload afresh
        gen.load_states(streams)
    gen.save_obs_chance = fit_fn.save_obs_chance
    # scripts swap or mutate these between generations (obj.py:81-83 decays lr / ac_std, nsra.py grows the archive): the
    # cached generation follows the callers' objects instead of keeping its own references
    gen.optim = policy.optim
    gen.ob_clip, gen.pos_scale, gen.nov_k = float(policy._module.ob_clip), float(fit_fn.env.pos_scale), int(fit_fn.nov_k)
    if fit_fn.archive is not None and getattr(gen, '_archive_src', None) is not fit_fn.archive:
        gen.archive = eng.to_device(fit_fn.archive, torch.float64)      # new array object (or first use): upload again
        gen._archive_src = fit_fn.archive
    gen.set_obstat(policy._module._obmean, policy._module._obstd)
    return gen


def _test_params_batched(comm, n: int, policy: Policy, nt: NoiseTable, gen_obstat: ObStat, fit_fn, rs):
    if not policy._module.is_tanh_mlp():
        raise NotImplementedError('the fused rollout evaluates tanh MLPs (FeedForward with torch.nn.Tanh)')
    streams = fit_fn.rank_streams if fit_fn.rank_streams is not None else [rs]
    gen = _device_generation(fit_fn, policy, nt, streams)
    fpos, fneg = gen.evaluate(n)
    # one device->host hop for everything the reference API returns as ndarrays
    eng = gen.eng
    # everything the reference API returns as ndarrays comes back through pinned staging with ONE synchronisation
    h_pos, h_neg, h_key, h_mtpos, h_stats = _queue_common_downloads(eng, gen, fpos, fneg)
    # the noise indices of ALL ranks: they travelled with the fitness rows (one allgather, like es.py:89-95's rows)
    idx_dev = gen.idx_all if gen.comm.size > 1 else gen.idx
    h_idx = eng.download_async(idx_dev, 'idx')
    eng.sync()
    version = gen.version
    valid = lambda g=gen, v=version: g.version == v
    pos = devcache.attach(h_pos.numpy().reshape(gen.K, gen.n_obj).copy(), fpos, valid)
    neg = devcache.attach(h_neg.numpy().reshape(gen.K, gen.n_obj).copy(), fneg, valid)
    gen.store_states(streams, h_key.numpy().copy(), h_mtpos.numpy().copy(), _host_gauss(gen))
    inds = h_idx.numpy().astype(np.float64)
    if gen.comm.size == 1:
        inds = devcache.attach(inds, gen.idx, valid)
    if h_stats is not None:
        gen_obstat.inc(*_obstat_from(h_stats, gen.obs_dim))
    steps = 2 * gen.K * (fit_fn.max_steps - 1)          # run_model returns the last loop index (gym_runner.py:50,67)
    return pos, neg, inds, steps


def test_params(comm, n: int, policy: Policy, nt: NoiseTable, gen_obstat: ObStat, fit_fn: Callable,
                rs: np.random.RandomState) -> Tuple[np.ndarray, np.ndarray, np.ndarray, int]:
    """Tests ``n`` antithetic perturbation pairs per rank and returns the positive / negative
    results of ALL ranks plus the noise indices (es.py:54-81):
    (pos[K, n_obj], neg[K, n_obj], inds[K], steps), rank-major, float64."""
    if getattr(fit_fn, 'is_batched_rollout', False):
        return _test_params_batched(comm, n, policy, nt, gen_obstat, fit_fn, rs)

    results_pos, results_neg, inds = [], [], []
    for _ in range(n):
        idx, noise = nt.sample(rs)
        inds.append(idx)
        results_pos.append(fit_fn(policy.pheno(noise)))
        results_neg.append(fit_fn(policy.pheno(-noise)))
        gen_obstat.inc(*results_pos[-1].ob_sum_sq_cnt)
        gen_obstat.inc(*results_neg[-1].ob_sum_sq_cnt)

    n_objectives = len(results_pos[0].result)
    results = _share_results(comm, [tr.result for tr in results_pos], [tr.result for tr in results_neg], inds)
    gen_obstat.mpi_inc(comm)
    steps = sum([tr.steps for tr in results_pos + results_neg])
    if comm.size > 1:
        steps = int(sum(dist.world().allgather_object(steps)))
    return results[:, 0:n_objectives], results[:, n_objectives:2 * n_objectives], results[:, -1], steps


def _share_results(comm, fits_pos: List[List[float]], fits_neg: List[List[float]], inds: List[int]) -> np.ndarray:
    """Share results and noise inds with all processes: rows ``f+... f-... idx`` (float64),
    ranks concatenated in order (es.py:84-95; the reference's Alltoall of tiled rows is an
    allgather)."""
    rows = np.array([list(fp) + list(fn) + [i] for fp, fn, i in zip(fits_pos, fits_neg, inds)], dtype=np.float64)
    objectives = len(fits_pos[0])
    rows = rows.reshape(-1, 1 + 2 * objectives)
    if comm.size == 1:
        return rows
    t = torch.from_numpy(rows)
    backend = torch.distributed.get_backend()
    if backend == 'nccl':
        t = t.cuda()
    out = torch.empty((comm.size,) + tuple(t.shape), dtype=t.dtype, device=t.device)
    dist.world().allgather_into(out, t)
    return out.cpu().numpy().reshape(-1, 1 + 2 * objectives)


def approx_grad(policy: Policy, ranker: Ranker, nt: NoiseTable, params: np.ndarray, batch_size: int, l2coeff: float):
    """Approximates the gradient and updates the policy (es.py:98-101):
    grad = scale_noise(ranked_fits, noise_inds) / n_fits_ranked;  theta += optim.step(l2coeff*theta - grad).
    Each process reconstructs the partial sum of its own shard of pairs; one allreduce."""
    if params is not policy.flat_params:
        raise NotImplementedError('approx_grad updates policy.flat_params in place; pass it as `params`')
    eng = get_engine()
    comm = dist.world()
    K = len(ranker.noise_inds)
    k0, k1 = dist.shard_bounds(K, comm.size, comm.rank) if K % comm.size == 0 else (0, K if comm.rank == 0 else 0)
    w_all = devcache.lookup(ranker.ranked_fits)
    if w_all is not None and w_all.numel() == K:
        w = w_all[k0:k1]
    else:
        w = eng.to_device(np.ascontiguousarray(ranker.ranked_fits[k0:k1], dtype=np.float32))
    idx_sh = devcache.lookup(ranker.noise_inds)
    if idx_sh is not None and comm.size == 1 and idx_sh.numel() == K:
        idx = idx_sh
    else:
        idx = eng.to_device(np.ascontiguousarray(ranker.noise_inds[k0:k1]).astype(np.int64))
    theta = policy.theta_dev(eng)
    gsum = eng.grad_reconstruct(nt.device_table(eng), idx, w, len(policy))
    comm.allreduce_sum(gsum)
    policy.optim.apply_fused(eng, theta, gsum, float(ranker.n_fits_ranked), float(l2coeff))
    policy.sync_host()
