"""One OpenAI-ES generation, resident on the GPU.

``DeviceGeneration`` owns the HBM-resident state of the hot path (noise table, theta,
optimizer moments, observation stream, per-rank MT19937 streams) and enqueues, on the
current CUDA stream and without any host synchronisation, the kernel sequence that
replaces ``es.test_params`` -> ``Ranker.rank`` -> ``es.approx_grad`` of the reference
(src/core/es.py:54-101):

    draw K indices            es_draw_indices        (noisetable.py:37-40, es.py:67-68)
    normalise obs stream      es_normalise_obs       (nn.py:45)
    theta +- sigma*eps, MLP rollout, fitness
                              es_rollout_openloop    (policy.py:61-64, nn.py:42-50, gym_runner.py:33-67)
    [novelty column]          es_novelty             (novelty.py:16-18)            NSRA only
    [obs statistics]          es_obs_colsum + es_obstat_accumulate_coins           (es.py:73-74)
    allgather fitness         NCCL (only when world size > 1)                       (es.py:84-95)
    rank shaping -> weights   es_centered_rank / es_rank_transform  (rankers.py:9-120)
    sum_k w_k eps_k           es_grad_reconstruct    (utils.py:14-39)
    allreduce partial grad    NCCL (only when world size > 1)
    /2K, l2, Adam/SGD, theta  es_adam_step ...       (es.py:100-101, optimizers.py)

Sharding (SURVEY.md section 8e): each process (GPU) owns ``n_streams`` virtual MPI ranks
and evaluates their pairs; ranks are global (fitness allgather), the gradient partial is
shard-local and summed by ONE allreduce; the optimizer step is replicated.
"""
from __future__ import annotations


from typing import List, Optional, Sequence

import numpy as np
import torch

from . import dist
from ._lib import ES_MT_N, ES_ROLLOUT_F32
from .engine import Engine, get_engine
from .nn.optimizers import Optimizer


class _NoTimer:
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


_NO_TIMER = _NoTimer()


class _Timed:
    """Brackets a kernel group with CUDA events on the launching stream."""

    def __init__(self, gen, name):
        self.gen, self.name = gen, name

    def __enter__(self):
        self.a = torch.cuda.Event(enable_timing=True)
        self.b = torch.cuda.Event(enable_timing=True)
        self.a.record()
        return self

    def __exit__(self, *exc):
        self.b.record()
        self.gen.timers.setdefault(self.name, []).append((self.a, self.b))
        return False


class DeviceGeneration:
    def __init__(self, table: torch.Tensor, theta: torch.Tensor, layer_sizes: Sequence[int], obs_stream: torch.Tensor,
                 rew_vec: torch.Tensor, rank_states: Sequence[np.random.RandomState], sigma: float, l2coeff: float,
                 optim: Optimizer, ob_clip: float = 5.0, pos_scale: float = 0.05, coins_per_eval: int = 0,
                 save_obs_chance: float = 0.0, archive: Optional[torch.Tensor] = None, nov_k: int = 10,
                 moo_w: float = 1.0, rollout_mode: int = ES_ROLLOUT_F32, comm: Optional[dist.Comm] = None,
                 engine: Optional[Engine] = None, ranker=None, ac_std: float = 0.0, closed=None, eps_per_policy: int = 1):
        self.eng = engine or get_engine()
        # closed-loop variant of the synthetic env (gym.synthetic_env.ClosedLoopEnv): (obs_0 [obs], A^T [band, obs], B^T [act, obs]);
        # row 0 of obs_stream is then the only one read and the rollout is es_rollout_closedloop
        self.closed = closed
        self.ranker = ranker                            # a utils.rankers.Ranker; None = Centered / MultiObjective(moo_w)
        e = self.eng
        self.comm = comm or dist.world()
        self.table = table
        self.theta = theta
        self.P = theta.numel()
        self.layer_sizes = [int(x) for x in layer_sizes]
        self.obs_dim, self.act_dim = self.layer_sizes[0], self.layer_sizes[-1]
        self.obs_stream = obs_stream                    # [T+1, obs_dim]
        self.rew_vec = rew_vec                          # [T, act_dim]
        self.T = rew_vec.shape[0]
        assert obs_stream.shape == (self.T + 1, self.obs_dim)
        self.sigma, self.l2coeff, self.optim = float(sigma), float(l2coeff), optim
        self.ob_clip, self.pos_scale = float(ob_clip), float(pos_scale)
        self.coins_per_eval, self.save_obs_chance = int(coins_per_eval), float(save_obs_chance)
        self.archive, self.nov_k, self.moo_w = archive, int(nov_k), float(moo_w)
        self.n_obj = 1 if archive is None else 2
        self.rollout_mode = rollout_mode
        # FeedForward._action_std (nn.py:47-48): != 0 -> every step adds rs.randn(act) * ac_std, drawn from the rank streams
        self.ac_std = float(ac_std or 0.0)
        self.act_noise = None
        # episodes per evaluation (obj.py's eps_per_policy): each draws its own T * act gaussians after the coin; on the open-loop
        # env they share the forward pass (es_rollout_openloop_episodes).  Without action noise they are all the same episode.
        self.eps_per_policy = max(1, int(eps_per_policy))
        assert self.coins_per_eval in (0, 1), 'fit_fns draw at most one save_obs coin per evaluation'

        # per-rank MT19937 streams, resident on the device between generations
        self.n_streams = len(rank_states)
        self._gauss = [(s.get_state()[3], s.get_state()[4]) for s in rank_states]
        key = np.stack([s.get_state()[1].astype(np.uint32) for s in rank_states]).view(np.int32)
        pos = np.array([s.get_state()[2] for s in rank_states], dtype=np.int32)
        # the whole stream state in one buffer (one download brings everything back):
        # [R*624 key words | R positions | R has_gauss | R cached gaussians (float64 = 2 words each)]
        R = self.n_streams
        has = np.array([g[0] for g in self._gauss], dtype=np.int32)
        gv = np.array([g[1] for g in self._gauss], dtype=np.float64).view(np.int32)
        self.mt_state = e.to_device(np.concatenate((key.reshape(-1), pos, has, gv)))
        self.mt_key = self.mt_state[:R * ES_MT_N].view(R, ES_MT_N)
        self.mt_pos = self.mt_state[R * ES_MT_N:R * ES_MT_N + R]
        self.mt_has = self.mt_state[R * ES_MT_N + R:R * ES_MT_N + 2 * R]
        self.mt_gauss = self.mt_state[R * ES_MT_N + 2 * R:].view(torch.float64)       # byte offset 2504 R: 8-byte aligned

        f32, f64 = torch.float32, torch.float64
        self.gsum = e.empty((self.P,), f32)
        self.ob_mean = torch.zeros(self.obs_dim, dtype=f64, device=e.device)
        self.ob_std = torch.ones(self.obs_dim, dtype=f64, device=e.device)
        self.obsn = e.empty((self.T, self.obs_dim), f32)
        # generation obs statistics (ObStat(shape, 0), es.py:41): sum, sumsq, [count, n_saved] -- a view into the
        # buffer this process shares with the others (see _ensure_buffers)
        self._gen_stats = self.gen_sum = self.gen_sumsq = self.gen_count = None
        self._bufs_for = None
        self._host_states = None    # (key, pos) host copies of what store_states last wrote into the callers' streams
        self.version = 0            # bumped by every evaluate(): validity token of the device shadows handed out
        self.timers = None          # optional {'name': [(start_event, end_event), ...]} filled by _timed()

    # ------------------------------------------------------------------------------------------
    def enable_timers(self, on: bool = True):
        """Bracket each kernel group with CUDA events on the launching stream (bench.py's roofline)."""
        self.timers = {} if on else None

    def _timed(self, name: str):
        return _Timed(self, name) if self.timers is not None else _NO_TIMER

    def _ensure_buffers(self, n_per_stream: int):
        if self._bufs_for == n_per_stream:
            return
        e, i64, f32, f64 = self.eng, torch.int64, torch.float32, torch.float64
        self.k_local = self.n_streams * n_per_stream
        self.K = self.k_local * self.comm.size
        self.k_begin = self.k_local * self.comm.rank
        self.idx = e.empty((self.k_local,), i64)
        self.extra_words = 4 * self.coins_per_eval       # 2 evaluations x coins x 2 words per double
        self.extras = e.empty((self.k_local, self.extra_words), torch.int32) if self.extra_words else None
        # What a process shares per generation is ONE float64 buffer -- the reference's _share_results rows (fitness of both
        # signs and the noise index as float64, es.py:89-91) plus the generation's obs statistics (ObStat.mpi_inc, es.py:77)
        # -- so that one allgather serves the ranks, the indices and the statistics:
        #   [fitness [pos|neg][k][obj] | idx [k] | obs sum, sumsq, count, n_saved]
        nf, ns = 2 * self.k_local * self.n_obj, 2 * self.obs_dim + 2
        self.share_local = torch.zeros(nf + self.k_local + ns, dtype=f64, device=e.device)
        self.fit_local = self.share_local[:nf].view(2, self.k_local, self.n_obj)
        self.idx_f64 = self.share_local[nf:nf + self.k_local]
        self._gen_stats = self.share_local[nf + self.k_local:]
        self.gen_sum = self._gen_stats[:self.obs_dim]
        self.gen_sumsq = self._gen_stats[self.obs_dim:2 * self.obs_dim]
        self.gen_count = self._gen_stats[2 * self.obs_dim:]
        G = self.comm.size
        self.share_all = e.empty((G, nf + self.k_local + ns), f64) if G > 1 else None
        self.fit_all = self.share_all[:, :nf].view(G, 2, self.k_local, self.n_obj) if G > 1 else None
        self.fpos_all = e.empty((self.K, self.n_obj), f64) if G > 1 else None
        self.fneg_all = e.empty((self.K, self.n_obj), f64) if G > 1 else None
        self.idx_all = e.empty((self.K,), i64) if G > 1 else None             # every process's indices, rank-major
        self.behv = e.empty((2, self.k_local, 3), f32) if self.n_obj == 2 else None
        self.weights = None
        self._bufs_for = n_per_stream

    def set_obstat(self, mean: np.ndarray, std: np.ndarray):
        """Policy.update_obstat -> BaseNet.set_ob_mean_std (policy.py:69-71, nn.py:19-21).  Uploaded when they changed."""
        mean = np.ascontiguousarray(mean, dtype=np.float64).reshape(-1)
        std = np.ascontiguousarray(std, dtype=np.float64).reshape(-1)
        last = getattr(self, '_obstat_host', None)
        if last is not None and np.array_equal(last[0], mean) and np.array_equal(last[1], std):
            return
        self._obstat_host = (mean.copy(), std.copy())
        self.eng.upload_async(self.ob_mean, mean, ('obmean', id(self)))
        self.eng.upload_async(self.ob_std, std, ('obstd', id(self)))

    # ------------------------------------------------------------------------------------------
    def evaluate(self, n_per_stream: int):
        """es.test_params on the device: draw, perturb+rollout, fitness (+novelty, obstat),
        allgather.  Leaves fpos/fneg [K, n_obj] (global) and idx [k_local] on the device."""
        e = self.eng
        self._ensure_buffers(n_per_stream)
        self.version += 1
        with self._timed('draw_indices'):
            if self.ac_std != 0.0:
                # indices, coins and the action noise of every rollout, in the reference's stream order (mt_gauss.cu); the
                # E episodes of an evaluation are E * T * act consecutive gaussians after its coin
                nrm = self.eps_per_policy * self.T * self.act_dim
                if self.act_noise is None or self.act_noise.shape != (self.k_local, 2, nrm):
                    self.act_noise = e.empty((self.k_local, 2, nrm), torch.float32)
                e.draw_noisy(self.mt_key, self.mt_pos, self.mt_has, self.mt_gauss, n_per_stream, self.table.numel() - self.P,
                             self.coins_per_eval, nrm, self.ac_std, self.idx, self.extras, self.act_noise)
            else:
                e.draw_indices(self.mt_key, self.mt_pos, n_per_stream, self.table.numel() - self.P, self.extra_words,
                               self.idx, self.extras)
        fp, fn = self.fit_local[0], self.fit_local[1]
        if self.closed is not None:
            if self.ac_std != 0.0:
                raise NotImplementedError('the closed-loop variant of the synthetic env is defined without action noise: set the '
                                          'network\'s ac_std to 0 (the open-loop env supports ac_std != 0 on the device)')
            self._gen_stats.zero_()
            obs0, env_a, env_b = self.closed
            with self._timed('rollout'):
                e.rollout_closed(self.table, self.idx, self.theta, self.sigma, self.layer_sizes, self.ob_mean, self.ob_std,
                                 self.ob_clip, obs0, env_a, env_b, self.rew_vec, self.pos_scale, fp, fn, self.n_obj,
                                 None if self.behv is None else self.behv[0], None if self.behv is None else self.behv[1],
                                 coin_words=self.extras if self.extra_words else None, save_obs_chance=self.save_obs_chance,
                                 ob_sum=self.gen_sum if self.extra_words else None,
                                 ob_sumsq=self.gen_sumsq if self.extra_words else None,
                                 ob_count=self.gen_count if self.extra_words else None)
            if self.n_obj == 2:
                e.novelty(self.behv.view(-1, 3), self.archive, self.nov_k, self.fit_local.view(-1)[1:], 2)
        else:
            self._evaluate_openloop(fp, fn)
        if self.comm.size > 1:
            nf = 2 * self.k_local * self.n_obj
            self.idx_f64.copy_(self.idx)                         # exact: indices < 2^53 (the reference shares them as float64 too)
            with self._timed('allgather'):
                self.comm.allgather_into(self.share_all, self.share_local)
            # [rank][pos|neg][k][obj] -> rank-major [K][obj] per sign (es.py:93-95 ordering)
            self.fpos_all.view(self.comm.size, self.k_local, self.n_obj).copy_(self.fit_all[:, 0])
            self.fneg_all.view(self.comm.size, self.k_local, self.n_obj).copy_(self.fit_all[:, 1])
            self.idx_all.view(self.comm.size, self.k_local).copy_(self.share_all[:, nf:nf + self.k_local])
            # obs statistics of all processes (rank order: the same float64 sum everywhere), in place of the local ones
            self._gen_stats.copy_(self.share_all[:, nf + self.k_local:].sum(dim=0))
            return self.fpos_all, self.fneg_all
        return fp, fn

    def _evaluate_openloop(self, fp, fn):
        e = self.eng
        e.normalise_obs(self.obs_stream[:self.T], self.ob_mean, self.ob_std, self.ob_clip, self.obsn)
        with self._timed('rollout'):
            e.rollout(self.table, self.idx, self.theta, self.sigma, self.layer_sizes, self.obsn, self.rew_vec,
                      self.pos_scale, fp, fn, self.n_obj, None if self.behv is None else self.behv[0],
                      None if self.behv is None else self.behv[1], self.rollout_mode,
                      act_noise=self.act_noise if self.ac_std != 0.0 else None,
                      n_episodes=self.eps_per_policy if self.ac_std != 0.0 else 1)
        if self.n_obj == 2:
            # second objective column = novelty of the final (x, y) (training_result.py:95-97)
            e.novelty(self.behv.view(-1, 3), self.archive, self.nov_k, self.fit_local.view(-1)[1:], 2)
        self._gen_stats.zero_()
        if self.extra_words:
            # column sums of the post-step observations of a rollout: the open-loop stream is the same for every rollout and
            # every generation, so they are computed once per content of the stream (torch's version counter sees every write)
            ver = self.obs_stream._version
            if getattr(self, '_colsum_for', None) != ver:
                self._colsum = e.obs_colsum(self.obs_stream[1:self.T + 1])
                self._colsum_for = ver
            s, q = self._colsum
            e.obstat_accumulate_coins(self.gen_sum, self.gen_sumsq, self.gen_count, s, q, self.T,
                                      self.extras.view(-1, 2), self.save_obs_chance)

    def update(self, fpos: torch.Tensor, fneg: torch.Tensor, all_weights: bool = False):
        """Ranker.rank + es.approx_grad on the device (rankers.py:46-50, es.py:98-101).  ``all_weights``: finalise the weights
        of all K pairs on every process (``self.weights_all``; what Ranker.rank hands to a script) instead of only this
        shard's -- a few microseconds more than the shard, and no collective."""
        e = self.eng
        kb, kc = (0, self.K) if (all_weights and self.comm.size > 1) else (self.k_begin, self.k_local)
        with self._timed('rank'):
            if self.ranker is not None:
                # any Ranker of utils.rankers: one weight per pair, n_fits_ranked as the reference
                w = self.ranker.rank_device(e, fpos, fneg, kb, kc)
                n_ranked = float(self.ranker.n_fits_ranked)
            else:
                w0, w1 = (1.0, 0.0) if self.n_obj == 1 else (self.moo_w, 1 - self.moo_w)
                w = e.centered_rank(fpos, fneg, w0, w1, kb, kc)
                n_ranked = float(2 * self.K)
            self.weights_all = w if kc == self.K else None
            self.weights = w[self.k_begin:self.k_begin + self.k_local] if (kc == self.K and self.comm.size > 1) else w
        with self._timed('reconstruct'):
            e.grad_reconstruct(self.table, self.idx, self.weights, self.P, self.gsum)
        with self._timed('allreduce'):
            self.comm.allreduce_sum(self.gsum)
        with self._timed('optimizer'):
            self.apply_optimizer(self.gsum, n_ranked)

    def noiseless_eval(self):
        """The noiseless evaluation of es.py:48 for the CURRENT theta on the device (sigma = 0, float32 rollout, one
        policy split over the SMs by time tiles).  Returns (fitness f64[2], behaviour f32[2,3]); row 0 is the result."""
        e = self.eng
        if getattr(self, '_nl_bufs', None) is None:
            self._nl_bufs = (torch.zeros(2, dtype=torch.float64, device=e.device),
                             torch.zeros(2, 3, dtype=torch.float32, device=e.device),
                             torch.zeros(1, dtype=torch.int64, device=e.device))
        fit0, behv0, idx0 = self._nl_bufs
        if self.closed is not None:
            obs0, env_a, env_b = self.closed
            e.rollout_closed(self.table, idx0, self.theta, 0.0, self.layer_sizes, self.ob_mean, self.ob_std, self.ob_clip, obs0,
                             env_a, env_b, self.rew_vec, self.pos_scale, fit0[0:1], fit0[1:2], 1, behv0[0].view(-1), behv0[1].view(-1))
            return fit0, behv0
        e.rollout(self.table, idx0, self.theta, 0.0, self.layer_sizes, self.obsn, self.rew_vec, self.pos_scale,
                  fit0[0:1], fit0[1:2], 1, behv0[0].view(-1), behv0[1].view(-1), ES_ROLLOUT_F32)
        return fit0, behv0

    def skip_eval_coins(self, n_evals: int = 1):
        """Every stream discards the save_obs coin(s) of ``n_evals`` evaluations (``coins_per_eval`` doubles = 2 words each):
        the reference's fit_fn draws ``rs.random()`` in EVERY call, including the noiseless ``fit_fn(policy.pheno(zeros),
        False)`` of es.py:48 that every rank executes (simple_example.py:38, obj.py:54)."""
        if self.coins_per_eval:
            self.eng.mt_skip(self.mt_key, self.mt_pos, 2 * self.coins_per_eval * int(n_evals))

    def apply_optimizer(self, gsum: torch.Tensor, n_ranked: float):
        """grad = gsum/n_ranked; theta += optim.step(l2coeff*theta - grad)  (es.py:100-101)."""
        self.optim.apply_fused(self.eng, self.theta, gsum, n_ranked, self.l2coeff)

    def run(self, n_per_stream: int):
        """One whole generation, fully asynchronous on the current stream."""
        fpos, fneg = self.evaluate(n_per_stream)
        self.update(fpos, fneg)

    # ------------------------------------------------------------------------------------------
    @staticmethod
    def _mt_view(rs: np.random.RandomState):
        """(key uint32[624] view, pos ctypes int) straight into the RandomState's MT19937 state block (numpy exposes its
        address through the documented ``BitGenerator.ctypes`` interface), or None.  Reading / writing 2.5 kB in place costs
        a fraction of a microsecond; get_state()/set_state() cost ~40 us per stream and per direction."""
        try:
            bg = rs._bit_generator
            if type(bg).__name__ != 'MT19937':
                return None
            addr = bg.ctypes.state_address
            import ctypes
            key = np.ctypeslib.as_array((ctypes.c_uint32 * ES_MT_N).from_address(addr))
            pos = ctypes.c_int.from_address(addr + ES_MT_N * 4)
            probe = rs.get_state()                                   # one-time check that the layout is what we think
            if not (np.array_equal(key, probe[1]) and pos.value == probe[2]):
                return None
            return key, pos
        except Exception:
            return None

    def _views(self, rank_states):
        cache = getattr(self, '_mt_views', None)
        if cache is None or len(cache[0]) != len(rank_states) or any(a is not b for a, b in zip(cache[0], rank_states)):
            views = [self._mt_view(rs) for rs in rank_states]
            cache = (list(rank_states), views if all(v is not None for v in views) else None)
            self._mt_views = cache
        return cache[1]

    def load_states(self, rank_states: Sequence[np.random.RandomState]):
        """Upload the callers' RandomState streams if they moved on the host since store_states wrote them."""
        assert len(rank_states) == self.n_streams
        views = None if self.ac_std != 0.0 else self._views(rank_states)     # action noise: the gaussian cache travels too
        if views is not None:
            key = np.empty((self.n_streams, ES_MT_N), dtype=np.uint32)
            pos = np.empty(self.n_streams, dtype=np.int32)
            for r, (k, p) in enumerate(views):
                key[r] = k
                pos[r] = p.value
        else:
            states = [s.get_state() for s in rank_states]
            self._gauss = [(st[3], st[4]) for st in states]
            key = np.stack([st[1] for st in states]).astype(np.uint32, copy=False)
            pos = np.array([st[2] for st in states], dtype=np.int32)
        hs = self._host_states
        gs = None
        if views is None:
            gs = (np.array([g[0] for g in self._gauss], dtype=np.int32), np.array([g[1] for g in self._gauss], dtype=np.float64))
        if hs is not None and np.array_equal(hs[1], pos) and np.array_equal(hs[0], key) and \
                (gs is None or (hs[2] is not None and np.array_equal(hs[2][0], gs[0]) and np.array_equal(hs[2][1], gs[1]))):
            return                                  # the device already holds exactly these streams
        self._host_states = None
        self.eng.upload_async(self.mt_key, key.view(np.int32), ('mtkey', id(self)))
        self.eng.upload_async(self.mt_pos, pos, ('mtpos', id(self)))
        if gs is not None:
            self.eng.upload_async(self.mt_has, gs[0], ('mthas', id(self)))
            self.eng.upload_async(self.mt_gauss, gs[1], ('mtgauss', id(self)))

    def store_states(self, rank_states: Sequence[np.random.RandomState], key=None, pos=None, gauss=None):
        """Write the advanced streams back into the callers' RandomState objects (``key``/``pos``: already
        downloaded host copies; otherwise this synchronises).  ``gauss`` = (has_gauss int32 [R], cached float64 [R]) host
        copies, used (and downloaded when missing) only when the generation drew action noise."""
        key = (self.eng.to_host(self.mt_key) if key is None else key).view(np.uint32)
        pos = self.eng.to_host(self.mt_pos) if pos is None else pos
        if self.ac_std != 0.0:
            if gauss is None:
                gauss = (self.eng.to_host(self.mt_has), self.eng.to_host(self.mt_gauss))
            self._gauss = [(int(h), float(g)) for h, g in zip(gauss[0], gauss[1])]
            gauss = (np.array(gauss[0], dtype=np.int32, copy=True), np.array(gauss[1], dtype=np.float64, copy=True))
        else:
            gauss = None
        self._host_states = (np.array(key, dtype=np.uint32, copy=True), np.array(pos, dtype=np.int32, copy=True), gauss)
        views = None if self.ac_std != 0.0 else self._views(rank_states)
        if views is not None:
            for r, (k, p) in enumerate(views):                       # the gaussian cache of the stream is left as it is
                k[:] = key[r]
                p.value = int(pos[r])
            return
        for r, rs in enumerate(rank_states):
            rs.set_state(('MT19937', key[r], int(pos[r]), self._gauss[r][0], self._gauss[r][1]))

    def rank_states(self) -> List[np.random.RandomState]:
        """Download the MT19937 streams back into numpy RandomState objects (synchronises)."""
        key = self.mt_key.cpu().numpy().view(np.uint32)
        pos = self.mt_pos.cpu().numpy()
        if self.ac_std != 0.0:
            self._gauss = [(int(h), float(g)) for h, g in zip(self.mt_has.cpu().numpy(), self.mt_gauss.cpu().numpy())]
        out = []
        for r in range(self.n_streams):
            rs = np.random.RandomState()
            rs.set_state(('MT19937', key[r], int(pos[r]), self._gauss[r][0], self._gauss[r][1]))
            out.append(rs)
        return out


def parity_report(gen: DeviceGeneration, mode_a: int, mode_b: int = ES_ROLLOUT_F32) -> dict:
    """How far rollout arithmetic ``mode_a`` is from ``mode_b`` on IDENTICAL inputs: the indices of ``gen``'s last
    ``evaluate()`` (this process's shard), the current theta and the normalised observation stream.  Both modes roll out
    the same 2*k_local policies; each fitness vector is ranked (``es_centered_rank``, ranks over the shard) and
    reconstructed (``es_grad_reconstruct``).  Reported: how many of the 2K integer ranks differ and by how much, the largest
    change of a rank weight, ||g_a - g_b|| / ||g_b|| of the reconstructed gradient sums, and the fitness error relative to
    the population's fitness spread.  No collectives; synchronises the stream.  Used by bench.py (``also.parity``) and by
    tests/test_gpu_generation.py at BASELINE config 3."""
    e = gen.eng
    k = gen.k_local
    f64 = torch.float64
    res = {}
    for m in (mode_a, mode_b):
        f = e.empty((2, k, 1), f64)
        e.rollout(gen.table, gen.idx, gen.theta, gen.sigma, gen.layer_sizes, gen.obsn, gen.rew_vec, gen.pos_scale,
                  f[0], f[1], 1, None, None, m)
        w, r = e.centered_rank(f[0], f[1], 1.0, 0.0, 0, k, want_ranks=True)
        g = e.grad_reconstruct(gen.table, gen.idx, w, gen.P)
        res[m] = (f, w, r, g)
    e.sync()
    (fa, wa, ra, ga), (fb, wb, rb, gb) = res[mode_a], res[mode_b]
    dr = (ra.to(torch.int64) - rb.to(torch.int64)).abs()
    spread = float(fb.std().item())
    gb64, ga64 = gb.to(f64), ga.to(f64)
    return dict(pairs=k, ranks_total=int(dr.numel()), ranks_differing=int((dr != 0).sum().item()),
                max_rank_shift=int(dr.max().item()), max_abs_dw=float((wa - wb).abs().max().item()),
                grad_rel_err=float(((ga64 - gb64).norm() / gb64.norm()).item()),
                fitness_max_abs_err=float((fa - fb).abs().max().item()),
                fitness_rms_err=float((fa - fb).pow(2).mean().sqrt().item()),
                fitness_spread_std=spread,
                fitness_rms_err_over_spread=float((fa - fb).pow(2).mean().sqrt().item()) / max(spread, 1e-30))
