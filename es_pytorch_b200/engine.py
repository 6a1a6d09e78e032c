"""Device engine: one ``es_ctx`` per GPU, thin typed wrappers over the C ABI.

PyTorch is the container only: tensors provide device memory, streams come from
``torch.cuda.current_stream()``; every computation is a libes_b200.so kernel.
"""
from __future__ import annotations

import ctypes as C
import weakref
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from ._lib import ES_ROLLOUT_F32, ES_ROLLOUT_TC, ES_ROLLOUT_TC3, ES_MT_N, check

_ENGINES = {}


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _req(t: torch.Tensor, dtype, name: str, device: torch.device):
    if not isinstance(t, torch.Tensor):
        raise TypeError(f'{name}: expected a torch tensor, got {type(t)}')
    if t.dtype != dtype:
        raise TypeError(f'{name}: expected dtype {dtype}, got {t.dtype}')
    if t.device != device:
        raise ValueError(f'{name}: tensor is on {t.device}, engine is on {device}')
    if not t.is_contiguous():
        raise ValueError(f'{name}: tensor must be contiguous')
    return t


class Engine:
    """All device work of one GPU goes through one Engine (one es_ctx)."""

    def __init__(self, device_index: int = 0):
        if not torch.cuda.is_available():
            raise _lib.EsLibraryError('es_pytorch_b200 needs a CUDA device (B200, sm_100a); there is no CPU path')
        self.lib = _lib.load()
        self.device = torch.device('cuda', device_index)
        torch.cuda.set_device(self.device)
        torch.zeros(1, device=self.device)          # make sure the primary context exists
        h = C.c_void_p()
        check(self.lib.es_ctx_create(device_index, C.byref(h)), 'es_ctx_create')
        self._ctx = h
        self.h2d_bytes = 0          # bytes copied host->device / device->host through this engine
        self.d2h_bytes = 0
        self._pin = {}
        self._pin_events = {}

    # ------------------------------------------------------------------ plumbing
    @property
    def stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    @property
    def launches(self) -> int:
        return int(self.lib.es_launch_count(self._ctx))

    @property
    def sm_count(self) -> int:
        return int(self.lib.es_sm_count(self._ctx))

    def empty(self, shape, dtype):
        return torch.empty(shape, dtype=dtype, device=self.device)

    def zeros(self, shape, dtype):
        return torch.zeros(shape, dtype=dtype, device=self.device)

    def to_device(self, a, dtype=None) -> torch.Tensor:
        if isinstance(a, torch.Tensor):
            t = a
        else:
            t = torch.from_numpy(np.ascontiguousarray(a))
        if dtype is not None and t.dtype != dtype:
            t = t.to(dtype)
        if not t.is_cuda:
            self.h2d_bytes += t.numel() * t.element_size()
        return t.to(self.device, non_blocking=True).contiguous()

    def upload_into(self, dst: torch.Tensor, src) -> torch.Tensor:
        """Copy a host array into an existing device tensor (counts the bytes)."""
        t = src if isinstance(src, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(src))
        self.h2d_bytes += t.numel() * t.element_size()
        dst.copy_(t.view(dst.shape) if t.numel() == dst.numel() else t, non_blocking=True)
        return dst

    # -- pinned staging: asynchronous transfers, one synchronisation per API call -------------------------------
    def _pinned(self, key, shape, dtype) -> torch.Tensor:
        buf = self._pin.get(key)
        if buf is None or buf.shape != torch.Size(shape) or buf.dtype != dtype:
            buf = self._pin[key] = torch.empty(shape, dtype=dtype, pin_memory=True)
        return buf

    def upload_async(self, dst: torch.Tensor, src, key, src_pinned: bool = False) -> torch.Tensor:
        """host array -> device without blocking the host.  ``src_pinned=True``: the caller guarantees the source
        lives in page-locked memory and is copied directly; anything else goes through a pinned staging buffer
        named ``key`` (no per-call cudaPointerGetAttributes query)."""
        a = src if isinstance(src, torch.Tensor) else torch.from_numpy(src if src.flags.c_contiguous else np.ascontiguousarray(src))
        self.h2d_bytes += a.numel() * a.element_size()
        if src_pinned:
            dst.copy_(a.view(dst.shape), non_blocking=True)
            return dst
        st = self._pinned(key, tuple(a.shape), a.dtype)
        ev = self._pin_events.get(key)
        if ev is not None and not ev.query():          # the previous use of this staging buffer is still in flight
            ev.synchronize()
        st.copy_(a)
        dst.copy_(st.view(dst.shape), non_blocking=True)
        if ev is None:
            ev = self._pin_events[key] = torch.cuda.Event()
        ev.record()
        return dst

    def download_async(self, t: torch.Tensor, key) -> torch.Tensor:
        """device -> pinned staging (asynchronous); call ``sync()`` before reading the returned pinned tensor."""
        st = self._pinned(('d2h', key), tuple(t.shape), t.dtype)
        st.copy_(t, non_blocking=True)
        self.d2h_bytes += t.numel() * t.element_size()
        return st

    def sync(self):
        """Synchronise the current stream, then surface what the kernels flagged asynchronously (a noise index outside
        the table: the reference's ``assert len(self) > i + size``, noisetable.py:34)."""
        torch.cuda.current_stream(self.device).synchronize()
        check(self.lib.es_check_async(self._ctx), 'es_check_async')

    def to_host(self, t: torch.Tensor) -> np.ndarray:
        """Device tensor -> numpy (synchronises the stream; counts the bytes)."""
        self.d2h_bytes += t.numel() * t.element_size()
        return t.cpu().numpy()

    # ------------------------------------------------------------------ a2
    def draw_indices(self, mt_key: torch.Tensor, mt_pos: torch.Tensor, n_per_stream: int, upper_bound: int,
                     extra_words: int = 0, idx_out: Optional[torch.Tensor] = None,
                     extra_out: Optional[torch.Tensor] = None):
        """mt_key int32/uint32-as-int32 [R,624], mt_pos int32 [R]; both updated in place."""
        d = self.device
        R = mt_key.shape[0]
        _req(mt_key, torch.int32, 'mt_key', d)
        _req(mt_pos, torch.int32, 'mt_pos', d)
        assert mt_key.shape == (R, ES_MT_N) and mt_pos.shape == (R,)
        if idx_out is None:
            idx_out = self.empty((R * n_per_stream,), torch.int64)
        _req(idx_out, torch.int64, 'idx_out', d)
        assert idx_out.numel() == R * n_per_stream
        if extra_words and extra_out is None:
            extra_out = self.empty((R * n_per_stream, extra_words), torch.int32)
        if extra_out is not None:
            _req(extra_out, torch.int32, 'extra_out', d)
            assert extra_out.numel() == R * n_per_stream * extra_words
        check(self.lib.es_draw_indices(self._ctx, _ptr(mt_key), _ptr(mt_pos), R, n_per_stream, int(upper_bound),
                                       extra_words, _ptr(idx_out), _ptr(extra_out), self.stream), 'es_draw_indices')
        return idx_out, extra_out

    def mt_skip(self, mt_key: torch.Tensor, mt_pos: torch.Tensor, n_words: int):
        """Advance every stream by ``n_words`` raw 32-bit outputs (a discarded ``rs.random()`` is 2 words)."""
        d = self.device
        _req(mt_key, torch.int32, 'mt_key', d); _req(mt_pos, torch.int32, 'mt_pos', d)
        check(self.lib.es_mt_skip(self._ctx, _ptr(mt_key), _ptr(mt_pos), mt_key.shape[0], int(n_words), self.stream),
              'es_mt_skip')

    def draw_noisy(self, mt_key, mt_pos, has_gauss, gauss, n_per_stream: int, upper_bound: int, coins_per_eval: int,
                   normals_per_eval: int, scale: float, idx_out=None, coin_out=None, noise_out=None):
        """All draws of a generation whose policy adds action noise, in the reference's stream order (es_draw_noisy):
        per pair randint, then per evaluation ``coins_per_eval`` doubles and ``normals_per_eval`` legacy gaussians.
        has_gauss int32 [R] / gauss float64 [R] are the streams' cached-gaussian state, updated in place.  Returns
        (idx int64 [R*n], coin words int32 [R*n, 4*coins] or None, noise float32 [R*n, 2, normals_per_eval])."""
        d = self.device
        R = mt_key.shape[0]
        _req(mt_key, torch.int32, 'mt_key', d); _req(mt_pos, torch.int32, 'mt_pos', d)
        _req(has_gauss, torch.int32, 'has_gauss', d); _req(gauss, torch.float64, 'gauss', d)
        assert mt_key.shape == (R, ES_MT_N) and mt_pos.numel() == R and has_gauss.numel() == R and gauss.numel() == R
        n = R * n_per_stream
        if idx_out is None:
            idx_out = self.empty((n,), torch.int64)
        if coins_per_eval and coin_out is None:
            coin_out = self.empty((n, 4 * coins_per_eval), torch.int32)
        if noise_out is None:
            noise_out = self.empty((n, 2, normals_per_eval), torch.float32)
        _req(idx_out, torch.int64, 'idx_out', d); _req(noise_out, torch.float32, 'noise_out', d)
        assert idx_out.numel() == n and noise_out.numel() == n * 2 * normals_per_eval
        if coin_out is not None:
            _req(coin_out, torch.int32, 'coin_out', d)
            assert coin_out.numel() == n * 4 * coins_per_eval
        check(self.lib.es_draw_noisy(self._ctx, _ptr(mt_key), _ptr(mt_pos), _ptr(has_gauss), _ptr(gauss), R, int(n_per_stream),
                                     int(upper_bound), int(coins_per_eval), int(normals_per_eval), float(scale), _ptr(idx_out),
                                     _ptr(coin_out), _ptr(noise_out), self.stream), 'es_draw_noisy')
        return idx_out, coin_out, noise_out

    # ------------------------------------------------------------------ a3
    def perturb(self, theta, table, idx, sigma: float, want_neg: bool = True):
        d = self.device
        _req(theta, torch.float32, 'theta', d); _req(table, torch.float32, 'table', d); _req(idx, torch.int64, 'idx', d)
        n, P = idx.numel(), theta.numel()
        out_pos = self.empty((n, P), torch.float32)
        out_neg = self.empty((n, P), torch.float32) if want_neg else None
        check(self.lib.es_perturb(self._ctx, _ptr(theta), _ptr(table), table.numel(), _ptr(idx), n, P, float(sigma),
                                  _ptr(out_pos), _ptr(out_neg), self.stream), 'es_perturb')
        return out_pos, out_neg

    # ------------------------------------------------------------------ a4
    def normalise_obs(self, obs, mean, std, clip: float, out: Optional[torch.Tensor] = None):
        d = self.device
        _req(obs, torch.float32, 'obs', d); _req(mean, torch.float64, 'mean', d); _req(std, torch.float64, 'std', d)
        rows, obs_dim = obs.shape
        assert mean.numel() == obs_dim and std.numel() == obs_dim
        if out is None:
            out = self.empty((rows, obs_dim), torch.float32)
        _req(out, torch.float32, 'out', d)
        check(self.lib.es_normalise_obs(self._ctx, _ptr(obs), _ptr(mean), _ptr(std), float(clip), rows, obs_dim,
                                        _ptr(out), self.stream), 'es_normalise_obs')
        return out

    def obs_colsum(self, obs):
        d = self.device
        _req(obs, torch.float32, 'obs', d)
        rows, obs_dim = obs.shape
        s = self.empty((obs_dim,), torch.float32)
        q = self.empty((obs_dim,), torch.float32)
        check(self.lib.es_obs_colsum(self._ctx, _ptr(obs), rows, obs_dim, _ptr(s), _ptr(q), self.stream), 'es_obs_colsum')
        return s, q

    def obstat_accumulate(self, osum, osumsq, s, q, n_rollouts: int):
        d = self.device
        _req(osum, torch.float64, 'sum', d); _req(osumsq, torch.float64, 'sumsq', d)
        _req(s, torch.float32, 's', d); _req(q, torch.float32, 'ssq', d)
        check(self.lib.es_obstat_accumulate(self._ctx, _ptr(osum), _ptr(osumsq), _ptr(s), _ptr(q), osum.numel(),
                                            int(n_rollouts), self.stream), 'es_obstat_accumulate')

    def obstat_accumulate_coins(self, osum, osumsq, count_io, s, q, rows_per_rollout: int, coin_words, chance: float):
        """coin_words int32 [n_coins, 2]; count_io float64 [2] (count in/out, n_saved out)."""
        d = self.device
        _req(osum, torch.float64, 'sum', d); _req(osumsq, torch.float64, 'sumsq', d)
        _req(count_io, torch.float64, 'count_io', d)
        _req(s, torch.float32, 's', d); _req(q, torch.float32, 'ssq', d)
        _req(coin_words, torch.int32, 'coin_words', d)
        check(self.lib.es_obstat_accumulate_coins(self._ctx, _ptr(osum), _ptr(osumsq), _ptr(count_io), _ptr(s), _ptr(q),
                                                  osum.numel(), int(rows_per_rollout), _ptr(coin_words),
                                                  coin_words.numel() // 2, float(chance), self.stream),
              'es_obstat_accumulate_coins')

    # ------------------------------------------------------------------ a3+a4+a5
    def rollout(self, table, idx, theta, sigma: float, layer_sizes: Sequence[int], obsn, rew_vec, pos_scale: float,
                fit_pos, fit_neg, fit_stride: int = 1, behv_pos=None, behv_neg=None, mode: int = ES_ROLLOUT_F32,
                act_noise=None, n_episodes: int = 1):
        """``act_noise``: float32 [n_pairs, 2, n_episodes, T, act] scaled action noise (``draw_noisy``), added to every
        action.  ``n_episodes`` > 1: every evaluation is that many episodes (obj.py's eps_per_policy), each with its own
        noise; fitness = their per-step average summed, behaviour = the last episode's (``rollout_episodes``)."""
        self._rollout(table, idx, theta, sigma, layer_sizes, obsn, rew_vec, pos_scale, fit_pos, fit_neg, fit_stride, behv_pos,
                      behv_neg, mode, act_noise, n_episodes, n_episodes != 1)

    def rollout_episodes(self, table, idx, theta, sigma: float, layer_sizes: Sequence[int], obsn, rew_vec, pos_scale: float,
                         fit_pos, fit_neg, fit_stride: int = 1, behv_pos=None, behv_neg=None, mode: int = ES_ROLLOUT_F32,
                         act_noise=None, n_episodes: int = 1):
        """es_rollout_openloop_episodes for any ``n_episodes`` (``rollout`` takes es_rollout_openloop_noisy for one episode;
        both give the same results then).  The library rejects n_episodes < 1 and n_episodes * T * act > INT_MAX."""
        self._rollout(table, idx, theta, sigma, layer_sizes, obsn, rew_vec, pos_scale, fit_pos, fit_neg, fit_stride, behv_pos,
                      behv_neg, mode, act_noise, n_episodes, True)

    def _rollout(self, table, idx, theta, sigma, layer_sizes, obsn, rew_vec, pos_scale, fit_pos, fit_neg, fit_stride, behv_pos,
                 behv_neg, mode, act_noise, n_episodes, episodes_entry):
        d = self.device
        _req(table, torch.float32, 'table', d); _req(idx, torch.int64, 'idx', d); _req(theta, torch.float32, 'theta', d)
        _req(obsn, torch.float32, 'obsn', d); _req(rew_vec, torch.float32, 'rew_vec', d)
        _req(fit_pos, torch.float64, 'fit_pos', d); _req(fit_neg, torch.float64, 'fit_neg', d)
        n = idx.numel()
        T = obsn.shape[0]
        assert obsn.shape[1] == layer_sizes[0] and rew_vec.shape == (T, layer_sizes[-1])
        assert fit_pos.numel() >= n * fit_stride and fit_neg.numel() >= n * fit_stride
        if behv_pos is not None:
            _req(behv_pos, torch.float32, 'behv_pos', d); _req(behv_neg, torch.float32, 'behv_neg', d)
            assert behv_pos.numel() == 3 * n and behv_neg.numel() == 3 * n
        if act_noise is not None:
            _req(act_noise, torch.float32, 'act_noise', d)
            assert n_episodes < 1 or act_noise.numel() == n * 2 * int(n_episodes) * T * layer_sizes[-1]
        ls = (C.c_int * len(layer_sizes))(*[int(x) for x in layer_sizes])
        if mode in (ES_ROLLOUT_TC, ES_ROLLOUT_TC3):
            # the library keeps a bf16 shadow of the table keyed by (pointer, length); a different tensor object (the
            # caching allocator reuses addresses) or an in-place torch write (version counter) invalidates it
            ref, ver = getattr(self, '_tc_table', (None, None))
            if ref is None or ref() is not table or ver != table._version:
                check(self.lib.es_noise_table_changed(self._ctx), 'es_noise_table_changed')
                self._tc_table = (weakref.ref(table), table._version)
        if episodes_entry:
            check(self.lib.es_rollout_openloop_episodes(self._ctx, _ptr(table), table.numel(), _ptr(idx), n, _ptr(theta),
                                                        theta.numel(), float(sigma), ls, len(layer_sizes) - 1, _ptr(obsn),
                                                        _ptr(rew_vec), T, float(pos_scale), _ptr(fit_pos), _ptr(fit_neg),
                                                        int(fit_stride), _ptr(behv_pos), _ptr(behv_neg), _ptr(act_noise),
                                                        int(n_episodes), int(mode), self.stream), 'es_rollout_openloop_episodes')
            return
        check(self.lib.es_rollout_openloop_noisy(self._ctx, _ptr(table), table.numel(), _ptr(idx), n, _ptr(theta),
                                                 theta.numel(), float(sigma), ls, len(layer_sizes) - 1, _ptr(obsn),
                                                 _ptr(rew_vec), T, float(pos_scale), _ptr(fit_pos), _ptr(fit_neg),
                                                 int(fit_stride), _ptr(behv_pos), _ptr(behv_neg), _ptr(act_noise), int(mode),
                                                 self.stream), 'es_rollout_openloop')

    def rollout_closed(self, table, idx, theta, sigma: float, layer_sizes: Sequence[int], ob_mean, ob_std, ob_clip: float,
                       obs0, env_a, env_b, rew_vec, pos_scale: float, fit_pos, fit_neg, fit_stride: int = 1, behv_pos=None,
                       behv_neg=None, coin_words=None, save_obs_chance: float = 0.0, ob_sum=None, ob_sumsq=None, ob_count=None):
        """Antithetic pairs on the closed-loop synthetic env (``gym.synthetic_env.ClosedLoopEnv``): ``env_a`` [band, obs] and
        ``env_b`` [act, obs] are the transposed transition matrices, ``obs0`` the start observation; the observation
        normalisation (``ob_mean`` / ``ob_std`` float64, ``ob_clip``) happens inside.  ``coin_words`` [n, 4] + the three
        float64 statistics buffers: ObStat increments of the evaluations whose save_obs coin fell."""
        d = self.device
        _req(table, torch.float32, 'table', d); _req(idx, torch.int64, 'idx', d); _req(theta, torch.float32, 'theta', d)
        _req(ob_mean, torch.float64, 'ob_mean', d); _req(ob_std, torch.float64, 'ob_std', d)
        _req(obs0, torch.float32, 'obs0', d); _req(env_a, torch.float32, 'env_a', d); _req(env_b, torch.float32, 'env_b', d)
        _req(rew_vec, torch.float32, 'rew_vec', d)
        _req(fit_pos, torch.float64, 'fit_pos', d); _req(fit_neg, torch.float64, 'fit_neg', d)
        n, T, obs, act = idx.numel(), rew_vec.shape[0], int(layer_sizes[0]), int(layer_sizes[-1])
        band = env_a.shape[0]
        assert env_a.shape == (band, obs) and env_b.shape == (act, obs) and obs0.numel() == obs and rew_vec.shape == (T, act)
        assert ob_mean.numel() == obs and ob_std.numel() == obs
        assert fit_pos.numel() >= n * fit_stride and fit_neg.numel() >= n * fit_stride
        if behv_pos is not None:
            _req(behv_pos, torch.float32, 'behv_pos', d); _req(behv_neg, torch.float32, 'behv_neg', d)
            assert behv_pos.numel() == 3 * n and behv_neg.numel() == 3 * n
        if coin_words is not None:
            assert coin_words.dtype == torch.int32 and coin_words.numel() == 4 * n and coin_words.is_contiguous()
        if ob_sum is not None:
            _req(ob_sum, torch.float64, 'ob_sum', d); _req(ob_sumsq, torch.float64, 'ob_sumsq', d); _req(ob_count, torch.float64, 'ob_count', d)
            assert ob_sum.numel() == obs and ob_sumsq.numel() == obs and ob_count.numel() == 2
        ls = (C.c_int * len(layer_sizes))(*[int(x) for x in layer_sizes])
        check(self.lib.es_rollout_closedloop(self._ctx, _ptr(table), table.numel(), _ptr(idx), n, _ptr(theta), theta.numel(),
                                             float(sigma), ls, len(layer_sizes) - 1, _ptr(ob_mean), _ptr(ob_std), float(ob_clip),
                                             _ptr(obs0), _ptr(env_a), int(band), _ptr(env_b), _ptr(rew_vec), T, float(pos_scale),
                                             _ptr(coin_words), float(save_obs_chance), _ptr(fit_pos), _ptr(fit_neg),
                                             int(fit_stride), _ptr(behv_pos), _ptr(behv_neg), _ptr(ob_sum), _ptr(ob_sumsq),
                                             _ptr(ob_count), self.stream), 'es_rollout_closedloop')

    # ------------------------------------------------------------------ a13
    def novelty(self, behv, archive, k: int, out, out_stride: int = 1):
        d = self.device
        _req(behv, torch.float32, 'behv', d); _req(archive, torch.float64, 'archive', d); _req(out, torch.float64, 'out', d)
        n = behv.numel() // 3
        A = archive.shape[0]
        assert archive.shape == (A, 2)
        check(self.lib.es_novelty(self._ctx, _ptr(behv), n, _ptr(archive), A, int(k), _ptr(out), int(out_stride),
                                  self.stream), 'es_novelty')

    # ------------------------------------------------------------------ a8/a9
    def centered_rank(self, fpos, fneg, w0: float = 1.0, w1: float = 0.0, k_begin: int = 0,
                      k_count: Optional[int] = None, want_ranks: bool = False):
        d = self.device
        _req(fpos, torch.float64, 'fpos', d); _req(fneg, torch.float64, 'fneg', d)
        if fpos.dim() == 1:
            fpos, fneg = fpos.view(-1, 1), fneg.view(-1, 1)
        K, n_obj = fpos.shape
        assert fneg.shape == (K, n_obj)
        if k_count is None:
            k_count = K - k_begin
        weights = self.empty((k_count,), torch.float32)
        ranks = self.empty((n_obj, 2, k_count), torch.int32) if want_ranks else None
        check(self.lib.es_centered_rank(self._ctx, _ptr(fpos), _ptr(fneg), K, n_obj, float(w0), float(w1), int(k_begin),
                                        int(k_count), _ptr(weights), _ptr(ranks), self.stream), 'es_centered_rank')
        return (weights, ranks) if want_ranks else weights

    # ------------------------------------------------------------------ f4 (rankers.py:61-103)
    def rank_transform(self, fpos, fneg, kind: int = 0, w0: float = 1.0, w1: float = 0.0, elite_n: int = 0,
                       k_begin: int = 0, k_count: Optional[int] = None, noise_idx=None, want64: bool = False,
                       want_ranks: bool = False, want_elite: bool = False):
        """Returns a dict: 'weights' f32[k_count] and, on request, 'weights64', 'ranks', 'elite_vals' / 'elite_fit' /
        'elite_idx' (compact EliteRanker lists in ascending rank order)."""
        d = self.device
        _req(fpos, torch.float64, 'fpos', d); _req(fneg, torch.float64, 'fneg', d)
        if fpos.dim() == 1:
            fpos, fneg = fpos.view(-1, 1), fneg.view(-1, 1)
        K, n_obj = fpos.shape
        assert fneg.shape == (K, n_obj)
        if k_count is None:
            k_count = K - k_begin
        out = {'weights': self.empty((k_count,), torch.float32)}
        if want64:
            out['weights64'] = self.empty((k_count,), torch.float64)
        if want_ranks:
            out['ranks'] = self.empty((n_obj, 2, k_count), torch.int32)
        if want_elite and elite_n > 0:
            out['elite_vals'] = self.zeros((elite_n,), torch.float64)
            out['elite_fit'] = self.zeros((elite_n,), torch.int32)
            if noise_idx is not None:
                _req(noise_idx, torch.int64, 'noise_idx', d)
                assert noise_idx.numel() == K
                out['elite_idx'] = self.zeros((elite_n,), torch.int64)
        check(self.lib.es_rank_transform(self._ctx, _ptr(fpos), _ptr(fneg), K, n_obj, int(kind), float(w0), float(w1),
                                         int(elite_n), int(k_begin), int(k_count), _ptr(noise_idx), _ptr(out['weights']),
                                         _ptr(out.get('weights64')), _ptr(out.get('ranks')), _ptr(out.get('elite_vals')),
                                         _ptr(out.get('elite_fit')), _ptr(out.get('elite_idx')), self.stream),
              'es_rank_transform')
        return out

    # ------------------------------------------------------------------ a10
    def grad_reconstruct(self, table, idx, weights, P: int, out: Optional[torch.Tensor] = None):
        d = self.device
        _req(table, torch.float32, 'table', d); _req(idx, torch.int64, 'idx', d); _req(weights, torch.float32, 'weights', d)
        assert idx.numel() == weights.numel()
        if out is None:
            out = self.empty((P,), torch.float32)
        _req(out, torch.float32, 'out', d)
        check(self.lib.es_grad_reconstruct(self._ctx, _ptr(table), table.numel(), _ptr(idx), _ptr(weights),
                                           idx.numel(), int(P), _ptr(out), self.stream), 'es_grad_reconstruct')
        return out

    # ------------------------------------------------------------------ a11/a12
    def adam_step(self, theta, m, v, gsum, n_ranked: float, l2coeff: float, neg_a: float, beta1: float, beta2: float,
                  epsilon: float):
        d = self.device
        for t, nme in ((theta, 'theta'), (m, 'm'), (v, 'v'), (gsum, 'gsum')):
            _req(t, torch.float32, nme, d)
        f = float   # ctypes rounds the double to float32 (round-to-nearest), as numpy does for a python scalar
        check(self.lib.es_adam_step(self._ctx, _ptr(theta), _ptr(m), _ptr(v), _ptr(gsum), f(n_ranked), f(l2coeff),
                                    f(neg_a), f(beta1), f(1 - beta1), f(beta2), f(1 - beta2), f(epsilon),
                                    theta.numel(), self.stream), 'es_adam_step')

    def sgd_step(self, theta, v, gsum, n_ranked: float, l2coeff: float, lr: float, momentum: float):
        d = self.device
        for t, nme in ((theta, 'theta'), (v, 'v'), (gsum, 'gsum')):
            _req(t, torch.float32, nme, d)
        f = float   # ctypes rounds the double to float32 (round-to-nearest), as numpy does for a python scalar
        check(self.lib.es_sgd_step(self._ctx, _ptr(theta), _ptr(v), _ptr(gsum), f(n_ranked), f(l2coeff), f(-lr),
                                   f(momentum), f(1. - momentum), theta.numel(), self.stream), 'es_sgd_step')

    def simple_step(self, theta, gsum, n_ranked: float, l2coeff: float, lr: float):
        d = self.device
        _req(theta, torch.float32, 'theta', d); _req(gsum, torch.float32, 'gsum', d)
        f = float   # ctypes rounds the double to float32 (round-to-nearest), as numpy does for a python scalar
        check(self.lib.es_simple_step(self._ctx, _ptr(theta), _ptr(gsum), f(n_ranked), f(l2coeff), f(lr),
                                      theta.numel(), self.stream), 'es_simple_step')

    def __del__(self):
        try:
            if getattr(self, '_ctx', None):
                self.lib.es_ctx_destroy(self._ctx)
                self._ctx = None
        except Exception:
            pass


def get_engine(device_index: Optional[int] = None) -> Engine:
    """Process-wide engine for a device (default: the current CUDA device)."""
    if device_index is None:
        if not torch.cuda.is_available():
            raise _lib.EsLibraryError('es_pytorch_b200 needs a CUDA device (B200, sm_100a); there is no CPU path')
        device_index = torch.cuda.current_device()
    eng = _ENGINES.get(device_index)
    if eng is None:
        eng = _ENGINES[device_index] = Engine(device_index)
    return eng
