"""``BatchedRollout``: the fit_fn that lets ``es.test_params`` / ``es.step`` evaluate ALL of a
rank's antithetic pairs in one fused launch.

The reference's ``fit_fn`` is an opaque per-policy python callback (src/core/es.py:28,71-72),
which forces one rollout per call.  A ``BatchedRollout`` is still callable like that (it is
what ``es.step`` uses for the noiseless evaluation, es.py:48) but it also *describes* the
evaluation -- env, episode length, how many ``rs.random()`` coins the script's fit_fn draws
per evaluation, how many episodes it averages (obj.py's eps_per_policy), which TrainingResult
adaptor it builds -- so the generation can run on the device with the same RNG consumption and
the same results layout.
"""
from __future__ import annotations

from typing import Optional, Sequence

import numpy as np

from .. import _lib
from .gym_runner import run_model
from .training_result import NSRResult, RewardResult, TrainingResult


class BatchedRollout:
    is_batched_rollout = True

    def __init__(self, env, max_steps: int, coins_per_eval: int = 1, save_obs_chance: float = 0.0,
                 archive: Optional[np.ndarray] = None, nov_k: int = 10,
                 rank_streams: Optional[Sequence[np.random.RandomState]] = None,
                 rollout_mode: int = _lib.ES_ROLLOUT_F32, eps_per_policy: int = 1):
        """``eps_per_policy``: episodes per evaluation, ``cfg.general.eps_per_policy`` of obj.py's fit_fn (obj.py:56-60): each
        draws its own action noise from the stream, the per-step rewards are averaged over them and the behaviour is the
        last episode's.  Values below 1 mean one episode, as ``max(1, eps_per_policy)`` does there."""
        if not (getattr(env, 'is_synthetic_openloop', False) or getattr(env, 'is_synthetic_closedloop', False)):
            raise TypeError('BatchedRollout needs a synthetic env (es_pytorch_b200.gym.synthetic_env: open- or closed-loop)')
        self.env = env
        self.max_steps = min(int(max_steps), env.T)
        self.coins_per_eval = int(coins_per_eval)
        self.save_obs_chance = float(save_obs_chance)
        self.archive = None if archive is None else np.asarray(archive, dtype=np.float64)
        self.nov_k = int(nov_k)
        self.rank_streams = list(rank_streams) if rank_streams is not None else None
        self.rollout_mode = rollout_mode
        self.eps_per_policy = max(1, int(eps_per_policy))
        if self.eps_per_policy > 1 and self.archive is not None:
            # nsra.py's fit_fn runs one episode; several episodes with a novelty objective have no reference counterpart
            raise ValueError('BatchedRollout: eps_per_policy > 1 averages the reward of several episodes (obj.py); it cannot be '
                             'combined with an archive (novelty objective, nsra.py runs one episode per evaluation)')
        self._gen = None            # cached DeviceGeneration (see core.es)
        self._streams_in_use = None  # the RandomState streams of the last batched evaluation (set by core.es)
        self.stream_env_from_host = False   # True: re-upload the env's obs/reward streams every generation

    @property
    def n_obj(self) -> int:
        return 1 if self.archive is None else 2

    def result_from_device(self, total: float, pos) -> TrainingResult:
        """The TrainingResult ``__call__`` would build, from an episode total and final position computed on the device."""
        rews = [float(total)]
        behv = [float(pos[0]), float(pos[1]), float(pos[2])] * int(self.max_steps)
        no_obs = np.array([np.zeros(self.env.observation_space.shape)])
        steps = self.max_steps - 1                              # run_model returns the last loop index (gym_runner.py:50,67)
        if self.archive is None:
            return RewardResult(rews, behv, no_obs, steps)
        return NSRResult(rews, behv[-3:], no_obs, steps, self.archive, self.nov_k)

    def __call__(self, model, use_ac_noise=True) -> TrainingResult:
        """Single-policy evaluation with the reference's fit_fn contract.  Like the scripts' fit_fn (simple_example.py:38,
        obj.py:54) it first draws the save_obs coin(s) -- from every stream this process carries: each stream is one
        reference rank, and every rank runs its own noiseless evaluation (es.py:48).  ``use_ac_noise`` (obj.py:53-55): the
        rollout draws the policy's action noise from the first stream; es.step's noiseless call passes False.
        ``eps_per_policy`` > 1 with action noise: obj.py's episode loop, one launch for all episodes on the open-loop env."""
        streams = self.rank_streams if self.rank_streams is not None else self._streams_in_use
        if streams is not None:
            for rs in streams:
                for _ in range(self.coins_per_eval):
                    rs.random()
        noise_rs = streams[0] if (use_ac_noise and streams is not None and len(streams)) else None
        closed = getattr(self.env, 'is_synthetic_closedloop', False)
        if (closed and hasattr(model, 'is_tanh_mlp') and model.is_tanh_mlp() and len(model.layer_sizes()) == 4
                and not (noise_rs is not None and float(getattr(model, '_action_std', 0) or 0) != 0)):
            # the closed-loop episode as one launch (the observations are not returned: this result never carries them)
            from .gym_runner import _device_episode_closed
            total, pos, _ = _device_episode_closed(model, self.env, self.max_steps)
            return self.result_from_device(total, pos)
        E = self.eps_per_policy
        if E > 1 and noise_rs is not None and float(getattr(model, '_action_std', 0) or 0) != 0:
            if getattr(self.env, 'is_synthetic_openloop', False) and hasattr(model, 'is_tanh_mlp') and model.is_tanh_mlp():
                from .gym_runner import _device_episode
                total, pos, _ = _device_episode(model, self.env, self.max_steps, noise_rs, n_episodes=E)
                return self.result_from_device(total, pos)
            rews = np.zeros(self.max_steps)                    # obj.py:55-60 as written
            for _ in range(E):
                rew, behv, obs, steps = run_model(model, self.env, self.max_steps, noise_rs)
                rews[:len(rew)] += np.array(rew)
            rews /= E
            return RewardResult(rews.tolist(), behv, np.array([np.zeros(self.env.observation_space.shape)]), steps)
        # without action noise every episode is the same one: their per-step average is its reward, exactly
        rews, behv, obs, steps = run_model(model, self.env, self.max_steps, noise_rs)
        no_obs = np.array([np.zeros(self.env.observation_space.shape)])
        if self.archive is None:
            return RewardResult(rews, behv, no_obs, steps)
        return NSRResult(rews, behv[-3:], no_obs, steps, self.archive, self.nov_k)
