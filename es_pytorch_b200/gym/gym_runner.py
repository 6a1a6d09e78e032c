"""Rollout runner (mirror of src/gym/gym_runner.py:33-67).

``run_model`` keeps the reference signature.  When the env is the synthetic open-loop env
and the model is a tanh ``FeedForward``, the whole episode is ONE launch of the fused rollout
kernel (per-policy compatibility path: theta' is the module's current weights, sigma = 0;
action noise, nn.py:47-48, is drawn from ``rs`` for the whole episode at once and added on
the device); any other env is stepped in the reference's python loop with the module's own
forward.
"""
from __future__ import annotations

import time
from typing import Callable, List, Tuple

import numpy as np
import torch


def pybullet_envs_pos(env):
    return env.robot.body_real_xyz


def pybullet_gym_pos(env):
    return env.robot.robot_body.pose().xyz()


def mujoco_pos(env):
    """Centre of mass of a mujoco model (gym_runner.py:25-30)."""
    mass = np.reshape(env.model.body_mass, (-1, 1))
    centre = np.sum(mass * env.data.xipos, 0) / np.sum(mass)
    return centre[0], centre[1], centre[2]


def hbaselines_pos(env):
    return tuple(env.wrapped_env.get_body_com('torso')[:3])


def _device_episode(model, env, max_steps: int, rs=None, n_episodes: int = 1):
    """``n_episodes`` > 1 (obj.py's eps_per_policy): that many episodes with their own action noise, one launch of
    es_rollout_openloop_episodes; the total is their per-step average summed, the position the last episode's."""
    from ..engine import get_engine
    from ..core.policy import Policy
    eng = get_engine()
    sizes = model.layer_sizes()
    T = min(int(max_steps), env.T)
    obs_dev, rew_dev = env.device_arrays(eng)
    theta = eng.to_device(Policy.get_flat(model), torch.float32)
    P = theta.numel()
    mean = eng.to_device(np.ascontiguousarray(model._obmean, dtype=np.float64).reshape(-1), torch.float64)
    std = eng.to_device(np.ascontiguousarray(model._obstd, dtype=np.float64).reshape(-1), torch.float64)
    obsn = eng.normalise_obs(obs_dev[:T], mean, std, float(model.ob_clip))
    table = torch.zeros(P + 1, dtype=torch.float32, device=eng.device)      # sigma = 0: the slice is irrelevant
    idx = torch.zeros(1, dtype=torch.int64, device=eng.device)
    fit = torch.zeros(2, dtype=torch.float64, device=eng.device)
    behv = torch.zeros(2, 3, dtype=torch.float32, device=eng.device)
    noise = None
    ac_std = float(getattr(model, '_action_std', 0) or 0)
    E = 1
    if rs is not None and ac_std != 0:
        # nn.py:47-48: T calls of rs.randn(act) * ac_std; one call of rs.randn(T * act) consumes the stream identically
        # (legacy gaussians are produced one by one, cached second value included); E episodes in a row: rs.randn(E * T * act).
        # [pair 0][+ | -][E][T][act]: both evaluations of the sigma = 0 "pair" see the same noise, only the first is used.
        E = max(1, int(n_episodes))
        nz = (rs.randn(E * T * sizes[-1]) * ac_std).astype(np.float32)
        noise = eng.to_device(np.stack([nz, nz]).reshape(1, 2, -1))
    eng.rollout(table, idx, theta, 0.0, sizes, obsn, rew_dev[:T].contiguous(), env.pos_scale, fit[0:1], fit[1:2], 1,
                behv[0:1].view(-1), behv[1:2].view(-1), act_noise=noise, n_episodes=E)
    return float(fit[0].item()), behv[0].cpu().numpy().astype(np.float64), T


def _device_episode_closed(model, env, max_steps: int):
    """One noise-free episode on the closed-loop synthetic env as one launch of es_rollout_closedloop (sigma = 0)."""
    from ..engine import get_engine
    from ..core.policy import Policy
    eng = get_engine()
    sizes = model.layer_sizes()
    T = min(int(max_steps), env.T)
    _, rew_dev = env.device_arrays(eng)
    obs0, env_a, env_b = env.device_closed(eng)
    theta = eng.to_device(Policy.get_flat(model), torch.float32)
    mean = eng.to_device(np.ascontiguousarray(model._obmean, dtype=np.float64).reshape(-1), torch.float64)
    std = eng.to_device(np.ascontiguousarray(model._obstd, dtype=np.float64).reshape(-1), torch.float64)
    table = torch.zeros(theta.numel() + 1, dtype=torch.float32, device=eng.device)      # sigma = 0: the slice is irrelevant
    idx = torch.zeros(1, dtype=torch.int64, device=eng.device)
    fit = torch.zeros(2, dtype=torch.float64, device=eng.device)
    behv = torch.zeros(2, 3, dtype=torch.float32, device=eng.device)
    eng.rollout_closed(table, idx, theta, 0.0, sizes, mean, std, float(model.ob_clip), obs0, env_a, env_b, rew_dev[:T].contiguous(),
                       env.pos_scale, fit[0:1], fit[1:2], 1, behv[0:1].view(-1), behv[1:2].view(-1))
    return float(fit[0].item()), behv[0].cpu().numpy().astype(np.float64), T


def run_model(model: torch.nn.Module, env, max_steps: int, rs: np.random.RandomState = None, render: bool = False,
              get_pos_fn: Callable = pybullet_gym_pos) -> Tuple[List[float], List[float], np.ndarray, int]:
    """(rewards, positions padded to max_steps triples, post-step observations, last loop index)."""
    fused = (getattr(env, 'is_synthetic_openloop', False) and hasattr(model, 'is_tanh_mlp') and model.is_tanh_mlp()
             and not render)
    if fused:
        total, pos, T = _device_episode(model, env, max_steps, rs)
        # the episode total is exact; it is reported as a one-element reward list so that
        # sum(rews) (training_result.py:28) reproduces it bit for bit
        rews = [total]
        behv = [float(pos[0]), float(pos[1]), float(pos[2])] * int(max_steps)
        return rews, behv, env.obs_stream[1:T + 1], T - 1

    behv, rews, obs = [], [], []
    with torch.no_grad():
        ob = env.reset()
        for step in range(max_steps):
            ob = torch.from_numpy(np.asarray(ob)).float()
            action = model(ob, rs=rs)
            ob, rew, done, _ = env.step(action.cpu().numpy() if torch.is_tensor(action) else np.asarray(action))
            rews += [rew]
            obs.append(ob)
            behv.extend(get_pos_fn(env.unwrapped))
            if render:
                env.render('human')
                time.sleep(1 / 60)
            if done:
                break
    behv += behv[-3:] * (max_steps - int(len(behv) / 3))
    return rews, behv, np.array(obs), step


def multi_agent_gym_runner(policies, env, max_steps: int, rs: np.random.RandomState = None, save_obs: bool = False,
                           render: bool = False):
    """gym_runner.py:70-110 drives a Unity ML-Agents environment (src/gym/unity.py); that simulator and its wrapper are
    outside this package's scope (DESIGN.md section 6)."""
    raise NotImplementedError('multi_agent_gym_runner needs the Unity ML-Agents wrapper (src.gym.unity), which is not part of '
                              'es_pytorch_b200: the device path covers single-agent rollouts on the synthetic env')
