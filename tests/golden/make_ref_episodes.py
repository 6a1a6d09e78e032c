"""Generates tests/golden/ref_episodes.npz by running the REAL reference (/root/reference, build container only) through its own
``es.step`` with obj.py's fit_fn shape (obj.py:53-61): the save_obs coin, then ``max(1, eps_per_policy)`` episodes of
``run_model`` drawing their action noise from the same stream, the per-step rewards added into a float64 array of length
``max_steps`` and divided by the episode count; behaviour, observations and steps are the last episode's.

Two generations with ``eps_per_policy = 3`` and ``ac_std = 0.01`` on the synthetic env record, per generation: the noise
indices, the fitnesses, the final stream state (key, position, has_gauss, cached gaussian), the rank weights, theta and the
noiseless result of es.py:48 (the same fit_fn with ``use_ac_noise=False``).

Same inert stand-ins for the absent third-party imports as make_ref_pipeline.py.  Nothing from /root/reference is copied: it is
imported and executed.

    python tests/golden/make_ref_episodes.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE)
from make_ref_pipeline import REF, install_stand_ins  # noqa: E402
from make_ref_step import Cfg, QuietReporter  # noqa: E402


def main():
    comm = install_stand_ins()
    sys.path.insert(0, REF)
    sys.path.insert(0, ROOT)
    import torch
    from src.core import es
    from src.core.noisetable import NoiseTable
    from src.core.policy import Policy
    from src.gym import gym_runner
    from src.gym.training_result import RewardResult
    from src.nn.nn import FeedForward
    from src.nn.optimizers import Adam
    from src.utils.rankers import CenteredRanker
    from es_pytorch_b200.gym.synthetic_env import SyntheticEnv        # the synthetic env is this repo's (SURVEY 8d), numpy only here

    obs_dim, act_dim, hidden, T, n_pairs = 17, 6, [64, 64], 40, 6
    eps_per_policy, ac_std, save_obs_chance = 3, 0.01, 0.3
    env = SyntheticEnv(obs_dim, act_dim, T)
    torch.manual_seed(2)
    net = FeedForward(list(hidden), torch.nn.Tanh(), env, ac_std, 5)
    policy = Policy(net, 0.02, Adam(len(Policy.get_flat(net)), 0.01))
    P = len(policy)
    theta0 = (np.random.RandomState(6).randn(P) * 0.1).astype(np.float32)
    policy.flat_params = theta0.copy()
    table = np.random.RandomState(5).randn(200_003).astype(np.float32)
    nt = NoiseTable(P, table)
    rs = np.random.RandomState(9000)
    cfg = Cfg(general=Cfg(policies_per_gen=2 * n_pairs, batch_size=500, eps_per_policy=eps_per_policy),
              policy=Cfg(l2coeff=0.005, save_obs_chance=save_obs_chance), env=Cfg(max_steps=T))

    def r_fn(model, use_ac_noise=True):                         # obj.py:53-61's shape
        save_obs = rs.random() < cfg.policy.save_obs_chance
        rews = np.zeros(cfg.env.max_steps)
        for _ in range(max(1, cfg.general.eps_per_policy)):
            rew, behv, obs, steps = gym_runner.run_model(model, env, cfg.env.max_steps, rs if use_ac_noise else None)
            rews[:len(rew)] += np.array(rew)
        rews /= max(1, cfg.general.eps_per_policy)
        return RewardResult(rews.tolist(), behv, obs if save_obs else np.array([np.zeros(env.observation_space.shape)]), steps)

    out = dict(theta0=theta0, table_seed=np.array(5), table_len=np.array(len(table)), cfg=np.array([obs_dim, act_dim, T, n_pairs]),
               hidden=np.array(hidden), save_obs_chance=np.array(save_obs_chance), seed=np.array(9000),
               eps_per_policy=np.array(eps_per_policy), ac_std=np.array(ac_std))
    ranker = CenteredRanker()
    for g in range(2):
        tr, gen_obstat = es.step(cfg, comm, policy, nt, env, r_fn, rs, ranker, QuietReporter())
        policy.update_obstat(gen_obstat)
        st = rs.get_state()
        fits = np.asarray(ranker.fits)
        out[f's{g}_theta'], out[f's{g}_noiseless'] = policy.flat_params.copy(), np.array(tr.result)
        out[f's{g}_rs_key'], out[f's{g}_rs_pos'] = st[1].copy(), np.array(st[2])
        out[f's{g}_rs_has_gauss'], out[f's{g}_rs_gauss'] = np.array(st[3]), np.array(st[4])
        out[f's{g}_fits'], out[f's{g}_inds'] = fits, np.asarray(ranker.noise_inds)
        out[f's{g}_w'] = np.asarray(ranker.ranked_fits)
        out[f's{g}_ob_sum'], out[f's{g}_ob_count'] = gen_obstat.sum.copy(), np.array(gen_obstat.count)
    np.savez_compressed(os.path.join(HERE, 'ref_episodes.npz'), **out)
    print('ref_episodes.npz', len(out), 'arrays')


if __name__ == '__main__':
    main()
