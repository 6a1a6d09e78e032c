"""Several episodes per evaluation (obj.py's eps_per_policy) without a GPU: the oracle's restatement of obj.py's fit_fn against
the real reference's es.step (tests/golden/ref_episodes.npz, made by make_ref_episodes.py), and the host-side validation of
BatchedRollout."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import es_oracle as orc

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import episodes_oracle as eps_orc  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(__file__), 'golden', 'ref_episodes.npz')


def test_oracle_episodes_reproduce_the_real_reference_step():
    """Two generations of the reference's es.step with obj.py's fit_fn, eps_per_policy = 3 and ac_std = 0.01: the indices, the
    stream after each step (key, position, has_gauss, cached gaussian) and the rank weights are exact; fitness within 2e-6 (the
    bound of the single-episode action-noise case: the reference's float32 forward runs in torch, the oracle's in numpy), theta
    within 2e-6, the noiseless result (three noise-free episodes) to float32 rounding."""
    v = np.load(GOLDEN)
    obs_dim, act_dim, T, n_pairs = [int(x) for x in v['cfg']]
    E, ac_std = int(v['eps_per_policy']), float(v['ac_std'])
    assert E == 3
    dims = orc.layer_dims(obs_dim, tuple(int(h) for h in v['hidden']), act_dim)
    P = orc.n_params(dims)
    table = np.random.RandomState(int(v['table_seed'])).randn(int(v['table_len'])).astype(np.float32)
    env = orc.SyntheticEnvSpec(obs_dim, act_dim, T)
    flat, opt = v['theta0'].copy(), orc.AdamOracle(P, 0.01)
    rs = np.random.RandomState(int(v['seed']))
    stat = orc.ObStatOracle((obs_dim,), 1e-2)
    obmean, obstd = np.zeros(obs_dim), np.ones(obs_dim)
    for g in range(2):
        out = eps_orc.es_step(table, flat, opt, 0.02, dims, env, [rs], n_pairs, obmean, obstd, 5.0, T, 500, 0.005, E,
                              coins_per_eval=1, save_obs_chance=float(v['save_obs_chance']), batched=False, ac_std=ac_std)
        assert np.array_equal(out['inds'], v[f's{g}_inds'])
        st = rs.get_state()
        assert np.array_equal(st[1], v[f's{g}_rs_key']) and st[2] == int(v[f's{g}_rs_pos']), f'stream after step {g}'
        assert st[3] == int(v[f's{g}_rs_has_gauss']) and st[4] == float(v[f's{g}_rs_gauss'])
        fits = np.concatenate((out['pos'], out['neg'])).ravel()
        want = v[f's{g}_fits'].ravel()
        assert fits.shape == want.shape
        assert np.abs(fits - want).max() <= 2e-6
        assert np.array_equal(np.asarray(out['weights']).ravel(), v[f's{g}_w'].ravel())
        assert np.abs(flat - v[f's{g}_theta']).max() <= 2e-6
        assert abs(out['noiseless'][0] - float(v[f's{g}_noiseless'][0])) <= 1e-5
        assert np.array_equal(out['obstat'].sum, v[f's{g}_ob_sum']) and out['obstat'].count == float(v[f's{g}_ob_count'])
        stat.inc(out['obstat'].sum, out['obstat'].sumsq, out['obstat'].count)
        obmean, obstd = stat.mean, stat.std


def test_oracle_noise_free_episodes_equal_one_episode():
    """With ac_std == 0 the reference's per-step average of E equal float32 rewards is that reward: the restatement of obj.py's
    loop gives bit-identical results to the oracle's one-episode evaluation, for E = 1 and E = 5."""
    dims = orc.layer_dims(17, (64, 64), 6)
    P = orc.n_params(dims)
    rs = np.random.RandomState(3)
    table, theta = rs.randn(P + 5000).astype(np.float32), (rs.randn(P) * 0.1).astype(np.float32)
    env = orc.SyntheticEnvSpec(17, 6, 30)
    one = orc.es_test_params(table, theta, 0.02, dims, env, [11], 3, np.zeros(17), np.ones(17), 5.0, 30, coins_per_eval=1)
    for E in (1, 5):
        many = eps_orc.es_test_params(table, theta, 0.02, dims, env, [11], 3, np.zeros(17), np.ones(17), 5.0, 30, E, coins_per_eval=1)
        for a, b in zip(one[:3], many[:3]):
            assert np.array_equal(a, b)


def _env_and_policy(act_std=0.01):
    from es_pytorch_b200.core.policy import Policy
    from es_pytorch_b200.gym.synthetic_env import SyntheticEnv
    from es_pytorch_b200.nn.nn import FeedForward
    from es_pytorch_b200.nn.optimizers import Adam
    env = SyntheticEnv(17, 6, 20)
    net = FeedForward([64, 64], torch.nn.Tanh(), env, act_std)
    return env, Policy(net, 0.02, Adam(len(Policy.get_flat(net)), 0.01))


def test_batched_rollout_episode_count_is_clamped_like_obj_py():
    from es_pytorch_b200.gym.batched import BatchedRollout
    env, _ = _env_and_policy()
    assert BatchedRollout(env, 20).eps_per_policy == 1
    assert BatchedRollout(env, 20, eps_per_policy=0).eps_per_policy == 1          # max(1, eps_per_policy), obj.py:57
    assert BatchedRollout(env, 20, eps_per_policy=-4).eps_per_policy == 1
    assert BatchedRollout(env, 20, eps_per_policy=10).eps_per_policy == 10
    assert BatchedRollout(env, 20, eps_per_policy=10).n_obj == 1


def test_batched_rollout_rejects_episodes_with_an_archive():
    """nsra.py's fit_fn runs one episode: several episodes with a novelty objective have no reference counterpart."""
    from es_pytorch_b200.gym.batched import BatchedRollout
    env, _ = _env_and_policy()
    with pytest.raises(ValueError, match='archive'):
        BatchedRollout(env, 20, archive=np.zeros((4, 2)), eps_per_policy=3)
    assert BatchedRollout(env, 20, archive=np.zeros((4, 2)), eps_per_policy=1).n_obj == 2
    assert BatchedRollout(env, 20, archive=np.zeros((4, 2)), eps_per_policy=0).n_obj == 2


def test_episodes_keep_the_single_synchronisation_step():
    from es_pytorch_b200 import dist
    from es_pytorch_b200.core import es
    from es_pytorch_b200.gym.batched import BatchedRollout
    from es_pytorch_b200.utils import rankers as R
    env, policy = _env_and_policy()
    fit_fn = BatchedRollout(env, 20, coins_per_eval=1, save_obs_chance=0.3, eps_per_policy=3)
    assert es._can_fuse_step(dist.world(), policy, fit_fn, R.CenteredRanker())
    assert es._can_fuse_step(dist.world(), policy, fit_fn, R.SemiCenteredRanker())


def test_c_abi_declares_the_episodes_entry():
    """The new entry is declared next to es_rollout_openloop_noisy and bound with one more int (n_episodes) before mode."""
    from es_pytorch_b200 import _lib
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(__file__)), 'include', 'es_b200.h')).read()
    assert 'int es_rollout_openloop_episodes(' in hdr
    noisy, eps = _lib.SIGNATURES['es_rollout_openloop_noisy'][1], _lib.SIGNATURES['es_rollout_openloop_episodes'][1]
    assert eps == noisy[:-2] + [_lib.C.c_int] + noisy[-2:]
