"""The boundary, proven by running it: a training script that touches ONLY the reference's import surface (``src.*``,
``mpi4py.MPI.COMM_WORLD``, ``gym.make``, ``utils.load_config``; tests/drivers/es_script.py, in the two shapes of the
reference's simple_example.py:45-58 and obj.py:67-83) is executed as a separate process against the compat shims -- on one
GPU, and under torchrun on two -- with the settings the shipped configs use (ac_std = 0.01, save_obs_chance > 0), and every
generation is replayed by the CPU oracle: indices and the ranks' RandomState streams bit-exact, fitness to float32
tolerance, theta within 1e-5 after three generations of Adam.

(The reference's own scripts are not part of this repository; tests/test_host_logic.py checks that their import statements,
recorded in tests/golden/ref_script_surface.json, resolve against the same shims.)"""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import es_oracle as orc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COMPAT = os.path.join(ROOT, 'es_pytorch_b200', 'compat')
DRIVER = os.path.join(ROOT, 'tests', 'drivers', 'es_script.py')


def _config(n_ranks, mode):
    cfg = {
        'env': {'name': 'HalfCheetahBulletEnv-v0', 'max_steps': 1000},
        'noise': {'tbl_size': 400_000, 'std': 0.02, 'std_limit': 0.002, 'std_decay': 0.9},
        'policy': {'layer_sizes': [64, 64], 'ac_std': 0.01, 'ac_std_decay': 0.5, 'l2coeff': 0.005, 'lr': 0.01, 'lr_limit': 0.001,
                   'lr_decay': 0.8, 'ob_clip': 5, 'save_obs_chance': 0.3},
        'general': {'name': 'drv', 'gens': 3, 'policies_per_gen': 2 * 3 * n_ranks, 'batch_size': 500,
                    'seed': [4100 + 7 * r for r in range(n_ranks)]},
    }
    if mode == 'explicit':                                   # simple_conf.json's schema: no decays, no env.max_steps
        del cfg['env']['max_steps']
        for k in ('std_limit', 'std_decay'):
            del cfg['noise'][k]
        for k in ('ac_std_decay', 'lr_limit', 'lr_decay'):
            del cfg['policy'][k]
    return cfg


def _run_script(tmp_path, mode, n_ranks):
    cfg = _config(n_ranks, mode)
    cfg_file = tmp_path / 'cfg.json'
    cfg_file.write_text(json.dumps(cfg))
    out_prefix = str(tmp_path / 'run')
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + COMPAT)
    if n_ranks == 1:
        cmd = [sys.executable, DRIVER, mode, str(cfg_file), out_prefix]
    else:
        with socket.socket() as sk:
            sk.bind(('127.0.0.1', 0))
            port = sk.getsockname()[1]
        cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', f'--nproc-per-node={n_ranks}', '--master-addr',
               '127.0.0.1', '--master-port', str(port), DRIVER, mode, str(cfg_file), out_prefix]
    out = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=900)
    assert out.returncode == 0 and 'SCRIPT_DONE' in out.stdout, (out.stdout + out.stderr)[-4000:]
    return cfg, [np.load(f'{out_prefix}.rank{r}.npz') for r in range(n_ranks)]


def _replay_with_the_oracle(cfg, logs, mode):
    n_ranks = len(logs)
    obs_dim, act_dim, T = 17, 6, 1000                        # the synthetic env gym.make returns for a HalfCheetah task
    spec = orc.SyntheticEnvSpec(obs_dim, act_dim, T)
    dims = orc.layer_dims(obs_dim, tuple(cfg['policy']['layer_sizes']), act_dim)
    P = orc.n_params(dims)
    seeds = cfg['general']['seed']
    table = np.random.RandomState(int(seeds[0])).randn(cfg['noise']['tbl_size']).astype(np.float32)   # create_shared(seed=seeds)
    flat = logs[0]['theta0'].copy()
    assert len(flat) == P and all(np.array_equal(l['theta0'], flat) for l in logs), 'identical initial parameters on every rank'
    states = [np.random.RandomState(int(s)) for s in seeds]
    opt = orc.AdamOracle(P, cfg['policy']['lr'])
    stat = orc.ObStatOracle((obs_dim,), 1e-2)
    obmean, obstd = np.zeros(obs_dim), np.ones(obs_dim)
    std, ac_std = cfg['noise']['std'], cfg['policy']['ac_std']
    n_per_rank = cfg['general']['policies_per_gen'] // n_ranks // 2
    for g in range(cfg['general']['gens']):
        kw = dict(coins_per_eval=1, save_obs_chance=cfg['policy']['save_obs_chance'], batched=False, ac_std=ac_std)
        if mode == 'explicit':
            out = orc.generation(table, flat, opt, std, dims, spec, [None] * n_ranks, n_per_rank, obmean, obstd, 5.0, T, 500,
                                 cfg['policy']['l2coeff'], rank_states=states, **kw)
        else:
            out = orc.es_step(table, flat, opt, std, dims, spec, states, n_per_rank, obmean, obstd, 5.0, T, 500,
                              cfg['policy']['l2coeff'], **kw)
        stat.inc(out['obstat'].sum, out['obstat'].sumsq, out['obstat'].count)
        obmean, obstd = stat.mean, stat.std
        for r, log in enumerate(logs):
            assert np.array_equal(log[f'g{g}_inds'], out['inds']), f'generation {g}: noise indices (all ranks, rank-major)'
            fits = np.concatenate((out['pos'], out['neg']))
            assert np.abs(log[f'g{g}_fits'] - fits).max() <= 1e-4, np.abs(log[f'g{g}_fits'] - fits).max()
            st = states[r].get_state()
            assert np.array_equal(log[f'g{g}_rs_key'], st[1]) and int(log[f'g{g}_rs_pos']) == st[2], f'generation {g}: stream of rank {r}'
            assert int(log[f'g{g}_rs_has_gauss']) == st[3] and abs(float(log[f'g{g}_rs_gauss']) - st[4]) <= 4 * np.spacing(abs(st[4]))
            assert float(log[f'g{g}_ob_count']) == stat.count
            assert np.abs(log[f'g{g}_theta'] - flat).max() <= 1e-5, (g, np.abs(log[f'g{g}_theta'] - flat).max())
            if mode == 'step':
                assert abs(float(log[f'g{g}_noiseless'][0]) - out['noiseless'][0]) <= 1e-4
        if mode == 'step':                                   # obj.py:81-83
            ac_std = ac_std * cfg['policy']['ac_std_decay']
            std = max(std * cfg['noise']['std_decay'], cfg['noise']['std_limit'])
            opt.lr = max(opt.lr * cfg['policy']['lr_decay'], cfg['policy']['lr_limit'])


@pytest.mark.parametrize('mode', ['explicit', 'step'])
def test_reference_shaped_script_runs_on_one_gpu(tmp_path, mode):
    cfg, logs = _run_script(tmp_path, mode, 1)
    _replay_with_the_oracle(cfg, logs, mode)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs 2 GPUs')
@pytest.mark.parametrize('mode', ['explicit', 'step'])
def test_reference_shaped_script_runs_under_torchrun_on_two_gpus(tmp_path, mode):
    cfg, logs = _run_script(tmp_path, mode, 2)
    _replay_with_the_oracle(cfg, logs, mode)
