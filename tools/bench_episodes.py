"""Timing of generations with several episodes per evaluation (obj.py's eps_per_policy) on the device, for the networks of the
shipped configs that use action noise, at their population size and episode length:

    config       network (synthetic shape)          pairs K   T
    obj          HalfCheetah 17-256-256-256-6       320       1 000
    simple_conf  Hopper 15-256-256-3                2 400     1 000
    flagrun      Ant 28-128-256-256-128-8           600       500

For E in {1, 10} and each of ES_ROLLOUT_F32 / TC / TC3: a DeviceGeneration with ac_std = 0.01 and eps_per_policy = E (8 virtual
ranks, one save_obs coin per evaluation), one warm-up generation, then --reps generations timed with CUDA events: the draw
(es_draw_noisy: indices, coins and E * T * act gaussians per evaluation), the rollout (es_rollout_openloop_episodes) and the
whole generation (host clock around run() + a synchronise).  The draw path (jump-ahead or sequential kernel) is the choice
mt_gauss.cu makes for the stream length, restated here.  For comparison, one es.step of the obj config through the
call-by-call route an opaque obj.py-style r_fn takes (2 K E single-policy launches, each with its own host-side rs.randn).
Writes <out>/bench_episodes.json with the GPU's name and power limit; needs a GPU.

    python tools/bench_episodes.py --out DIR [--reps 3] [--configs obj,simple_conf,flagrun] [--no-call-by-call]
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tools.bench_wide import gpu_info  # noqa: E402

CONFIGS = {
    'obj': dict(sizes=[17, 256, 256, 256, 6], K=320, T=1000),
    'simple_conf': dict(sizes=[15, 256, 256, 3], K=2400, T=1000),
    'flagrun': dict(sizes=[28, 128, 256, 256, 128, 8], K=600, T=500),
}
STREAMS = 8
EPISODES = (1, 10)
MT_NW = 624


def draw_path(n_per_stream: int, normals: int, coins: int = 1) -> dict:
    """es_draw_noisy's choice (mt_gauss.cu): the words a stream may need (mean + 12 sigma of the polar method's attempts) in
    MT19937 blocks; >= 2 048 blocks take the jump-ahead path unless the stream needs 2^20 blocks or more (654 M words)."""
    p_acc, n_acc = math.pi / 4, (normals + 1) / 2
    att_mean, att_sd = n_acc / p_acc, math.sqrt(n_acc * (1 - p_acc)) / p_acc
    evals = 2.0 * n_per_stream
    words = 624 + n_per_stream * (8 + 4 * coins) + 4 * (evals * att_mean + 12 * math.sqrt(evals) * att_sd + 64) + 2 * 5888 + 16 * MT_NW
    blocks = int(words / MT_NW) + 1
    path = 'jump-ahead' if 2048 <= blocks < (1 << 20) else 'sequential'
    return dict(blocks_per_stream=blocks, path=path)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--configs', default=','.join(CONFIGS))
    ap.add_argument('--no-call-by-call', action='store_true')
    args = ap.parse_args()
    import numpy as np
    import torch
    from es_pytorch_b200 import _lib
    from es_pytorch_b200.engine import get_engine
    from es_pytorch_b200.generation import DeviceGeneration
    from es_pytorch_b200.gym.synthetic_env import SyntheticEnv
    from es_pytorch_b200.nn.optimizers import Adam
    if not torch.cuda.is_available():
        sys.exit('bench_episodes.py needs a CUDA device')
    eng = get_engine(0)
    modes = {'f32': _lib.ES_ROLLOUT_F32, 'tc': _lib.ES_ROLLOUT_TC, 'tc3': _lib.ES_ROLLOUT_TC3}
    g = torch.Generator(device=eng.device).manual_seed(2024)
    table = torch.randn(250_000_000, generator=g, device=eng.device, dtype=torch.float32)
    result = dict(gpu=gpu_info(), table_floats=int(table.numel()), reps=args.reps, streams=STREAMS, ac_std=0.01, configs={})

    def ev_ms(pairs):
        return sum(a.elapsed_time(b) for a, b in pairs) / len(pairs)

    for name in args.configs.split(','):
        c = CONFIGS[name]
        sizes, K, T = c['sizes'], c['K'], c['T']
        P = sum(i * o + o for i, o in zip(sizes[:-1], sizes[1:]))
        env = SyntheticEnv(sizes[0], sizes[-1], max_episode_steps=T)
        rec = dict(sizes=sizes, K=K, T=T, P=P, episodes={})
        for E in EPISODES:
            normals = E * T * sizes[-1]
            er = dict(normals_per_eval=normals, noise_bytes=2 * K * normals * 4, draw=draw_path(K // STREAMS, normals), modes={})
            for mname, m in modes.items():
                theta = eng.to_device((np.random.RandomState(7).randn(P) * 0.1).astype(np.float32))
                gen = DeviceGeneration(table, theta, sizes, eng.to_device(env.obs_stream), eng.to_device(env.rew_vec),
                                       [np.random.RandomState(1000 + r) for r in range(STREAMS)], 0.02, 0.005, Adam(P, 0.01),
                                       coins_per_eval=1, save_obs_chance=0.01, rollout_mode=m, engine=eng, ac_std=0.01,
                                       eps_per_policy=E)
                gen.run(K // STREAMS)                                        # warm-up (scratch, shadows, module load)
                eng.sync()
                gen.enable_timers(True)
                t0 = time.perf_counter()
                for _ in range(args.reps):
                    gen.run(K // STREAMS)
                eng.sync()
                wall = (time.perf_counter() - t0) * 1e3 / args.reps
                er['modes'][mname] = dict(draw_ms=ev_ms(gen.timers['draw_indices']), rollout_ms=ev_ms(gen.timers['rollout']),
                                          generation_ms=wall)
                del gen
                torch.cuda.empty_cache()
            rec['episodes'][E] = er
            print(name, f'E={E}', er['draw'], json.dumps({k: {kk: round(vv, 3) for kk, vv in v.items()}
                                                          for k, v in er['modes'].items()}), flush=True)
        for mname in modes:
            e1, e10 = rec['episodes'][1]['modes'][mname], rec['episodes'][10]['modes'][mname]
            rec.setdefault('ratio_e10_over_e1', {})[mname] = {k: e10[k] / e1[k] for k in e1}
        result['configs'][name] = rec
    if not args.no_call_by_call and 'obj' in args.configs.split(','):
        result['call_by_call'] = call_by_call(eng, args, np, torch)
    result['gpu_after'] = gpu_info()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, 'bench_episodes.json'), 'w') as f:
        json.dump(result, f, indent=1)
    print(json.dumps(dict(gpu=result['gpu'], call_by_call=result.get('call_by_call'),
                          configs={k: {E: {m: round(v['episodes'][E]['modes'][m]['generation_ms'], 2) for m in modes}
                                       for E in EPISODES} for k, v in result['configs'].items()})))


def call_by_call(eng, args, np, torch):
    """One es.step of the obj config with an opaque obj.py-style r_fn (E = 10): the reference's per-perturbation loop, each
    episode one single-policy launch with its host-side rs.randn(T * act); against the same step with BatchedRollout."""
    from es_pytorch_b200 import dist
    from es_pytorch_b200.core import es
    from es_pytorch_b200.core.noisetable import NoiseTable
    from es_pytorch_b200.core.policy import Policy
    from es_pytorch_b200.gym import gym_runner
    from es_pytorch_b200.gym.batched import BatchedRollout
    from es_pytorch_b200.gym.synthetic_env import SyntheticEnv
    from es_pytorch_b200.gym.training_result import RewardResult
    from es_pytorch_b200.nn.nn import FeedForward
    from es_pytorch_b200.nn.optimizers import Adam
    from es_pytorch_b200.utils.rankers import CenteredRanker
    from es_pytorch_b200.utils.reporters import Reporter
    c, E = CONFIGS['obj'], 10
    sizes, K, T = c['sizes'], c['K'], c['T']

    class Cfg(dict):
        __getattr__ = dict.__getitem__

    cfg = Cfg(general=Cfg(policies_per_gen=2 * K, batch_size=500), policy=Cfg(l2coeff=0.005))
    env = SyntheticEnv(sizes[0], sizes[-1], max_episode_steps=T)
    out = dict(config='obj', K=K, T=T, eps_per_policy=E)
    for route in ('batched', 'call_by_call'):
        torch.manual_seed(0)
        net = FeedForward(sizes[1:-1], torch.nn.Tanh(), env, 0.01, 5)
        P = len(Policy.get_flat(net))
        policy = Policy(net, 0.02, Adam(P, 0.01))
        nt = NoiseTable(P, np.random.RandomState(5).randn(20_000_000).astype(np.float32))
        rs = np.random.RandomState(11)
        if route == 'batched':
            fit_fn = BatchedRollout(env, T, coins_per_eval=1, save_obs_chance=0.01, eps_per_policy=E)
        else:
            def fit_fn(model, use_ac_noise=True):                  # obj.py:53-61
                save_obs = rs.random() < 0.01
                rews = np.zeros(T)
                for _ in range(E):
                    rew, behv, obs, steps = gym_runner.run_model(model, env, T, rs if use_ac_noise else None)
                    rews[:len(rew)] += np.array(rew)
                rews /= E
                return RewardResult(rews.tolist(), behv, obs if save_obs else np.array([np.zeros(env.observation_space.shape)]), steps)
        if route == 'batched':
            es.step(cfg, dist.world(), policy, nt, env, fit_fn, rs, CenteredRanker(), Reporter())  # warm-up
            eng.sync()
        t0 = time.perf_counter()
        es.step(cfg, dist.world(), policy, nt, env, fit_fn, rs, CenteredRanker(), Reporter())
        eng.sync()
        out[f'{route}_step_ms'] = (time.perf_counter() - t0) * 1e3
        print(route, round(out[f'{route}_step_ms'], 1), 'ms per es.step', flush=True)
    out['speedup'] = out['call_by_call_step_ms'] / out['batched_step_ms']
    return out


if __name__ == '__main__':
    main()
