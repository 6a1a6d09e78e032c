"""Timing of the open-loop rollout in ES_ROLLOUT_F32, ES_ROLLOUT_TC and ES_ROLLOUT_TC3 on the networks of the four shipped
training configs, at their population size and episode length, in one process (bench.py measures the 376-64-64-17
headline only):

    config       network (synthetic shape)          pairs K   T
    simple_conf  Hopper 15-256-256-3                2 400     1 000
    nsra         Hopper 15-256-256-3, 2 objectives  4 800     2 000
    obj          HalfCheetah 17-256-256-256-6       320       1 000
    flagrun      Ant 28-128-256-256-128-8           600       500

Per shape: one warm-up launch per mode, then CUDA events over --reps launches of the rollout alone (250 M-float noise
table: the slices the rollout reads are spread over 1 GB, so they cannot stay in L2), and one whole DeviceGeneration.run
(draws, rollout, ranking, gradient, Adam) with ac_std = 0.01 per mode after a warm-up generation.  TC3 against F32 through
generation.parity_report on the same indices.  Writes <out>/bench_wide.json; needs a GPU.

    python tools/bench_wide.py --out DIR [--reps 5] [--configs simple_conf,nsra,obj,flagrun]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FP16_DENSE_PEAK = 2250e12          # FLOP/s, dense FP16 / BF16 tensor rate of one B200 (data sheet, 1000 W card)
HBM_PEAK = 7.7e12                  # bytes/s

CONFIGS = {
    'simple_conf': dict(sizes=[15, 256, 256, 3], K=2400, T=1000, n_obj=1),
    'nsra': dict(sizes=[15, 256, 256, 3], K=4800, T=2000, n_obj=2),
    'obj': dict(sizes=[17, 256, 256, 256, 6], K=320, T=1000, n_obj=1),
    'flagrun': dict(sizes=[28, 128, 256, 256, 128, 8], K=600, T=500, n_obj=1),
}
STREAMS = 8


def gpu_info():
    q = 'name,power.limit,clocks.max.sm'
    try:
        out = subprocess.run(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader'], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [x.strip() for x in out.split(',')]
        return dict(name=name, power_limit=plim, sm_clock_max=clk)
    except Exception as e:                                   # noqa: BLE001
        return dict(error=str(e))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--configs', default=','.join(CONFIGS))
    args = ap.parse_args()
    import numpy as np
    import torch
    from es_pytorch_b200 import _lib
    from es_pytorch_b200.engine import get_engine
    from es_pytorch_b200.generation import DeviceGeneration, parity_report
    from es_pytorch_b200.gym.synthetic_env import SyntheticEnv
    from es_pytorch_b200.nn.optimizers import Adam
    if not torch.cuda.is_available():
        sys.exit('bench_wide.py needs a CUDA device')
    eng = get_engine(0)
    modes = {'f32': _lib.ES_ROLLOUT_F32, 'tc': _lib.ES_ROLLOUT_TC, 'tc3': _lib.ES_ROLLOUT_TC3}
    g = torch.Generator(device=eng.device).manual_seed(2024)
    table = torch.randn(250_000_000, generator=g, device=eng.device, dtype=torch.float32)
    result = dict(gpu=gpu_info(), table_floats=int(table.numel()), reps=args.reps, streams=STREAMS, configs={})

    def timed(fn, reps):
        fn()                                                                 # warm-up
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    for name in args.configs.split(','):
        c = CONFIGS[name]
        sizes, K, T = c['sizes'], c['K'], c['T']
        P = sum(i * o + o for i, o in zip(sizes[:-1], sizes[1:]))
        macs = sum(i * o for i, o in zip(sizes[:-1], sizes[1:]))
        flop = 2.0 * macs * 2 * K * T                                        # algorithmic work of one rollout launch
        env = SyntheticEnv(sizes[0], sizes[-1], max_episode_steps=T)
        theta = eng.to_device((np.random.RandomState(7).randn(P) * 0.1).astype(np.float32))
        archive = None
        if c['n_obj'] == 2:                                                  # nsra: novelty against a behaviour archive
            archive = eng.to_device(np.random.RandomState(3).randn(16, 2) * 0.5)
        gen = DeviceGeneration(table, theta, sizes, eng.to_device(env.obs_stream), eng.to_device(env.rew_vec),
                               [np.random.RandomState(1000 + r) for r in range(STREAMS)], 0.02, 0.005, Adam(P, 0.01),
                               coins_per_eval=1, archive=archive, engine=eng, ac_std=0.01)
        gen.evaluate(K // STREAMS)                                           # draws the indices the rollouts below use
        eng.sync()
        rec = dict(sizes=sizes, K=K, T=T, n_obj=c['n_obj'], P=P, algorithmic_tflop=flop / 1e12, modes={})
        fit = torch.zeros(2, K, c['n_obj'], dtype=torch.float64, device=eng.device)
        behv = torch.zeros(2, K, 3, dtype=torch.float32, device=eng.device)
        for mname, m in modes.items():
            def roll():
                eng.rollout(gen.table, gen.idx, gen.theta, gen.sigma, sizes, gen.obsn, gen.rew_vec, gen.pos_scale,
                            fit[0].view(-1), fit[1].view(-1), c['n_obj'], behv[0], behv[1], m)
            ms = timed(roll, args.reps)
            issued = flop * (3 if mname == 'tc3' else 1)
            t_min_compute = issued / FP16_DENSE_PEAK
            t_min_bytes = (2 * K * P * 4 + P * 4) / HBM_PEAK                  # every pair's noise slice + theta, once
            bound = 'fp16 dense tensor compute' if t_min_compute >= t_min_bytes else 'HBM bandwidth'
            r = dict(ms=ms, algorithmic_tflops=flop / (ms * 1e-3) / 1e12, issued_tflops=issued / (ms * 1e-3) / 1e12,
                     share_of_peak=max(t_min_compute, t_min_bytes) / (ms * 1e-3), bound=bound)
            if mname == 'tc3':
                r['issued_work_note'] = 'three MMAs per product: issued work = 3x the algorithmic work'
            rec['modes'][mname] = r
        # one whole generation per mode (ac_std = 0.01: es_draw_noisy + the noisy rollout)
        for mname, m in modes.items():
            gen.rollout_mode = m
            rec['modes'][mname]['generation_ms'] = timed(lambda: gen.run(K // STREAMS), max(1, args.reps // 2))
        gen.rollout_mode = _lib.ES_ROLLOUT_TC3
        gen.evaluate(K // STREAMS)
        rec['parity_tc3_vs_f32'] = parity_report(gen, _lib.ES_ROLLOUT_TC3, _lib.ES_ROLLOUT_F32)
        rec['parity_tc_vs_f32'] = parity_report(gen, _lib.ES_ROLLOUT_TC, _lib.ES_ROLLOUT_F32)
        for mname in ('tc', 'tc3'):
            rec['modes'][mname]['speedup_vs_f32'] = rec['modes']['f32']['ms'] / rec['modes'][mname]['ms']
        result['configs'][name] = rec
        print(name, json.dumps({k: {kk: round(vv, 4) if isinstance(vv, float) else vv for kk, vv in v.items()}
                                for k, v in rec['modes'].items()}), flush=True)
        del gen
        torch.cuda.empty_cache()
    result['gpu_after'] = gpu_info()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, 'bench_wide.json'), 'w') as f:
        json.dump(result, f, indent=1)
    print(json.dumps(dict(gpu=result['gpu'], configs={k: {m: round(v['modes'][m]['ms'], 3) for m in modes}
                                                       for k, v in result['configs'].items()})))


if __name__ == '__main__':
    main()
