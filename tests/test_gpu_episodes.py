"""Several episodes per evaluation (obj.py's eps_per_policy) on the device: es_rollout_openloop_episodes in the four open-loop
rollout kernels and both tensor-core precisions, DeviceGeneration's draw of E * T * act gaussians per evaluation, and es.step
with BatchedRollout(eps_per_policy=E), against the oracle's restatement of obj.py's fit_fn and the real reference's es.step
(tests/golden/ref_episodes.npz)."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import es_oracle as orc

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import episodes_oracle as eps_orc  # noqa: E402

pytestmark = pytest.mark.gpu

F32 = np.float32
SMALL, HUM, HOPPER, ANT = [17, 64, 64, 6], [376, 64, 64, 17], [15, 256, 256, 3], [28, 128, 256, 256, 128, 8]
POS_SCALE = 0.05


def dev(eng, a):
    return eng.to_device(np.ascontiguousarray(a))


def _inputs(sizes, T, n, E, seed, sigma=0.02):
    rs = np.random.RandomState(seed)
    P = sum(i * o + o for i, o in zip(sizes[:-1], sizes[1:]))
    L = P + 200_000
    c = dict(sizes=sizes, T=T, n=n, E=E, P=P, sigma=sigma, table=rs.randn(L).astype(F32), theta=(rs.randn(P) * 0.1).astype(F32),
             idx=rs.randint(0, L - P - 1, size=n).astype(np.int64),
             obsn=np.clip(rs.randn(T, sizes[0]), -5, 5).astype(F32), rew=rs.randn(T, sizes[-1]).astype(F32))
    c['noise'] = (rs.randn(n, 2, E, T, sizes[-1]) * 0.01).astype(F32)
    return c


def _run(eng, c, mode, E=None, noise=True, noisy_entry=False):
    """fitness [2, n] and final positions [2, n, 3] of one launch: the episodes entry (E episodes) or, with ``noisy_entry``,
    es_rollout_openloop_noisy (the noise array must then hold one episode)"""
    n = c['n']
    fit = torch.full((2, n), -1.0, dtype=torch.float64, device=eng.device)
    b = torch.zeros(2, n, 3, dtype=torch.float32, device=eng.device)
    args = (dev(eng, c['table']), dev(eng, c['idx']), dev(eng, c['theta']), c['sigma'], c['sizes'], dev(eng, c['obsn']),
            dev(eng, c['rew']), POS_SCALE, fit[0], fit[1], 1, b[0], b[1])
    nz = dev(eng, c['noise']) if noise else None
    if noisy_entry:
        eng.rollout(*args, mode, act_noise=nz)
    else:
        eng.rollout_episodes(*args, mode, act_noise=nz, n_episodes=c['E'] if E is None else E)
    eng.sync()
    return fit.cpu().numpy(), b.cpu().numpy()


def _oracle(c, pairs):
    """obj.py's loop over the episodes of every evaluation in ``pairs``, with the given float32 noise rows: per step the float32
    reward of each episode's noisy action, rews[t] += r in float64, rews /= E, fitness = sum(rews); the position integrator of
    the last episode.  The forward pass is the oracle's float32 MLP."""
    sizes, P, T, E = c['sizes'], c['P'], c['T'], c['E']
    dims = list(zip(sizes[:-1], sizes[1:]))
    fit, pos = {}, {}
    for k in pairs:
        for s, sign in enumerate((1.0, -1.0)):
            layers = orc.unflatten(orc.pheno_params(c['theta'], c['sigma'], sign * c['table'][c['idx'][k]:c['idx'][k] + P]), dims)
            acts = orc.mlp_forward(layers, c['obsn']).astype(F32)
            rews = np.zeros(T)
            for e in range(E):
                a = (acts + c['noise'][k, s, e]).astype(F32)
                r = np.zeros(T, dtype=F32)
                for j in range(sizes[-1]):                         # float32 dot in index order
                    r = (r + (a[:, j] * c['rew'][:, j]).astype(F32)).astype(F32)
                rews += r.astype(np.float64)
            rews /= E
            fit[s, k] = float(sum(rews.tolist()))
            p = np.zeros(3, dtype=F32)
            for t in range(T):
                for j in range(3):
                    p[j] = F32(p[j] + F32(F32(POS_SCALE) * a[t, j % sizes[-1]]))
            pos[s, k] = p
    return fit, pos


# ---- 1. E = 1 is es_rollout_openloop_noisy ---------------------------------------------------------------------------------
@pytest.mark.parametrize('sizes', [SMALL, HUM, HOPPER])
@pytest.mark.parametrize('mode', [0, 1, 2])
def test_one_episode_is_the_noisy_entry(eng, sizes, mode):
    c = _inputs(sizes, 150, 20, 1, seed=sum(sizes) + mode)
    f1, b1 = _run(eng, c, mode)
    f0, b0 = _run(eng, c, mode, noisy_entry=True)
    assert np.array_equal(f1, f0) and np.array_equal(b1, b0)


# ---- 2. no noise: E episodes are one episode ---------------------------------------------------------------------------------
@pytest.mark.parametrize('sizes', [SMALL, HOPPER])
@pytest.mark.parametrize('mode', [0, 2])
def test_noise_free_episodes_collapse_to_one(eng, sizes, mode):
    c = _inputs(sizes, 129, 9, 5, seed=3 + mode)
    launches = eng.launches
    f5, b5 = _run(eng, c, mode, noise=False)
    n5 = eng.launches - launches
    launches = eng.launches
    f1, b1 = _run(eng, c, mode, E=1, noise=False)
    assert np.array_equal(f5, f1) and np.array_equal(b5, b1)
    assert n5 == eng.launches - launches                                 # the same launches: no E-fold work


def test_noise_free_generation_and_call_collapse_to_one(eng):
    """DeviceGeneration(eps_per_policy=5, ac_std=0) and BatchedRollout(eps_per_policy=5).__call__ with a noise-free policy give
    bit-identical results to one episode, and draw the same words."""
    from es_pytorch_b200.generation import DeviceGeneration
    from es_pytorch_b200.gym.batched import BatchedRollout
    from es_pytorch_b200.nn.optimizers import Adam
    sizes, T = SMALL, 40
    dims = orc.layer_dims(17, (64, 64), 6)
    P = orc.n_params(dims)
    rs = np.random.RandomState(21)
    table, theta = rs.randn(P + 50_000).astype(F32), (rs.randn(P) * 0.1).astype(F32)
    spec = orc.SyntheticEnvSpec(17, 6, T)
    out = []
    for E in (1, 5):
        streams = [np.random.RandomState(31), np.random.RandomState(32)]
        gen = DeviceGeneration(eng.to_device(table), eng.to_device(theta.copy()), sizes, eng.to_device(spec.obs_stream),
                               eng.to_device(spec.rew_vec), streams, 0.02, 0.005, Adam(P, 0.01), coins_per_eval=1, engine=eng,
                               eps_per_policy=E)
        fpos, fneg = gen.evaluate(6)
        eng.sync()
        out.append((fpos.cpu().numpy(), fneg.cpu().numpy(), gen.mt_state.cpu().numpy()))
    for a, b in zip(out[0], out[1]):
        assert np.array_equal(a, b)
    env, net, policy = _api_objects(sizes[1:-1], spec, theta)
    res = []
    for E in (1, 5):
        rs_call = np.random.RandomState(44)
        fit_fn = BatchedRollout(env, T, coins_per_eval=1, rank_streams=[rs_call], eps_per_policy=E)
        tr = fit_fn(policy.pheno(np.zeros(len(policy))))
        res.append((tr.result, tr.behaviour, rs_call.get_state()[1:3]))
    assert res[0][0] == res[1][0] and np.array_equal(res[0][1], res[1][1])
    assert np.array_equal(res[0][2][0], res[1][2][0]) and res[0][2][1] == res[1][2][1]


# ---- 3. kernel parity ----------------------------------------------------------------------------------------------------------
_PARITY = [(SMALL, 129, 1, 2), (SMALL, 1000, 5, 10), (SMALL, 129, 160, 10), (HUM, 1, 3, 10), (HUM, 129, 150, 2),
           (HOPPER, 129, 40, 2), (HOPPER, 1000, 6, 10), (ANT, 129, 3, 10), (ANT, 1000, 2, 2)]


@pytest.mark.parametrize('sizes,T,n,E', _PARITY)
def test_episodes_match_the_oracle_and_float32(eng, sizes, T, n, E):
    """F32 against obj.py's loop (fitness within 1e-5 of the episode's |reward| mass, the last episode's position within float32
    sums of T terms); TC3 and TC against F32 within the bounds of the single-episode tests for the same shape."""
    c = _inputs(sizes, T, n, E, seed=sum(sizes) + T + n + E)
    f32, b32 = _run(eng, c, 0)
    pairs = sorted({0, n // 2, n - 1})
    fit, pos = _oracle(c, pairs)
    mass = np.abs(c['rew']).sum() * 1.0
    for (s, k), want in fit.items():
        assert abs(f32[s, k] - want) <= 1e-5 * max(1.0, mass / 8), (s, k, f32[s, k], want)
        assert np.abs(b32[s, k] - pos[s, k]).max() <= 2e-6 * POS_SCALE * T + 1e-6
    f3, b3 = _run(eng, c, 2)
    assert np.abs(f3 - f32).max() <= 1e-5 * max(1.0, mass / 8), (np.abs(f3 - f32).max(), mass)
    assert np.abs(b3 - b32).max() <= 2e-6 * POS_SCALE * T + 1e-6
    ftc, btc = _run(eng, c, 1)
    spread = max(f32.std(), 1e-3 * np.sqrt(T))
    assert np.abs(ftc - f32).max() <= 0.02 * spread + 1e-3 * np.sqrt(T) * POS_SCALE
    assert np.sqrt(((ftc - f32) ** 2).mean()) <= 5e-3 * spread + 2e-4
    assert np.abs(btc - b32).max() <= 2e-3 * POS_SCALE * T + 1e-4


def test_episodes_general_float32_kernel(eng, monkeypatch):
    """the general float32 kernel (ES_F32_GENERAL=1; staged global weights for the wide shape) against the packed-FMA kernel"""
    for sizes in (SMALL, HOPPER):
        c = _inputs(sizes, 200, 90, 3, seed=5)
        fa, ba = _run(eng, c, 0)
        monkeypatch.setenv('ES_F32_GENERAL', '1')
        fb, bb = _run(eng, c, 0)
        monkeypatch.delenv('ES_F32_GENERAL')
        assert np.abs(fa - fb).max() <= 1e-5 * max(1.0, np.abs(c['rew']).sum() / 8)
        assert np.abs(ba - bb).max() <= 2e-6 * POS_SCALE * 200 + 1e-6


# ---- 4. a generation ---------------------------------------------------------------------------------------------------------
def _api_objects(hidden, spec, theta):
    from es_pytorch_b200.core.policy import Policy
    from es_pytorch_b200.gym.synthetic_env import SyntheticEnv
    from es_pytorch_b200.nn.nn import FeedForward
    from es_pytorch_b200.nn.optimizers import Adam
    env = SyntheticEnv(spec.obs_dim, spec.act_dim, spec.T)
    net = FeedForward(list(hidden), torch.nn.Tanh(), env, 0.0, 5)
    policy = Policy(net, 0.02, Adam(len(theta), 0.01))
    policy.flat_params[...] = theta
    policy.set_nn_params(policy.flat_params)
    return env, net, policy


@pytest.mark.parametrize('jump', ['0', '1'])
def test_generation_with_episodes_matches_the_oracle(eng, monkeypatch, jump):
    """DeviceGeneration(eps_per_policy=3, ac_std=0.01), 3 virtual ranks, one coin per evaluation: E * T * act gaussians per
    evaluation after its coin.  Indices, coin words and the final key / position / has_gauss exact, the cached gaussian to an
    ulp, fitness within the F32 bound, weights exact."""
    from es_pytorch_b200.generation import DeviceGeneration
    from es_pytorch_b200.nn.optimizers import Adam
    monkeypatch.setenv('ES_MT_JUMP', jump)
    if jump == '1':
        monkeypatch.setenv('ES_MT_JUMP_LB', '2')
    obs_dim, act_dim, T, n, E = 17, 5, 37, 4, 3                       # T * act odd: the gaussian cache crosses episodes
    dims = orc.layer_dims(obs_dim, (64, 64), act_dim)
    P = orc.n_params(dims)
    rs0 = np.random.RandomState(12)
    table, theta = rs0.randn(P + 150_000).astype(F32), (rs0.randn(P) * 0.1).astype(F32)
    spec = orc.SyntheticEnvSpec(obs_dim, act_dim, T)
    seeds = [400, 401, 402]
    streams, ref_streams = [np.random.RandomState(s) for s in seeds], [np.random.RandomState(s) for s in seeds]
    streams[1].randn(1); ref_streams[1].randn(1)
    gen = DeviceGeneration(eng.to_device(table), eng.to_device(theta.copy()), [obs_dim, 64, 64, act_dim], eng.to_device(spec.obs_stream),
                           eng.to_device(spec.rew_vec), streams, 0.02, 0.005, Adam(P, 0.01), coins_per_eval=1, save_obs_chance=0.3,
                           engine=eng, ac_std=0.01, eps_per_policy=E)
    fpos, fneg = gen.evaluate(n)
    eng.sync()
    assert gen.act_noise.shape == (3 * n, 2, E * T * act_dim)
    pos, neg, inds, _, stat = eps_orc.es_test_params(table, theta, 0.02, dims, spec, seeds, n, np.zeros(obs_dim), np.ones(obs_dim),
                                                     5.0, T, E, coins_per_eval=1, save_obs_chance=0.3, batched=False,
                                                     rank_states=ref_streams, ac_std=0.01)
    assert np.array_equal(gen.idx.cpu().numpy(), inds.astype(np.int64))
    mass = np.abs(spec.rew_vec).sum()
    assert np.abs(fpos.cpu().numpy() - pos).max() <= 1e-5 * max(1.0, mass / 8)
    assert np.abs(fneg.cpu().numpy() - neg).max() <= 1e-5 * max(1.0, mass / 8)
    assert float(gen.gen_count[0].item()) + 0.0 == stat.count
    # the coin words are those of numpy's rs.random() at the same stream positions
    cw = gen.extras.cpu().numpy().view(np.uint32).reshape(3, n, 2, 2)
    chk = [np.random.RandomState(s) for s in seeds]
    chk[1].randn(1)
    for r, rs in enumerate(chk):
        for k in range(n):
            rs.randint(0, len(table) - P)
            for sg in range(2):
                assert orc.words_to_double(int(cw[r, k, sg, 0]), int(cw[r, k, sg, 1])) == rs.random()
                rs.randn(E * T * act_dim)
    for a, b in zip(gen.rank_states(), ref_streams):
        sa, sb = a.get_state(), b.get_state()
        assert np.array_equal(sa[1], sb[1]) and sa[2] == sb[2] and sa[3] == sb[3]
        assert abs(sa[4] - sb[4]) <= np.spacing(abs(sb[4]))
    gen.update(fpos, fneg)
    w, _ = orc.centered_ranker(pos, neg)
    got = np.concatenate((fpos.cpu().numpy(), fneg.cpu().numpy())).ravel()
    gaps = np.diff(np.sort(got))
    if gaps.size and gaps.min() > 1e-4:                                  # no near-tie the fitness tolerance could swap
        assert np.array_equal(gen.weights.cpu().numpy(), np.asarray(w).ravel())


# ---- 5. es.step ---------------------------------------------------------------------------------------------------------------
class _Cfg(dict):
    __getattr__ = dict.__getitem__


@pytest.mark.parametrize('mode', [0, 2])
def test_api_step_with_episodes_matches_the_real_reference(eng, mode):
    """es.step with BatchedRollout(eps_per_policy=3) for the two generations of ref_episodes.npz (the real reference's es.step with
    obj.py's fit_fn), and the oracle's es_step alongside: indices, the caller's stream (key, position, has_gauss) exact, the
    cached gaussian to 2 ulp, fitness and theta to float32 tolerance, rank weights equal, the noiseless result."""
    from es_pytorch_b200 import dist
    from es_pytorch_b200.core import es
    from es_pytorch_b200.core.noisetable import NoiseTable
    from es_pytorch_b200.gym.batched import BatchedRollout
    from es_pytorch_b200.utils.rankers import CenteredRanker
    from es_pytorch_b200.utils.reporters import Reporter
    v = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'ref_episodes.npz'))
    obs_dim, act_dim, T, n_pairs = [int(x) for x in v['cfg']]
    E, ac_std = int(v['eps_per_policy']), float(v['ac_std'])
    hidden = tuple(int(h) for h in v['hidden'])
    dims = orc.layer_dims(obs_dim, hidden, act_dim)
    table = np.random.RandomState(int(v['table_seed'])).randn(int(v['table_len'])).astype(F32)
    spec = orc.SyntheticEnvSpec(obs_dim, act_dim, T)
    env, net, policy = _api_objects(hidden, spec, v['theta0'].copy())
    net._action_std = ac_std
    nt = NoiseTable(len(policy), table)
    rs, ref_rs = np.random.RandomState(int(v['seed'])), np.random.RandomState(int(v['seed']))
    fit_fn = BatchedRollout(env, T, coins_per_eval=1, save_obs_chance=float(v['save_obs_chance']), rollout_mode=mode,
                            eps_per_policy=E)
    cfg = _Cfg(general=_Cfg(policies_per_gen=2 * n_pairs, batch_size=500), policy=_Cfg(l2coeff=0.005))
    ranker = CenteredRanker()
    assert es._can_fuse_step(dist.world(), policy, fit_fn, ranker)
    flat = v['theta0'].copy()
    opt = orc.AdamOracle(len(flat), 0.01)
    stat = orc.ObStatOracle((obs_dim,), 1e-2)
    obmean, obstd = np.zeros(obs_dim), np.ones(obs_dim)
    tol = 2e-5 if mode == 0 else 6e-5
    for g in range(2):
        tr, gen_obstat = es.step(cfg, dist.world(), policy, nt, env, fit_fn, rs, ranker, Reporter())
        policy.update_obstat(gen_obstat)
        ref = eps_orc.es_step(table, flat, opt, 0.02, dims, spec, [ref_rs], n_pairs, obmean, obstd, 5.0, T, 500, 0.005, E,
                              coins_per_eval=1, save_obs_chance=float(v['save_obs_chance']), batched=False, ac_std=ac_std)
        stat.inc(ref['obstat'].sum, ref['obstat'].sumsq, ref['obstat'].count)
        obmean, obstd = stat.mean, stat.std
        assert np.array_equal(np.asarray(ranker.noise_inds), v[f's{g}_inds']) and np.array_equal(ref['inds'], v[f's{g}_inds'])
        st = rs.get_state()
        assert np.array_equal(st[1], v[f's{g}_rs_key']) and st[2] == int(v[f's{g}_rs_pos']) and st[3] == int(v[f's{g}_rs_has_gauss'])
        assert abs(st[4] - float(v[f's{g}_rs_gauss'])) <= 2 * np.spacing(abs(float(v[f's{g}_rs_gauss'])))
        fits = np.concatenate((ranker.fits_pos, ranker.fits_neg)).ravel()
        assert np.abs(fits - v[f's{g}_fits'].ravel()).max() <= tol
        assert np.abs(ranker.fits_pos - ref['pos']).max() <= tol and np.abs(ranker.fits_neg - ref['neg']).max() <= tol
        assert np.array_equal(np.asarray(ranker.ranked_fits).ravel(), v[f's{g}_w'].ravel())
        assert np.array_equal(gen_obstat.sum, v[f's{g}_ob_sum']) and gen_obstat.count == float(v[f's{g}_ob_count'])
        assert np.abs(policy.flat_params - v[f's{g}_theta']).max() <= 3e-6
        assert np.abs(policy.flat_params - flat).max() <= 3e-6
        assert abs(tr.result[0] - float(v[f's{g}_noiseless'][0])) <= 1e-4 and abs(tr.result[0] - ref['noiseless'][0]) <= 1e-4


def test_per_policy_call_with_episodes_matches_the_oracle(eng):
    """fit_fn(policy.pheno(zeros), True) of a BatchedRollout(eps_per_policy=4): the coin, ONE rs.randn(E * T * act) from the
    stream, one launch; fitness, the last episode's position and the stream afterwards as obj.py's r_fn."""
    from es_pytorch_b200.gym.batched import BatchedRollout
    obs_dim, act_dim, T, E = 17, 6, 60, 4
    spec = orc.SyntheticEnvSpec(obs_dim, act_dim, T)
    dims = orc.layer_dims(obs_dim, (64, 64), act_dim)
    theta = (np.random.RandomState(2).randn(orc.n_params(dims)) * 0.1).astype(F32)
    env, net, policy = _api_objects((64, 64), spec, theta)
    net._action_std = 0.01
    a, b = np.random.RandomState(78), np.random.RandomState(78)
    a.randn(1); b.randn(1)
    fit_fn = BatchedRollout(env, T, coins_per_eval=1, save_obs_chance=0.5, rank_streams=[a], eps_per_policy=E)
    launches = eng.launches
    tr = fit_fn(policy.pheno(np.zeros(len(policy))), True)
    assert eng.launches - launches <= 4, 'one normalise + rollout launches, not E episodes'
    b.random()
    rews, behv, _, step = eps_orc.run_episodes(spec, orc.unflatten(theta, dims), np.zeros(obs_dim), np.ones(obs_dim), 5.0, T, E,
                                               batched=False, ac_std=0.01, rs=b)
    assert tr.steps == step and abs(tr.result[0] - sum(rews)) <= 1e-5 * max(1.0, np.abs(rews).sum())
    assert np.allclose(tr.positions[-3:], behv[-3:], rtol=1e-4, atol=1e-5)
    sa, sb = a.get_state(), b.get_state()
    assert np.array_equal(sa[1], sb[1]) and sa[2:] == sb[2:]


# ---- 6. rejections --------------------------------------------------------------------------------------------------------
def test_episode_rejections(eng):
    from es_pytorch_b200 import _lib
    c = _inputs(SMALL, 40, 3, 2, seed=9)
    with pytest.raises(_lib.EsLibraryError, match='n_episodes must be >= 1'):
        _run(eng, c, 0, E=0)
    with pytest.raises(_lib.EsLibraryError, match='n_episodes must be >= 1'):
        _run(eng, c, 0, E=-3, noise=False)
    # E * T * act > INT_MAX (es_draw_noisy's normals_per_eval is an int): ES_ERR_INVALID before any launch, so the small noise
    # array of this call is never read.  Straight through the C ABI: Engine checks the array's size first.
    import ctypes as C
    keep = [dev(eng, x) for x in (c['table'], c['idx'], c['theta'], c['obsn'], c['rew'], c['noise'])]
    fit = torch.zeros(2, 3, dtype=torch.float64, device=eng.device)
    ptr = [C.c_void_p(x.data_ptr()) for x in keep]
    ls = (C.c_int * 4)(*SMALL)
    E_big = (1 << 31) // (40 * 6) + 1
    launches = eng.launches
    rc = eng.lib.es_rollout_openloop_episodes(eng._ctx, ptr[0], len(c['table']), ptr[1], 3, ptr[2], c['P'], 0.02, ls, 3, ptr[3], ptr[4],
                                              40, POS_SCALE, C.c_void_p(fit[0].data_ptr()), C.c_void_p(fit[1].data_ptr()), 1, None,
                                              None, ptr[5], E_big, 0, eng.stream)
    assert rc == -1                                                      # ES_ERR_INVALID
    assert b'INT_MAX' in eng.lib.es_last_error() and eng.launches == launches
    # tensor-core shapes outside the domain
    w = _inputs([15, 96, 96, 3], 40, 2, 2, seed=10)
    for mode in (1, 2):
        with pytest.raises(_lib.EsLibraryError, match='tensor-core path'):
            _run(eng, w, mode)
    # an index outside the table is flagged asynchronously, as in the single-episode entries
    bad = dict(c, idx=np.array([0, len(c['table']) - 10, 1], dtype=np.int64))
    with pytest.raises(_lib.EsLibraryError, match='outside the table'):
        _run(eng, bad, 0)
    eng.sync()
    f, _ = _run(eng, c, 0)                                               # the ctx works again afterwards
    assert np.isfinite(f).all()
