"""CPU (no GPU): the C-ABI library loads and exports every symbol include/es_b200.h declares, the
host-side mirror keeps the reference's API surface, the shims let the reference scripts import,
and the multi-process plumbing (gloo, world_size 2) keeps the reference's result layout."""
import importlib.util
import json
import os
import re
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from oracle import es_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COMPAT = os.path.join(ROOT, 'es_pytorch_b200', 'compat')


def test_c_abi_exports_every_declared_symbol():
    from es_pytorch_b200 import _lib, build
    build.build()
    hdr = open(os.path.join(ROOT, 'include', 'es_b200.h')).read()
    declared = set(re.findall(r'\b(es_[a-z0-9_]+)\s*\(', hdr))
    declared.discard('es_ctx')
    assert len(declared) >= 18
    lib = _lib.load()
    for name in sorted(declared):
        assert hasattr(lib, name), f'{name} declared in include/es_b200.h but not exported'
    assert declared == set(_lib.SIGNATURES), (declared ^ set(_lib.SIGNATURES))
    assert lib.es_abi_version() == 1


def test_no_gpu_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    from es_pytorch_b200._lib import EsLibraryError
    from es_pytorch_b200.engine import get_engine
    with pytest.raises(EsLibraryError, match='no CPU path'):
        get_engine()
    from es_pytorch_b200.utils.rankers import CenteredRanker
    with pytest.raises(EsLibraryError):
        CenteredRanker().rank(np.zeros((2, 1)), np.ones((2, 1)), np.arange(2))


def test_product_never_imports_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, 'es_pytorch_b200')):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh')):
                src = open(os.path.join(dirpath, f)).read()
                assert 'oracle' not in src.replace('the oracle', '').replace('CPU oracle', ''), os.path.join(dirpath, f)


def test_synthetic_env_matches_oracle_spec():
    from es_pytorch_b200.gym.synthetic_env import SyntheticEnv, make
    spec = orc.SyntheticEnvSpec(17, 6, 30)
    env = SyntheticEnv(17, 6, 30)
    assert np.array_equal(env.obs_stream, spec.obs_stream) and np.array_equal(env.rew_vec, spec.rew_vec)
    rs = np.random.RandomState(0)
    acts = rs.randn(30, 6).astype(np.float32)
    ob = env.reset()
    assert np.array_equal(ob, spec.obs_stream[0])
    rews = []
    for t in range(30):
        ob, r, done, _ = env.step(acts[t])
        rews.append(r)
        assert np.array_equal(ob, spec.obs_stream[t + 1]) and done == (t == 29)
    # same arithmetic as the oracle's run_model reward / position integrator
    pos = np.zeros(3, dtype=np.float32)
    for t in range(30):
        acc = np.float32(0)
        for j in range(6):
            acc = np.float32(acc + np.float32(acts[t, j] * spec.rew_vec[t, j]))
        assert rews[t] == float(acc)
        for j in range(3):
            pos[j] = np.float32(pos[j] + np.float32(np.float32(0.05) * acts[t, j]))
    assert np.array_equal(env.pos, pos) and env.robot.robot_body.pose().xyz() == tuple(float(x) for x in pos)
    with pytest.raises(RuntimeError):
        env.step(acts[0])
    assert make('HalfCheetahBulletEnv-v0').obs_dim == 17 and make('HumanoidBulletEnv-v0').act_dim == 17
    with pytest.raises(ValueError):
        make('NoSuchEnv-v0')


def test_noisetable_api():
    from es_pytorch_b200.core.noisetable import NoiseTable
    nt = NoiseTable(50, np.arange(100))
    assert len(nt) == 100 and (nt.get(3, 50) == np.arange(3, 53)).all() and (nt[7] == np.arange(7, 57)).all()
    with pytest.raises(AssertionError):
        nt.get(50, 50)                                   # noisetable.py:34: len > i + size
    with pytest.raises(ValueError):
        NoiseTable(100, np.arange(100)).sample_idx(np.random.RandomState(0), 100)   # noisetable.py:39
    rs, ref = np.random.RandomState(5), np.random.RandomState(5)
    idx, sl = nt.sample(rs)
    assert idx == ref.randint(0, 50) and (sl == np.arange(idx, idx + 50)).all()
    assert np.array_equal(NoiseTable.make_noise(5, 1), np.random.RandomState(1).randn(5).astype(np.float32))


def test_obstat_api():
    from es_pytorch_b200.nn.obstat import ObStat
    a, b, ref = ObStat((4,), 1e-2), ObStat((4,), 0), orc.ObStatOracle((4,), 1e-2)
    x = np.random.RandomState(0).randn(10, 4).astype(np.float32)
    b.inc(x.sum(0), np.square(x).sum(0), 10)
    a += b
    r2 = orc.ObStatOracle((4,), 0)
    r2.inc(x.sum(0), np.square(x).sum(0), 10)
    ref.merge(r2)
    assert np.array_equal(a.sum, ref.sum) and np.array_equal(a.mean, ref.mean) and np.array_equal(a.std, ref.std)


def test_policy_flat_layout_and_pickle(tmp_path):
    import pickle
    import torch
    from es_pytorch_b200.core.policy import Policy
    from es_pytorch_b200.gym.synthetic_env import SyntheticEnv
    from es_pytorch_b200.nn.nn import FeedForward
    from es_pytorch_b200.nn.optimizers import Adam
    env = SyntheticEnv(17, 6, 8)
    net = FeedForward([64, 64], torch.nn.Tanh(), env, 0.0, 5)
    pol = Policy(net, 0.02, Adam(5702, 0.01))
    assert len(pol) == 5702 == orc.n_params(orc.layer_dims(17, (64, 64), 6)) and pol.flat_params.dtype == np.float32
    assert net.layer_sizes() == [17, 64, 64, 6] and net.is_tanh_mlp()
    # state_dict order = weight[out,in] row-major then bias (policy.py:33-35): oracle.unflatten reads it back
    layers = orc.unflatten(pol.flat_params, orc.layer_dims(17, (64, 64), 6))
    assert np.array_equal(layers[0][0], net.model[0].weight.detach().numpy())
    assert np.array_equal(layers[2][1], net.model[4].bias.detach().numpy())
    flat2 = np.random.RandomState(0).randn(5702).astype(np.float32)
    pol.set_nn_params(flat2)
    assert np.array_equal(Policy.get_flat(net), flat2)
    # forward of the module == oracle forward (float64 normalise, tanh after every layer)
    net.set_ob_mean_std(np.full(17, 0.1), np.full(17, 2.0))
    ob = np.random.RandomState(1).randn(17).astype(np.float32)
    got = net(torch.from_numpy(ob), rs=None).detach().numpy()
    want = orc.mlp_forward(orc.unflatten(flat2, orc.layer_dims(17, (64, 64), 6)),
                           orc.normalise_obs(ob, np.full(17, 0.1), np.full(17, 2.0), 5))
    assert np.allclose(got, want, rtol=1e-6, atol=1e-7)
    pol.save(str(tmp_path), 'x')
    pol2 = Policy.load(os.path.join(str(tmp_path), 'policy-x'))
    assert np.array_equal(pol2.flat_params, pol.flat_params) and pol2.optim.t == 0 and pol2.std == 0.02


def test_reference_scripts_import_against_the_shims(tmp_path):
    """Every import statement of simple_example.py / obj.py / nsra.py / multi_agent.py (their module-level code is imports
    and function definitions) resolves against es_pytorch_b200/compat, and the shims' load_config reads
    configs/simple_conf.json; both recorded from the reference by tests/golden/make_ref_cases.py."""
    with open(os.path.join(ROOT, 'tests', 'golden', 'ref_script_surface.json')) as f:
        surface = json.load(f)
    assert sorted(surface['imports']) == ['multi_agent', 'nsra', 'obj', 'simple_example']
    conf = tmp_path / 'simple_conf.json'
    conf.write_text(json.dumps(surface['simple_conf']))
    code = textwrap.dedent('''
        import json, sys
        surface = json.load(open(sys.argv[1]))
        for script, rows in surface['imports'].items():
            for row in rows:
                if 'names' in row:
                    exec('from %s import %s' % (row['module'], ', '.join(row['names'])), {})
                else:
                    exec('import ' + row['module'], {})
        import src.core.es, es_pytorch_b200.core.es
        assert src.core.es is es_pytorch_b200.core.es
        from src.utils import utils
        cfg = utils.load_config(sys.argv[2])
        assert cfg.general.policies_per_gen == 4800 and cfg.noise.std == 0.02
        print('OK')
    ''')
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + COMPAT)
    out = subprocess.run([sys.executable, '-c', code, os.path.join(ROOT, 'tests', 'golden', 'ref_script_surface.json'), str(conf)],
                         capture_output=True, text=True, env=env)
    assert out.returncode == 0 and 'OK' in out.stdout, out.stderr[-2000:]


def test_shard_bounds():
    from es_pytorch_b200.dist import shard_bounds
    assert [shard_bounds(40000, 8, r) for r in (0, 7)] == [(0, 5000), (35000, 40000)]
    with pytest.raises(ValueError):
        shard_bounds(10, 3, 0)


_GLOO_WORKER = '''
import os, sys
sys.path.insert(0, {root!r})
import numpy as np, torch
from es_pytorch_b200 import dist
from es_pytorch_b200.core.es import _share_results
from es_pytorch_b200.nn.obstat import ObStat
comm = dist.init_from_env('gloo')
assert comm.size == 2
# test/es/es_runner_test.py:10-31 on two real processes
evals, objectives = 5, 4
pf = evals * comm.rank + 1
inds = (np.arange(evals) + pf) * 10
fp = [[i + i * 10 ** j if j != 0 else i for j in range(objectives)] for i in range(pf, pf + evals)]
fn = (-np.array(fp)).tolist()
res = _share_results(comm, fp, fn, inds)
expected = []
for i in range(1, evals * comm.size + 1):
    p = [i + i * 10 ** j if j != 0 else i for j in range(objectives)]
    expected.append(p + (-np.array(p)).tolist() + [i * 10])
assert res.dtype == np.float64 and (res == expected).all()
# test/utils/obstat_test.py:8-23
ob = ObStat(5, 0)
ob.inc(np.arange(5) * (comm.rank + 1), np.square(np.arange(5) * (comm.rank + 1)), 1)
ob.mpi_inc(comm)
es_, eq = np.zeros(5), np.zeros(5)
for i in range(comm.size):
    es_ += np.arange(5) * (i + 1); eq += np.square(np.arange(5) * (i + 1))
assert (ob.sum == es_).all() and (ob.sumsq == eq).all() and ob.count == comm.size
# the two collectives of the sharded generation: rank-major allgather, summed partial gradient
loc = torch.full((3, 2), float(comm.rank))
out = torch.empty(2, 3, 2)
comm.allgather_into(out, loc)
assert out[0].eq(0).all() and out[1].eq(1).all()
g = torch.arange(4, dtype=torch.float32) * (comm.rank + 1)
comm.allreduce_sum(g)
assert torch.equal(g, torch.arange(4, dtype=torch.float32) * 3)
assert comm.broadcast_object('seed-%d' % comm.rank, 0) == 'seed-0'
# mpi4py shim over the same group
sys.path.insert(0, {compat!r})
from mpi4py import MPI
c = MPI.COMM_WORLD
assert c.rank == comm.rank and c.size == 2
assert c.alltoall([c.rank * 10 + 1] * 2) == [1, 11] and c.scatter(['a', 'b']) == 'ab'[c.rank] and c.allreduce(c.rank + 1, MPI.SUM) == 3
send = np.tile(np.arange(3, dtype=np.float64) + 10 * c.rank, 2)
recv = np.empty(6)
c.Alltoall(send, recv)
assert (recv == np.concatenate([np.arange(3), np.arange(3) + 10])).all()
os.write(1, ('RANK_OK_%d\\n' % comm.rank).encode())
'''


def test_two_process_gloo(tmp_path):
    script = tmp_path / 'w.py'
    script.write_text(_GLOO_WORKER.format(root=ROOT, compat=COMPAT))
    import socket
    with socket.socket() as sk:
        sk.bind(('127.0.0.1', 0))
        port = sk.getsockname()[1]
    out = subprocess.run([sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node=2',
                          '--master-addr', '127.0.0.1', '--master-port', str(port), str(script)],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, (out.stdout + out.stderr)[-3000:]
    assert 'RANK_OK_0' in out.stdout and 'RANK_OK_1' in out.stdout


# ---- host-side descriptions of the device calls (no GPU needed) ------------------------------------------------------
def test_ranker_specs_describe_the_device_call():
    """Every ranker of src/utils/rankers.py is (shaping kind, blend weights, elite count); the combinations the reference
    itself cannot run are refused."""
    from es_pytorch_b200 import _lib
    from es_pytorch_b200.utils import rankers as R
    assert R.CenteredRanker()._spec(1, 200) == (_lib.ES_RANK_CENTERED, 1.0, 0.0, 0)
    assert R.DoublePositiveCenteredRanker()._spec(1, 200)[0] == _lib.ES_RANK_DOUBLE_POSITIVE
    assert R.SemiCenteredRanker()._spec(1, 200)[0] == _lib.ES_RANK_SEMI_CENTERED and not R.SemiCenteredRanker().squeeze
    assert R.MaxNormalizedRanker()._spec(1, 200)[0] == _lib.ES_RANK_MAX_NORMALIZED
    assert R.MultiObjectiveRanker(R.CenteredRanker(), 0.3)._spec(2, 200) == (_lib.ES_RANK_CENTERED, 0.3, 0.7, 0)
    # rankers.py:94: n_elite = max(1, int(ranked.size * elite_percent))
    assert R.EliteRanker(R.CenteredRanker(), 0.1)._spec(1, 200)[3] == 20
    assert R.EliteRanker(R.CenteredRanker(), 0.0)._spec(1, 200)[3] == 1
    assert R.EliteRanker(R.DoublePositiveCenteredRanker(), 1.0)._spec(1, 200) == (_lib.ES_RANK_DOUBLE_POSITIVE, 1.0, 0.0, 200)
    with pytest.raises(ValueError):
        R.CenteredRanker()._spec(2, 200)                      # two objectives need MultiObjectiveRanker
    with pytest.raises(NotImplementedError):
        R.EliteRanker(R.MultiObjectiveRanker(R.CenteredRanker(), 0.5), 0.1)
    with pytest.raises(NotImplementedError):
        R.MultiObjectiveRanker(R.EliteRanker(R.CenteredRanker(), 0.1), 0.5)
    with pytest.raises(AssertionError):
        R.EliteRanker(R.CenteredRanker(), 1.5)                 # rankers.py:89


def test_step_takes_the_single_sync_route_only_when_results_are_identical():
    """es.step keeps a generation on the device for float32 shapings without elite selection evaluated by a BatchedRollout
    of a tanh MLP; everything else goes call by call (same results, more synchronisations)."""
    import torch
    from es_pytorch_b200 import dist
    from es_pytorch_b200.core import es
    from es_pytorch_b200.core.policy import Policy
    from es_pytorch_b200.gym.batched import BatchedRollout
    from es_pytorch_b200.gym.synthetic_env import SyntheticEnv
    from es_pytorch_b200.nn.nn import FeedForward
    from es_pytorch_b200.nn.optimizers import Adam
    from es_pytorch_b200.utils import rankers as R
    from es_pytorch_b200.utils.reporters import Reporter, ReporterSet, StdoutReporter
    env = SyntheticEnv(17, 6, 20)
    net = FeedForward([64, 64], torch.nn.Tanh(), env, 0.0)
    policy = Policy(net, 0.02, Adam(len(Policy.get_flat(net)), 0.01))
    comm = dist.world()
    batched, batched2 = BatchedRollout(env, 20), BatchedRollout(env, 20, archive=np.zeros((4, 2)))
    assert es._can_fuse_step(comm, policy, batched, R.CenteredRanker())
    assert es._can_fuse_step(comm, policy, batched, R.SemiCenteredRanker())
    assert es._can_fuse_step(comm, policy, batched2, R.MultiObjectiveRanker(R.CenteredRanker(), 0.5))
    assert not es._can_fuse_step(comm, policy, batched, R.EliteRanker(R.CenteredRanker(), 0.1))     # compact host lists
    assert not es._can_fuse_step(comm, policy, batched, R.MaxNormalizedRanker())                    # float64 weights
    assert not es._can_fuse_step(comm, policy, batched2, R.CenteredRanker())                        # needs two objectives
    assert not es._can_fuse_step(comm, policy, lambda model: None, R.CenteredRanker())              # opaque fit_fn
    relu = FeedForward([64, 64], torch.nn.ReLU(), env, 0.0)
    assert not es._can_fuse_step(comm, Policy(relu, 0.02, Adam(len(Policy.get_flat(relu)), 0.01)), batched, R.CenteredRanker())

    class FakeComm:
        size, rank = 3, 0
    assert not es._can_fuse_step(FakeComm(), policy, batched, R.CenteredRanker())                   # not this package's world
    assert es._silent(Reporter()) and es._silent(ReporterSet()) and not es._silent(StdoutReporter(comm))


def test_mt19937_streams_are_read_and_written_in_place():
    """DeviceGeneration reads / writes the callers' RandomState streams through numpy's BitGenerator.ctypes interface:
    equivalent to get_state()/set_state() on the key and position, the gaussian cache is left alone."""
    from es_pytorch_b200.generation import DeviceGeneration
    a, b = np.random.RandomState(123), np.random.RandomState(123)
    a.randn(3); b.randn(3)                                     # odd count: a cached gaussian is pending in both
    view = DeviceGeneration._mt_view(a)
    assert view is not None
    key, pos = view
    st = a.get_state()
    assert np.array_equal(key, st[1]) and pos.value == st[2]
    # advance b the official way, then write b's stream into a through the view
    for _ in range(1000):
        b.randint(0, 250_000_000); b.random()
    sb = b.get_state()
    key[:] = sb[1]
    pos.value = sb[2]
    assert a.get_state()[3:] == st[3:]                         # has_gauss / cached value untouched
    assert [a.randint(0, 10 ** 9) for _ in range(50)] == [b.randint(0, 10 ** 9) for _ in range(50)]
    assert a.randn() == b.randn()                              # both return their cached gaussian first
    assert DeviceGeneration._mt_view(np.random.default_rng(1)) is None if hasattr(np.random, 'default_rng') else True


# ---- bench.py's multi-rank control flow (the round-1 SCALE hang: per-rank iteration counts around collectives) -----------
_BENCH_LOOP_WORKER = '''
import os, sys, time
sys.path.insert(0, {root!r})
import torch, torch.distributed as td
import bench
from es_pytorch_b200 import dist
comm = dist.init_from_env('gloo')
assert comm.size == 2
calls = [0]
def step():                                   # stands for gen.run(): an allgather and two allreduces per generation
    calls[0] += 1
    out = torch.empty(2, 3)
    comm.allgather_into(out, torch.full((3,), float(comm.rank)))
    g = torch.ones(4); comm.allreduce_sum(g); comm.allreduce_sum(g)
class SkewedTimer:                            # rank 1's device clock reads 20x less than rank 0's: a per-rank `extra`
    def start(self): pass                     # would differ by 20x and desynchronise the collectives inside step()
    def stop(self): return 0.010 if comm.rank == 0 else 0.0005
def allreduce_max(x):
    t = torch.tensor([x], dtype=torch.float64); td.all_reduce(t, op=td.ReduceOp.MAX); return float(t.item())
marks = []
max_s, extra = bench.timed_region(step, 5, 2, comm, lambda: None, SkewedTimer(), allreduce_max, min_load_s=0.05,
                                  on_timed_start=lambda: marks.append(calls[0]), on_timed_end=lambda: marks.append(calls[0]))
assert max_s == 0.010, max_s                  # MAX over ranks, identical everywhere
assert extra == int((0.05 - 0.010) / (0.010 / 5)) + 1 == 21, extra
assert marks == [2, 7] and calls[0] == 2 + 5 + extra
both = [None, None]
td.all_gather_object(both, (calls[0], extra, max_s))
assert both[0] == both[1], both               # every rank ran the same number of generations
# no continuation needed -> none run
max_s, extra = bench.timed_region(step, 3, 1, comm, lambda: None, SkewedTimer(), allreduce_max)
assert extra == 0
# argument plumbing of the strong-scaling mode
a = bench.parse(['--gpus', '8', '--scaling', 'strong'])
assert bench.total_pairs(a, bench.WORKLOADS['humanoid'], 8) == 40000 and bench.total_pairs(a, bench.WORKLOADS['humanoid-nsra'], 8) == 10000
a = bench.parse(['--gpus', '8'])
assert bench.total_pairs(a, bench.WORKLOADS['humanoid'], 8) == 80000
os.write(1, ('LOOP_OK_%d\\n' % comm.rank).encode())
'''


def test_bench_timed_region_is_collective_safe(tmp_path):
    script = tmp_path / 'w.py'
    script.write_text(_BENCH_LOOP_WORKER.format(root=ROOT))
    import socket
    with socket.socket() as sk:
        sk.bind(('127.0.0.1', 0))
        port = sk.getsockname()[1]
    out = subprocess.run([sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node=2',
                          '--master-addr', '127.0.0.1', '--master-port', str(port), str(script)],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, (out.stdout + out.stderr)[-3000:]
    assert 'LOOP_OK_0' in out.stdout and 'LOOP_OK_1' in out.stdout


def test_remaining_nets_and_results_keep_the_reference_contracts():
    """nn.py:53-117 and training_result.py:33-79 (SURVEY 8f.4): the networks that post-process their outputs and the other
    fitness adaptors.  Against the real reference classes where the checkout is mounted, else against their documented
    arithmetic."""
    import torch
    from es_pytorch_b200.gym.synthetic_env import SyntheticEnv
    from es_pytorch_b200.gym.training_result import DistResult, MeanRewardResult, MultiAgentTrainingResult, RewardResult, XDistResult
    from es_pytorch_b200.nn.nn import FeedForward, FFBinned, FFIntegGausAction, FFIntegGausActionMulti
    env = SyntheticEnv(5, 4, 10)
    ob = torch.from_numpy(np.random.RandomState(0).randn(5).astype(np.float32))
    torch.manual_seed(3)
    a = FFIntegGausAction([8], torch.nn.Tanh(), env, 0.0)
    raw = a.model(ob).detach().numpy()
    out = a(ob, rs=np.random.RandomState(5))
    assert out.shape == (3,) and np.allclose(out, raw[1:] + np.random.RandomState(5).standard_normal(3) * raw[0])
    assert np.array_equal(a(ob, rs=None), raw[1:]) and not a.is_tanh_mlp()
    m = FFIntegGausActionMulti([8], torch.nn.Tanh(), env, 0.0)
    raw = m.model(ob).detach().numpy()
    assert np.allclose(m(ob, rs=np.random.RandomState(6)), raw[:2] + np.random.RandomState(6).standard_normal(2) * np.abs(raw[2:]))
    b = FFBinned([8], torch.nn.Tanh(), env, 5)
    raw = b.model(ob).detach().numpy().reshape(4, 5)
    assert np.allclose(b(ob, rs=None).numpy(), raw.argmax(1) / 4. * 2. - 1.) and not b.is_tanh_mlp()
    assert FeedForward([8], torch.nn.Tanh(), env, 0.0).is_tanh_mlp()
    rews, pos, obs = [1., 2., 3.], [0., 0., 0., 3., 4., 9.], np.ones((3, 5))
    assert RewardResult(rews, pos, obs, 2).result == [6.] and MeanRewardResult(rews, pos, obs, 2).result == [3.]
    assert DistResult(rews, pos, obs, 2).result == [5.] and XDistResult(rews, pos, obs, 2).result == [3.]
    ma = MultiAgentTrainingResult(np.array([[1., 10.], [2., 20.]]), pos, np.ones((2, 2, 5)), 1)
    assert ma.result == [3., 30.] and len(ma.ob_sum_sq_cnt) == 2 and ma.ob_sum_sq_cnt[1][2] == 2
    assert [t.result for t in ma.trainingresults(RewardResult)] == [[3.], [30.]]


def test_run_state_checkpoint_round_trip(tmp_path):
    """SURVEY 8f.3: the policy pickle plus what the reference omits -- the ranks' RandomState streams (position AND cached
    gaussian), the table seed, the generation counter.  A resumed run draws exactly what the original would have drawn."""
    import torch
    from es_pytorch_b200.core.policy import Policy
    from es_pytorch_b200.gym.synthetic_env import SyntheticEnv
    from es_pytorch_b200.nn.nn import FeedForward
    from es_pytorch_b200.nn.optimizers import Adam
    from es_pytorch_b200.utils.checkpoint import load_run_state, save_run_state
    env = SyntheticEnv(5, 2, 10)
    policy = Policy(FeedForward([8], torch.nn.Tanh(), env, 0.01, 5), 0.02, Adam(74, 0.01))
    streams = [np.random.RandomState(50 + r) for r in range(3)]
    streams[1].randn(3)                                     # cached gaussian
    streams[2].randint(0, 1000, size=700)
    path = save_run_state(str(tmp_path), 'g7', policy, streams, table_seed=123, generation=7, extra={'best': 1.5})
    want = [(s.randint(0, 10 ** 6), s.random(), s.randn(3).tolist()) for s in streams]
    st = load_run_state(path)
    assert st['table_seed'] == 123 and st['generation'] == 7 and st['extra'] == {'best': 1.5}
    assert [(s.randint(0, 10 ** 6), s.random(), s.randn(3).tolist()) for s in st['streams']] == want
    assert np.array_equal(st['policy'].flat_params, policy.flat_params) and st['policy'].std == 0.02
    assert st['policy']._module._action_std == 0.01


def test_gym_017_seed_hash_restatement_is_self_consistent():
    """gym 0.17.1 hashes the table seed before seeding the RandomState (noisetable.py:63); the shim's restatement
    (unpinned: the package is not available offline) must at least be deterministic, differ from the direct seeding and
    round-trip its big-int helpers."""
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + COMPAT)
    code = ('from gym.utils import seeding as s; import numpy as np\n'
            'a = s.np_random(123, hashed=True)[0].randn(3); b = s.np_random(123, hashed=True)[0].randn(3)\n'
            'c = s.np_random(123)[0].randn(3)\n'
            'assert np.array_equal(a, b) and not np.array_equal(a, c)\n'
            'h = s.hash_seed(123); assert 0 <= h < 2 ** 64 and s._int_list_from_bigint(h) == [h % 2 ** 32, h >> 32]\n'
            'assert s._bigint_from_bytes(bytes([1, 0, 0, 0, 2, 0, 0, 0])) == 1 + 2 * 2 ** 32\n'
            'print("OK")')
    out = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, env=env)
    assert out.returncode == 0 and 'OK' in out.stdout, out.stderr[-2000:]


def test_reporter_set_saves_fits_and_best_policy(tmp_path, monkeypatch):
    """DefaultMpiReporterSet (obj.py:24-28): per-generation np.save of the fitness matrix (reporters.py:188) and a policy
    checkpoint whenever the noiseless reward or distance improves; only rank 0 writes."""
    from es_pytorch_b200.gym.training_result import RewardResult
    from es_pytorch_b200.utils.reporters import DefaultMpiReporterSet, Reporter
    monkeypatch.chdir(tmp_path)

    class Comm:
        rank, size = 0, 1

    class Rec(Reporter):
        def __init__(self): self.logged, self.lines = {}, []
        def log(self, d): self.logged.update(d)
        def print(self, s): self.lines.append(s)

    class Pol:
        saved = []
        def save(self, folder, suffix): Pol.saved.append((folder, suffix))

    rec = Rec()
    rep = DefaultMpiReporterSet(Comm(), 'run', rec, None)
    fits = np.array([[1.0], [3.0], [2.0], [6.0]])
    for g, total in enumerate((5.0, 4.0, 9.0)):
        rep.start_gen()
        rep.log_gen(fits + g, RewardResult([total], [0., 0., 0., 3., 4., 0.] , np.zeros((1, 2)), 7), Pol(), 10)
        rep.end_gen()
        assert np.array_equal(np.load(os.path.join('saved', 'run', 'fits', f'{g}.np.npy')), fits + g)
    assert [s for _, s in Pol.saved] == ['0', '2']                    # generation 1 improved neither reward nor distance
    assert rec.logged['avg-0'] == 5.0 and rec.logged['max-0'] == 8.0 and rec.logged['cum steps'] == 30 and rec.logged['dist'] == 5.0
    assert rec.logged['n fits ranked'] == 4 and 'time' in rec.logged and rec.logged['gen'] == 2


def test_closed_loop_env_is_the_oracles_env():
    """gym.synthetic_env.ClosedLoopEnv (reset / step, what run_model's python loop drives) and the oracle's ClosedLoopEnvSpec are
    the same transition bit for bit; a perturbed start state is forgotten (the map is contractive: device / oracle rounding
    differences cannot grow along an episode)."""
    from oracle import es_oracle as orc
    from es_pytorch_b200.gym.synthetic_env import ClosedLoopEnv, make
    env, spec = ClosedLoopEnv(17, 6, 40), orc.ClosedLoopEnvSpec(17, 6, 40)
    assert np.array_equal(env.env_a, spec.env_a) and np.array_equal(env.env_b, spec.env_b)
    rs = np.random.RandomState(0)
    ob, ob_ref, other = env.reset(), spec.obs_stream[0].copy(), spec.obs_stream[0] + np.float32(0.3)
    for t in range(40):
        a = np.tanh(rs.randn(6)).astype(np.float32)
        ob, rew, done, _ = env.step(a)
        ob_ref = spec.step_obs(ob_ref, a)
        other = spec.step_obs(other, a)
        assert np.array_equal(ob, ob_ref) and done == (t == 39)
    assert np.abs(other - ob_ref).max() < 1e-6
    assert isinstance(make('HumanoidClosedLoop-v0'), ClosedLoopEnv) and make('HumanoidClosedLoop-v0').obs_dim == 376
    assert not isinstance(make('Humanoid-v2'), ClosedLoopEnv)


def test_run_model_python_loop_on_the_closed_loop_env_is_the_oracles_loop():
    """gym_runner.run_model's python loop (module forward + ClosedLoopEnv.step: the route of an opaque fit_fn, and the
    reference's own loop shape, src/gym/gym_runner.py:50-54) against the oracle's run_model_closed on the same parameters
    and a non-trivial observation normalisation: rewards, positions, post-step observations, last index."""
    import torch
    from es_pytorch_b200.core.policy import Policy
    from es_pytorch_b200.gym.gym_runner import run_model
    from es_pytorch_b200.gym.synthetic_env import ClosedLoopEnv
    from es_pytorch_b200.nn.nn import FeedForward
    from es_pytorch_b200.nn.optimizers import Adam
    obs_dim, act_dim, T = 17, 6, 25
    env, spec = ClosedLoopEnv(obs_dim, act_dim, T), orc.ClosedLoopEnvSpec(obs_dim, act_dim, T)
    dims = orc.layer_dims(obs_dim, (64, 64), act_dim)
    P = orc.n_params(dims)
    net = FeedForward([64, 64], torch.nn.Tanh(), env, 0.0, 5)
    pol = Policy(net, 0.02, Adam(P, 0.01))
    flat = (np.random.RandomState(2).randn(P) * 0.1).astype(np.float32)
    pol.set_nn_params(flat)
    mean, std = np.random.RandomState(3).randn(obs_dim) * 0.05, 0.5 + np.random.RandomState(4).rand(obs_dim)
    net.set_ob_mean_std(mean, std)
    rews, behv, obs, step = run_model(net, env, T)
    r_ref, b_ref, o_ref, s_ref = orc.run_model(spec, orc.unflatten(flat, dims), mean, std, 5.0, T)
    assert step == s_ref == T - 1 and len(rews) == T
    assert np.allclose(rews, r_ref, rtol=0, atol=2e-6) and np.allclose(behv, b_ref, rtol=0, atol=2e-6)
    assert np.allclose(obs, o_ref, rtol=0, atol=2e-6)


def test_jump_polynomials_against_numpys_mt19937():
    """es_pytorch_b200/mt_jump_polys.npy (x^(624 m 16^q) mod phi, what mt_fill_kernel jumps with): for a sample of (q, m) the
    relation x[n + 624 m 16^q] = XOR_{i : g_i = 1} x[n + i] on the raw words of numpy's own generator, and the C initialisers
    the kernels compile (csrc/mt_jump_polys.inc) are the same numbers."""
    sys.path.insert(0, os.path.join(ROOT, 'tools', 'mt_jump'))
    import make_jump_polys as mjp
    polys = np.load(os.path.join(ROOT, 'es_pytorch_b200', 'mt_jump_polys.npy'))
    assert polys.shape == (5, 15, 624) and polys.dtype == np.uint32
    raw = mjp.numpy_raw_words(77, 15 * 256 * 624 + 2 * mjp.DEG + 2048)
    for q, m in ((0, 1), (0, 3), (0, 15), (1, 5), (1, 8), (2, 1), (2, 15)):
        g = sum(int(w) << (32 * i) for i, w in enumerate(polys[q, m - 1]))
        assert g.bit_length() <= mjp.DEG and mjp.check_against_numpy(g, m * 16 ** q, raw), (q, m)
    with open(os.path.join(ROOT, 'es_pytorch_b200', 'csrc', 'mt_jump_polys.inc')) as f:
        rows = [ln for ln in f if ln.startswith('{')]
    assert len(rows) == 75
    for r in (0, 17, 74):
        vals = np.array([int(t.rstrip('u'), 16) for t in rows[r].strip().strip('{},').split(',')], dtype=np.uint64)
        assert np.array_equal(vals.astype(np.uint32), polys[r // 15, r % 15])
