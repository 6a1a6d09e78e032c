"""Generates tests/golden/ref_ranker_cases.npz and tests/golden/ref_script_surface.json from a checkout of the original
es_pytorch project (needs its ``src`` package importable, numpy and torch):

    python tests/golden/make_ref_cases.py <path to the original es_pytorch checkout>

  * ``ref_ranker_cases.npz`` -- the rank shapings (Centered / DoublePositiveCentered / SemiCentered / MaxNormalized) and
    EliteRanker of the REAL src/utils/rankers.py on seeded random inputs of the kinds a property test draws: sizes 1..40,
    distinct float64 values from +-1e-300 to +-1e6, integers, values next to zero and to the bounds.
    tests/test_oracle_properties.py checks the oracle against them.
  * ``ref_script_surface.json`` -- the import statements of the original training scripts (simple_example.py, obj.py,
    nsra.py, multi_agent.py: module and imported names) and the content of configs/simple_conf.json.
    tests/test_host_logic.py resolves every one of those imports against es_pytorch_b200/compat.
"""
import ast
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SCRIPTS = ('simple_example', 'obj', 'nsra', 'multi_agent')
SHAPINGS = ('centered', 'double_positive', 'semi_centered', 'max_normalized')
N_SHAPING_CASES, N_ELITE_CASES = 80, 40


def _distinct_values(rs, n):
    """n distinct float64 in [-1e6, 1e6] from one of several regimes (the inputs a hypothesis float strategy favours)."""
    while True:
        kind = rs.randint(5)
        if kind == 0:
            v = rs.uniform(-1e6, 1e6, n)
        elif kind == 1:
            v = rs.randint(-3 * n, 3 * n + 1, n).astype(np.float64)
        elif kind == 2:
            v = rs.choice([-1.0, 1.0], n) * 10.0 ** rs.uniform(-300, 6, n)
        elif kind == 3:
            v = rs.randn(n) * 10.0 ** rs.randint(-8, 4)
        else:
            v = np.concatenate((rs.choice([0.0, 1e6, -1e6, 5e-324, -5e-324, 1.0, -1.0], min(n, 3), replace=False),
                                rs.uniform(-1e6, 1e6, n)))[:n]
        v = np.clip(v, -1e6, 1e6)
        if len(np.unique(v)) == n:                  # tie order is unpinned in the reference
            return v


def ranker_cases(R):
    """Cases packed flat: case i of a kind owns x[off[i]:off[i + 1]] (2k fitness values, pos then neg); a shaping's k weights
    are w[off[i] // 2:off[i + 1] // 2] in float64, to be cast back to the stored dtype and ndim."""
    plain = {'centered': R.CenteredRanker, 'double_positive': R.DoublePositiveCenteredRanker,
             'semi_centered': R.SemiCenteredRanker, 'max_normalized': R.MaxNormalizedRanker}
    rs = np.random.RandomState(31337)
    sx, sw, sname, sdtype, sndim = [], [], [], [], []
    while len(sname) < N_SHAPING_CASES:
        name = SHAPINGS[len(sname) % len(SHAPINGS)]
        k = int(rs.choice([1, 2, 40, rs.randint(1, 41)]))
        x = _distinct_values(rs, 2 * k).reshape(2 * k, 1)
        if name == 'max_normalized' and (x.max() + (-x.min() if x.min() > 0 else x.min())) == 0:
            continue                                # the reference divides by zero
        w = plain[name]().rank(x[:k].copy(), x[k:].copy(), np.arange(k))
        assert w.shape in ((k,), (k, 1)) and w.dtype in (np.float32, np.float64)
        sx.append(x.ravel()), sw.append(w.astype(np.float64).ravel()), sname.append(SHAPINGS.index(name))
        sdtype.append(w.dtype.str), sndim.append(w.ndim)
    ex, ev, ei, en, ename, epct = [], [], [], [], [], []
    for i in range(N_ELITE_CASES):
        name = ('centered', 'double_positive')[i % 2]
        k = int(rs.choice([1, 2, 40, rs.randint(1, 41)]))
        pct = float(rs.choice([0.0, 1.0, rs.uniform(0, 1), rs.uniform(0, 1)]))
        x = _distinct_values(rs, 2 * k).reshape(2 * k, 1)
        inds = np.arange(100, 100 + k).astype(np.float64)
        e = R.EliteRanker(plain[name](), pct)
        vals = np.asarray(e.rank(x[:k].copy(), x[k:].copy(), inds.copy()), dtype=np.float64)
        order = np.lexsort((e.noise_inds, vals))    # argpartition's order is unspecified: stored sorted
        assert e.n_fits_ranked == len(vals)
        ex.append(x.ravel()), ev.append(vals[order]), ei.append(np.asarray(e.noise_inds, dtype=np.float64)[order])
        en.append(len(vals)), ename.append(SHAPINGS.index(name)), epct.append(pct)
    offsets = lambda parts: np.cumsum([0] + [len(p) for p in parts]).astype(np.int64)
    out = dict(shapings=np.array(SHAPINGS),
               shape_name=np.array(sname, dtype=np.int8), shape_off=offsets(sx), shape_x=np.concatenate(sx),
               shape_w=np.concatenate(sw), shape_w_dtype=np.array(sdtype), shape_w_ndim=np.array(sndim, dtype=np.int8),
               elite_name=np.array(ename, dtype=np.int8), elite_pct=np.array(epct), elite_off=offsets(ex),
               elite_x=np.concatenate(ex), elite_off_out=offsets(ev), elite_vals=np.concatenate(ev), elite_inds=np.concatenate(ei))
    np.savez_compressed(os.path.join(HERE, 'ref_ranker_cases.npz'), **out)
    print('ref_ranker_cases.npz', len(sname), 'shaping and', len(ename), 'elite cases')


def script_surface(ref_dir):
    imports = {}
    for s in SCRIPTS:
        with open(os.path.join(ref_dir, s + '.py')) as f:
            tree = ast.parse(f.read())
        rows = []
        for node in tree.body:
            if isinstance(node, ast.Import):
                rows += [{'module': a.name} for a in node.names]
            elif isinstance(node, ast.ImportFrom):
                rows.append({'module': node.module, 'names': [a.name for a in node.names]})
        imports[s] = rows
    with open(os.path.join(ref_dir, 'configs', 'simple_conf.json')) as f:
        conf = json.load(f)
    with open(os.path.join(HERE, 'ref_script_surface.json'), 'w') as f:
        json.dump({'imports': imports, 'simple_conf': conf}, f, indent=1)
        f.write('\n')
    print('ref_script_surface.json', sum(map(len, imports.values())), 'imports')


if __name__ == '__main__':
    ref = os.path.abspath(sys.argv[1])
    sys.path.insert(0, ref)
    from src.utils import rankers
    ranker_cases(rankers)
    script_surface(ref)
