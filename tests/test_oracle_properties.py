"""CPU property tests (hypothesis): the oracle's restatements against live third-party / reference behaviour on random inputs,
beyond the fixed golden vectors.
  * the MT19937 + masked-rejection restatement against numpy's legacy RandomState (the pinned RNG of the reference);
  * the rank shapings and EliteRanker against outputs of the REAL reference module on 120 seeded random cases
    (tests/golden/ref_ranker_cases.npz, written by tests/golden/make_ref_cases.py)."""
import os

import numpy as np
from hypothesis import given, settings, strategies as st

from oracle import es_oracle as orc


@settings(max_examples=25, deadline=None)
@given(seed=st.integers(0, 2 ** 32 - 1), burn=st.integers(0, 700), n=st.integers(1, 120),
       ub=st.one_of(st.integers(2, 5000), st.integers(2 ** 20, 2 ** 32 - 2), st.just(250_000_000 - 29_393)),
       extra=st.sampled_from([0, 1, 2, 4, 7]))
def test_mt_draw_restatement_matches_numpy_legacy_randomstate(seed, burn, n, ub, extra):
    rs = np.random.RandomState(seed)
    for _ in range(burn):
        rs.random()                                   # arbitrary starting position inside / across 624-word blocks
    st0 = rs.get_state()
    want_idx, want_extra = [], []
    for _ in range(n):
        want_idx.append(int(rs.randint(0, ub)))
        want_extra.append([int.from_bytes(rs.bytes(4), 'little') for _ in range(extra)])
    idx, ext, key, pos = orc.mt_draw_indices(st0[1], int(st0[2]), n, ub, extra)
    assert idx == want_idx and ext == want_extra
    st1 = rs.get_state()
    # numpy may stop at pos == 624 where the restatement has already regenerated (or the reverse): compare by continuing
    cont = np.random.RandomState()
    cont.set_state(('MT19937', np.array(key, dtype=np.uint32), int(pos), st1[3], st1[4]))
    assert [int(cont.randint(0, 1 << 30)) for _ in range(5)] == [int(rs.randint(0, 1 << 30)) for _ in range(5)]


def _ranker_cases():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'ref_ranker_cases.npz'))


def test_shapings_match_the_real_reference_rankers():
    v = _ranker_cases()
    off = v['shape_off']
    for i, code in enumerate(v['shape_name']):
        name = str(v['shapings'][code])
        x = v['shape_x'][off[i]:off[i + 1]].reshape(-1, 1)
        k = len(x) // 2
        want = v['shape_w'][off[i] // 2:off[i + 1] // 2].astype(v['shape_w_dtype'][i]).reshape((k,) if v['shape_w_ndim'][i] == 1 else (k, 1))
        got, n = orc.shaped_ranker(x[:k], x[k:], name)
        assert n == 2 * k and got.dtype == want.dtype and got.shape == want.shape, (i, name)
        assert np.array_equal(got, want, equal_nan=True), (i, name)


def test_elite_matches_the_real_reference_ranker():
    v = _ranker_cases()
    off, off_out = v['elite_off'], v['elite_off_out']
    for i, code in enumerate(v['elite_name']):
        name = str(v['shapings'][code])
        x = v['elite_x'][off[i]:off[i + 1]].reshape(-1, 1)
        k = len(x) // 2
        want, want_inds = v['elite_vals'][off_out[i]:off_out[i + 1]], v['elite_inds'][off_out[i]:off_out[i + 1]]
        inds = np.arange(100, 100 + k).astype(np.float64)
        vals_o, inds_o, _, n = orc.elite_ranker(x[:k], x[k:], inds, name, float(v['elite_pct'][i]))
        assert n == len(want), (i, name)
        b = np.lexsort((inds_o, vals_o))                                                  # argpartition's order is unspecified
        assert np.array_equal(want, vals_o[b]) and np.array_equal(want_inds, inds_o[b]), (i, name)
