"""Pins `oracle/hsc_oracle.py` against the reference: golden vectors of the reference's own tests,
traces recorded from the unmodified reference (tests/golden/*.npz, made by make_golden.py), and -
where a copy of the reference is supplied (HSC_REFERENCE_ROOT or baseline/_ref) - the live reference, bit for bit.  CPU only."""
import os
import sys

import numpy as np
import pytest
import scipy.sparse

from helpers import load_npz, case_kwargs, coo_sorted, stored_code, GOLDEN

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden'))
import ref_loader  # noqa: E402
from oracle import hsc_oracle as O  # noqa: E402

HAVE_REF = ref_loader.reference_available()


# ---------------- utils golden vectors (tests/hsc/test_utils.py:113-218 of the reference) -------

def test_reference_utils_known_answers():
    # peek: even width 4 centred at t=5 covers [4..7]; odd width 5 covers [3..7]
    s = np.arange(10)
    assert np.array_equal(O.peek(s, 4, 5), [4, 5, 6, 7])
    assert np.array_equal(O.peek(s, 5, 5), [3, 4, 5, 6, 7])
    assert np.array_equal(O.peek(s, 4, 0), [0, 1, 2])
    assert np.array_equal(O.peek(s, 4, 9), [8, 9])
    assert O.peek(s, 4, -6).size == 0
    # overlapAdd fully out of range is a no-op (tests/hsc/test_utils.py:153-184)
    z = np.zeros(8)
    assert np.array_equal(O.overlap_add(z.copy(), np.ones(4), -6), z)
    assert np.array_equal(O.overlap_add(z.copy(), np.ones(4), -20), z)
    assert np.array_equal(O.overlap_add(z.copy(), np.ones(4), 0), [1, 1, 1, 0, 0, 0, 0, 0])
    assert np.array_equal(O.overlap_replace(np.arange(8.0), -np.ones(3), 7), [0, 1, 2, 3, 4, 5, -1, -1])


def test_utils_vectors_from_reference():
    z = load_npz('utils_vectors.npz')
    n = int(z['count'])
    assert n > 300
    for i in range(n):
        T, width, t = [int(v) for v in z['case%d_in' % i]]
        exp_add = z['case%d_add' % i]
        if exp_add.ndim == 1:
            base = np.arange(T, dtype=np.float64) + 1.0
            elem = (np.arange(width, dtype=np.float64) + 1.0) * 10.0
        else:
            base = np.arange(24, dtype=np.float64).reshape(8, 3)
            elem = -np.arange(width * 3, dtype=np.float64).reshape(width, 3)
        assert np.array_equal(O.peek(base, width, t), z['case%d_peek' % i]), (T, width, t)
        assert np.array_equal(O.overlap_add(base.copy(), elem, t), exp_add), (T, width, t)
        assert np.array_equal(O.overlap_replace(base.copy(), elem, t), z['case%d_rep' % i]), (T, width, t)


# ---------------- correlation (hsc/modeling.py:149-188; tests/hsc/test_modeling.py:678-725) -----

def test_correlate_alignment_known_answer():
    # c[i+off, i] == ||filter_i||^2 when the signal holds filter i placed at start i
    rs = np.random.RandomState(0)
    for F in (1, 2, 5):
        for L in (5, 6):
            D = rs.randn(4, L, F)
            for i in range(4):
                x = np.zeros((40, F))
                x[10:10 + L] = D[i]
                c = O.correlate(x, D, 'same')
                off = O.centre_offset(L)
                assert np.isclose(c[10 + off, i], np.sum(D[i] ** 2))
                assert np.argmax(np.abs(c[:, i])) == 10 + off


def test_correlate_matches_reference_vectors():
    z = load_npz('correlate.npz')
    for i in range(int(z['count'])):
        x, D = z['c%d_x' % i], z['c%d_D' % i]
        same = O.correlate(x, D, 'same')
        valid = O.correlate(x, D, 'valid')
        assert same.dtype == z['c%d_same' % i].dtype
        tol = 1e-12 if x.dtype == np.float64 else 2e-6
        assert np.allclose(same, z['c%d_same' % i], rtol=0, atol=tol)
        assert np.allclose(valid, z['c%d_valid' % i], rtol=0, atol=tol)
    with pytest.raises(Exception):
        O.correlate(np.zeros(8), np.zeros((2, 3)), 'full')


# ---------------- selection (hsc/modeling.py:899-982; tests/hsc/test_modeling.py:272-325) -------

def test_select_atoms_reference_golden_lists():
    ramp = np.arange(256).reshape((64, 4)).astype(np.float64)
    ramp[-1] = ramp[-1][::-1]
    a = O.select_atoms(ramp, 5, 4, False)
    assert [x[0] for x in a] == [63, 47, 31, 15] and [x[1] for x in a] == [0, 3, 3, 3]
    a = O.select_atoms(ramp, 5, 4, True)
    assert [x[0] for x in a] == [63, 55, 39, 23, 7] and [x[1] for x in a] == [0, 3, 3, 3, 3]
    a = O.select_atoms(ramp, 3, 'auto', False)
    assert [x[0] for x in a] == [63, 59, 47, 35, 23, 11] and [x[1] for x in a] == [0, 3, 3, 3, 3, 3]
    a = O.select_atoms(ramp, 5, 5, False)
    assert [x[0] for x in a] == [59, 47, 35, 23, 11] and [x[1] for x in a] == [3, 3, 3, 3, 3]


def test_select_atoms_vectors_from_reference():
    z = load_npz('select_atoms.npz')
    for i in range(int(z['count'])):
        inner = z['s%d_inner' % i]
        L, nb, off = [int(v) for v in z['s%d_par' % i]]
        nb = 'auto' if nb < 0 else nb
        w = z['s%d_w' % i]
        w = None if w.size == 0 else w
        got = O.select_atoms(inner, L, nb, bool(off), float(z['s%d_thres' % i]), w)
        assert [g[0] for g in got] == z['s%d_t' % i].tolist(), i
        assert [g[1] for g in got] == z['s%d_k' % i].tolist(), i
        assert np.array_equal(np.array([g[2] for g in got], dtype=np.float64), z['s%d_c' % i]), i


# ---------------- MP / LoCOMP traces ------------------------------------------------------------

def _check_case(z, name):
    method = str(z[name + '_method'])
    x, D = z[name + '_x'], z[name + '_D']
    kw = case_kwargs(z, name)
    fn = O.mp_encode if method == 'cmp' else O.locomp_encode
    coef, res, tr = fn(x, D, return_trace=True, **kw)
    t, k, c = tr.arrays()
    assert t.tolist() == z[name + '_trace_t'].tolist(), name
    assert k.tolist() == z[name + '_trace_k'].tolist(), name
    assert np.array_equal(c, z[name + '_trace_c']), name
    r, cc, v = coo_sorted(coef)
    assert r.tolist() == z[name + '_coo_t'].tolist(), name
    assert cc.tolist() == z[name + '_coo_k'].tolist(), name
    assert np.allclose(v, z[name + '_coo_v'], rtol=1e-12, atol=0), name
    assert res.shape == z[name + '_res'].shape and res.dtype == z[name + '_res'].dtype
    assert np.array_equal(res, z[name + '_res']), name


def test_mp_cases_match_reference_traces():
    z = load_npz('mp_cases.npz')
    names = [str(n) for n in z['names']]
    assert len(names) >= 50
    for name in names:
        _check_case(z, name)


def test_planted_atoms_known_answer():
    # tests/hsc/test_modeling.py:379-396: MP recovers the 6 planted atoms exactly
    rs = np.random.RandomState(5)
    D = O.normalize(rs.random_sample(size=(4, 32)), axis=1)
    ref = scipy.sparse.coo_matrix(([1.0, 1.0, 0.5, 1.0, 0.75, 2.0], ([32, 48, 64, 96, 128, 192], [0, 3, 1, 0, 2, 2])),
                                  shape=(256, 4))
    x = O.reconstruct(ref, D)
    coef, res = O.mp_encode(x, D, nbNonzeroCoefs=8, minCoefficients=1e-6)
    assert coef.nnz == ref.nnz
    assert np.allclose(coef.toarray(), ref.toarray())
    assert np.allclose(res, 0.0, atol=1e-6)
    coef, res = O.locomp_encode(x, D, minCoefficients=1e-10)
    assert coef.nnz == ref.nnz
    assert np.allclose(coef.toarray(), ref.toarray(), atol=1e-1)


def test_lil_bookkeeping_is_equivalent():
    z = load_npz('mp_cases.npz')
    for name in ('snr20_f32', 'randn_T50_L16_F3_f64', 'blocks8_locomp_f64', 'f7_nnz16_locomp_f32'):
        method = str(z[name + '_method'])
        fn = O.mp_encode if method == 'cmp' else O.locomp_encode
        a, ra = fn(z[name + '_x'], z[name + '_D'], bookkeeping='dict', **case_kwargs(z, name))
        b, rb = fn(z[name + '_x'], z[name + '_D'], bookkeeping='lil', **case_kwargs(z, name))
        assert (a != b).nnz == 0 and np.array_equal(ra, rb)


@pytest.mark.skipif(not os.path.exists(os.path.join(GOLDEN, 'c1_toy.npz')), reason='dataset fixture missing')
def test_config1_toy_matches_reference():
    z = load_npz('c1_toy.npz')
    for name in ('c1_cmp', 'c1_locomp', 'c2s_cmp'):
        _check_case(z, name)
    assert len(z['c1_cmp_trace_t']) == 289          # SURVEY 8(d): 289 atoms, 20.078 dB


@pytest.mark.skipif(not os.path.exists(os.path.join(GOLDEN, 'c3_complex.npz')), reason='dataset fixture missing')
def test_config3_hierarchical_matches_reference():
    z = load_npz('c3_complex.npz')
    nl = int(z['nb_levels'])
    raw = [z['raw_l%d' % i] for i in range(nl)]
    rep = [z['rep_l%d' % i] for i in range(nl)]
    cns = z['counts_no_singletons']
    x = z['x']
    for tag, method, nb in (('cmp_b10', 'cmp', 10), ('cmp_b1', 'cmp', 1), ('locomp_b10', 'locomp', 10)):
        for dist in (True, False):
            codes, res = O.hierarchical_encode(x, raw, cns, rep, toleranceSnr=10.0, nbBlocks=nb, singletonWeight=0.95,
                                               returnDistributed=dist, method=method)
            sfx = '' if dist else '_nodist'
            for lvl, c in enumerate(codes):
                r, cc, v = coo_sorted(c)
                assert r.tolist() == z['%s%s_l%d_t' % (tag, sfx, lvl)].tolist(), (tag, lvl)
                assert cc.tolist() == z['%s%s_l%d_k' % (tag, sfx, lvl)].tolist(), (tag, lvl)
                assert np.allclose(v, z['%s%s_l%d_v' % (tag, sfx, lvl)], rtol=1e-10, atol=0), (tag, lvl)
            assert np.allclose(res, z['%s%s_res' % (tag, sfx)], rtol=0, atol=1e-12)


def test_ksvd_update_matches_reference():
    z = load_npz('ksvd_update.npz')
    for i in range(int(z['count'])):
        D0 = z['k%d_D0' % i]
        T = z['k%d_x' % i].shape[0]
        code = scipy.sparse.coo_matrix((z['k%d_code_v' % i], (z['k%d_code_t' % i], z['k%d_code_k' % i])),
                                       shape=(T, D0.shape[0])).tocsc()
        D1, code1, alpha = O.ksvd_dictionary_update(code, D0)
        assert np.allclose(D1, z['k%d_D1' % i], atol=1e-10)
        r, c, v = coo_sorted(code1)
        keep = z['k%d_code1_v' % i] != 0.0       # the reference's CSC keeps explicit zeros (hsc/modeling.py:603)
        assert r.tolist() == z['k%d_code1_t' % i][keep].tolist()
        assert c.tolist() == z['k%d_code1_k' % i][keep].tolist()
        assert np.allclose(v, z['k%d_code1_v' % i][keep], atol=1e-10)
        assert alpha > 0


def test_ksvd_update_pca_matches_reference():
    """usePCA=True (hsc/modeling.py:618-625, pca :48-80): fixture recorded from the reference's own statements."""
    z = load_npz('ksvd_update_pca.npz')
    for i in range(int(z['count'])):
        D0 = z['k%d_D0' % i]
        T = z['k%d_x' % i].shape[0]
        code = scipy.sparse.coo_matrix((z['k%d_code_v' % i], (z['k%d_code_t' % i], z['k%d_code_k' % i])),
                                       shape=(T, D0.shape[0])).tocsc()
        D1, code1, alpha = O.ksvd_dictionary_update(code, D0, use_pca=True)
        assert np.allclose(D1, z['k%d_D1' % i], atol=1e-10)
        r, c, v = coo_sorted(code1)
        keep = z['k%d_code1_v' % i] != 0.0
        assert r.tolist() == z['k%d_code1_t' % i][keep].tolist()
        assert c.tolist() == z['k%d_code1_k' % i][keep].tolist()
        assert np.allclose(v, z['k%d_code1_v' % i][keep], atol=1e-10)
        assert alpha > 0


# ---------------- stored random cases, and the live reference where a copy is supplied ----------

def test_oracle_equals_live_reference_bit_for_bit():
    """24 small random MP / LoCOMP cases (tests/golden/oracle_trials.npz, make_golden_dropin.py): the oracle returns
    exactly the stored codes and residuals; where a copy of the reference is supplied, so does the reference."""
    z = load_npz('oracle_trials.npz')
    live = None
    if HAVE_REF:
        ref_loader.load_reference()
        from hsc.modeling import ConvolutionalMatchingPursuit, LoCOMP
        import logging
        logging.getLogger('hsc').setLevel(logging.ERROR)
        live = {'cmp': ConvolutionalMatchingPursuit, 'locomp': LoCOMP}
    assert int(z['count']) == 24
    for trial in range(int(z['count'])):
        name = 'trial%d' % trial
        x, D, kw = z[name + '_x'], z[name + '_D'], case_kwargs(z, name)
        for method, fn in (('cmp', O.mp_encode), ('locomp', O.locomp_encode)):
            key = '%s_%s' % (name, method)
            c_st, r_st = stored_code(z, key), z[key + '_res']
            outs = [fn(x, D, **kw)] + ([live[method]().computeCoefficients(x, D, **kw)] if live else [])
            for c, r in outs:
                assert all(np.array_equal(a, b) for a, b in zip(coo_sorted(c), coo_sorted(c_st))), (key, kw)
                assert r.dtype == r_st.dtype and r.shape == r_st.shape and np.array_equal(r, r_st), (key, kw)


def test_kmeans_oracle_matches_reference_golden():
    """oracle.kmeans_train replays ConvolutionalDictionaryLearner(algorithm='kmean').train of the reference
    (hsc/modeling.py:420-526) under the same np.random seed: fixtures recorded by tests/golden/make_golden_kmeans.py,
    including the window-0 quirk of the reference's empty-centroid test (:479-481)."""
    import ast
    z = np.load(os.path.join(GOLDEN, 'kmeans.npz'), allow_pickle=False)
    for i in range(int(z['count'])):
        data = z['m%d_data' % i]
        k, W, nb, seed, iters = [int(v) for v in z['m%d_par' % i]]
        kw = ast.literal_eval(str(z['m%d_kw' % i]))
        for it in (1, iters):
            np.random.seed(seed)
            D, hist = O.kmeans_train(data, k, W, nb, maxIterations=it, **kw)
            ref = z['m%d_D_it%d' % (i, it)]
            assert D.shape == ref.shape and D.dtype == ref.dtype, (i, it)
            assert np.array_equal(D, ref), (i, it, np.abs(D - ref).max())
    # the window-0 cases do reset a centroid that owns window 0 alone
    i = int(z['window0_case_first'])
    data = z['m%d_data' % i]
    k, W, nb, seed, iters = [int(v) for v in z['m%d_par' % i]]
    np.random.seed(seed)
    lo = np.random.randint(low=0, high=data.shape[0] - 2 * W, size=(nb,))
    windows = np.stack([data[j:j + 2 * W] for j in lo])
    i0 = np.random.randint(low=0, high=data.shape[0] - W, size=(k,))
    D0 = O.normalize(np.stack([data[j:j + W] for j in i0]))
    pos, idx, _ = O.kmeans_assign(windows, D0)
    assert np.sum(idx == idx[0]) == 1
    _, _, resets, _, _ = O.kmeans_iteration(windows, D0)
    assert resets == (k - len(np.unique(idx))) + 1          # the empty centroids AND the one that owns only window 0


def test_converters_oracle_matches_reference_golden():
    z = np.load(os.path.join(GOLDEN, 'converters.npz'), allow_pickle=False)
    T, counts = int(z['T']), [int(c) for c in z['counts']]
    codes = [scipy.sparse.coo_matrix((z['code%d_v' % l], (z['code%d_t' % l], z['code%d_k' % l])), shape=(T, K)).tocsr() for l, K in enumerate(counts)]
    ev = O.sparse_matrices_to_events(codes)
    assert ev.dtype == O.EVENT_DTYPE
    assert np.array_equal(np.stack([ev['f0'], ev['f1'], ev['f2']], axis=1), z['events']) and np.array_equal(ev['f3'], z['events_v'])
    back = O.events_to_sparse_matrices(ev, counts, T)
    for l, m in enumerate(back):
        c = m.tocoo()
        assert m.format == 'csr' and np.array_equal(c.row, z['back%d_t' % l]) and np.array_equal(c.col, z['back%d_k' % l]) and np.array_equal(c.data, z['back%d_v' % l])
