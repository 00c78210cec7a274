"""Drop-in proof (INTEGRATION.md section 1): the B200 approximators, composed the way the reference composes its own,
return what the reference returns.

The reference injects a sparse approximator by composition - ConvolutionalSparseCoder(D, approximator)
(hsc/modeling.py:1656-1669), HierarchicalConvolutionalSparseCoder(multilevelDict, approximator) (:1671-1705) - and its
K-SVD learner constructs one by name (:580-589).  Every test compares this package's coder / learner classes, driving the
B200 approximators, with the reference's outputs stored in tests/golden/dropin.npz (tests/golden/make_golden_dropin.py).
Where a copy of the unmodified reference is supplied (HSC_REFERENCE_ROOT or baseline/_ref, read through the Python-2
import hook tests/golden/ref_loader.py), each test also checks that the reference returns exactly the stored outputs and
runs the reference's OWN classes with this package's approximators.
"""
import os
import sys

import numpy as np
import pytest
import scipy.sparse

from helpers import load_npz, snr_db, code_diff, coo_sorted, stored_code

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden'))
import ref_loader  # noqa: E402
from make_golden_dropin import CODER_RUNS, HIER_KW, KSVD, coder_kwargs  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def ref():
    """The reference package where a copy is supplied, else None (the tests then compare with the stored outputs only)."""
    if not ref_loader.reference_available():
        return None
    import logging
    import warnings
    warnings.simplefilter('ignore')
    mod = ref_loader.load_reference()
    logging.getLogger('hsc').setLevel(logging.ERROR)
    return mod


@pytest.fixture(scope='module')
def hsc():
    import torch
    assert torch.cuda.is_available()
    import hierarchical_sparse_coding_b200 as pkg
    return pkg


@pytest.fixture(scope='module')
def golden():
    return load_npz('dropin.npz')


def _same_code(a, b):
    return all(np.array_equal(u, v) for u, v in zip(coo_sorted(a), coo_sorted(b)))


def _check_flat(x, c_ref, r_ref, c_got, r_got, rel):
    assert scipy.sparse.issparse(c_got) and c_got.format == 'csc' and c_got.shape == c_ref.shape and c_got.dtype == np.float64
    assert r_got.shape == r_ref.shape and r_got.dtype == r_ref.dtype
    ratio, mism = code_diff(c_ref, c_got, rel=rel)
    assert mism == 0 and ratio <= 1.0, (x.shape, rel, ratio, mism)
    assert abs(snr_db(x, r_ref) - snr_db(x, r_got)) <= 0.01


def test_reference_coder_with_b200_approximator(ref, hsc, golden):
    """ConvolutionalSparseCoder (:1656-1669) with the B200 MP and LoCOMP: encode + reconstruct, three shapes."""
    z = golden
    i = 0
    while 'coder%d_x' % i in z.files:
        x, D, n = z['coder%d_x' % i], z['coder%d_D' % i], int(z['coder%d_n' % i])
        for tag, method, stop in CODER_RUNS:
            key = 'coder%d_%s' % (i, tag)
            kw = coder_kwargs(stop, n)
            c_ref, r_ref = stored_code(z, key), z[key + '_res']
            approx = hsc.ConvolutionalMatchingPursuit if method == 'cmp' else hsc.LoCOMP
            ours = hsc.ConvolutionalSparseCoder(D, approximator=approx())
            c_got, r_got = ours.encode(x, **kw)
            rel = 1e-5 if method == 'cmp' else (2e-4 if x.dtype == np.float32 else 1e-6)
            _check_flat(x, c_ref, r_ref, c_got, r_got, rel)
            if method == 'cmp':
                assert np.allclose(ours.reconstruct(c_got) + r_got, x, atol=1e-5)
                assert np.allclose(hsc.reconstructSignal(c_ref, D), z[key + '_decoded'], atol=1e-6)
            if ref is not None:
                ref_approx = ref.modeling.ConvolutionalMatchingPursuit if method == 'cmp' else ref.modeling.LoCOMP
                c_live, r_live = ref.modeling.ConvolutionalSparseCoder(D, approximator=ref_approx()).encode(x, **kw)
                assert c_live.format == 'csc' and c_live.dtype == np.float64, key
                assert _same_code(c_live, c_ref) and np.array_equal(r_live, r_ref), key
                c_in, r_in = ref.modeling.ConvolutionalSparseCoder(D, approximator=approx()).encode(x, **kw)
                _check_flat(x, c_ref, r_ref, c_in, r_in, rel)
        i += 1
    assert i == 3


def test_reference_hierarchical_coder_with_b200_approximator(ref, hsc, golden):
    """HierarchicalConvolutionalSparseCoder (:1671-1705) over a MultilevelDictionary (hsc/dataset.py:110), approximator =
    this package's hierarchical MP: config 3's dictionaries and the first 6000 samples of its signal."""
    z = golden
    z3 = load_npz('c3_complex.npz')
    nl = int(z3['nb_levels'])
    raw = [z3['raw_l%d' % i] for i in range(nl)]
    rep = [z3['rep_l%d' % i] for i in range(nl)]
    scales = [int(v) for v in z3['scales']]
    r_ref = z['hier_res']
    x = z3['x'][:len(r_ref)]
    c_ref = [stored_code(z, 'hier_l%d' % l) for l in range(nl)]

    def check(c_got, r_got):
        assert len(c_got) == nl
        assert abs(snr_db(x, r_ref) - snr_db(x, r_got)) <= 0.01
        for l in range(nl):
            assert c_got[l].shape == c_ref[l].shape
            ratio, mism = code_diff(c_ref[l], c_got[l], rel=1e-5)
            assert mism == 0 and ratio <= 1.0, (l, ratio, mism, c_ref[l].nnz, c_got[l].nnz)

    mld = hsc.MultilevelDictionary(raw, scales, rep, z3['counts_no_singletons'], hasSingletonBases=True)
    ours = hsc.HierarchicalConvolutionalSparseCoder(mld, hsc.HierarchicalConvolutionalMatchingPursuit(method='cmp'))
    c_got, r_got = ours.encode(x, **HIER_KW)
    check(c_got, r_got)
    assert np.allclose(ours.reconstruct(c_got) + r_got, x, atol=1e-5)
    if ref is not None:
        rmld = ref.dataset.MultilevelDictionary(raw, scales, rep, None, hasSingletonBases=True)
        assert np.array_equal(rmld.countsNoSingletons, z3['counts_no_singletons'])
        c_live, r_live = ref.modeling.HierarchicalConvolutionalSparseCoder(
            rmld, ref.modeling.HierarchicalConvolutionalMatchingPursuit(method='cmp')).encode(x, **HIER_KW)
        for l in range(nl):        # the oracle's tolerance against the reference (tests/test_oracle_golden.py, config 3)
            t, k, v = coo_sorted(c_live[l])
            tr, kr, vr = coo_sorted(c_ref[l])
            assert np.array_equal(t, tr) and np.array_equal(k, kr) and np.allclose(v, vr, rtol=1e-10, atol=0), l
        assert np.allclose(r_live, r_ref, rtol=0, atol=1e-12)
        check(*ref.modeling.HierarchicalConvolutionalSparseCoder(
            rmld, hsc.HierarchicalConvolutionalMatchingPursuit(method='cmp')).encode(x, **HIER_KW))


def test_reference_ksvd_loop_with_b200_inference(ref, hsc, golden, monkeypatch):
    """_train_ksvd (:528-641) from the reference's np.random initialisation (no initD) learns the reference's dictionary
    with B200 inference: this package's learner, and - with a copy of the reference - the reference's own loop with its
    approximator names bound to this package's classes (the one-line change INTEGRATION.md shows)."""
    z = golden
    x = z['ksvd_x']
    p = KSVD
    kw = dict(maxIterations=p['maxIterations'], nbNonzeroCoefs=p['nbNonzeroCoefs'], toleranceSnr=p['toleranceSnr'])

    def same_up_to_sign(D_got, D_ref, atol):
        # the sign of a singular pair is LAPACK's choice inside the dictionary update (:627-633): compare up to it
        assert D_got.shape == D_ref.shape
        sgn = np.sign(np.sum(D_got * D_ref, axis=1))[:, None]
        assert np.allclose(D_got * sgn, D_ref, atol=atol), float(np.abs(D_got * sgn - D_ref).max())

    for method in ('cmp', 'locomp'):
        D_ref = z['ksvd_%s_D' % method]
        np.random.seed(p['seed'])
        same_up_to_sign(hsc.ConvolutionalDictionaryLearner(p['K'], p['L'], algorithm='ksvd').train(x, method=method, **kw), D_ref, 1e-6)
        if ref is not None:
            np.random.seed(p['seed'])
            same_up_to_sign(ref.modeling.ConvolutionalDictionaryLearner(p['K'], p['L'], algorithm='ksvd').train(x, method=method, **kw),
                            D_ref, 1e-10)
            with monkeypatch.context() as m:
                m.setattr(ref.modeling, 'ConvolutionalMatchingPursuit', hsc.ConvolutionalMatchingPursuit)
                m.setattr(ref.modeling, 'LoCOMP', hsc.LoCOMP)
                np.random.seed(p['seed'])
                same_up_to_sign(ref.modeling.ConvolutionalDictionaryLearner(p['K'], p['L'], algorithm='ksvd').train(x, method=method, **kw),
                                D_ref, 1e-6)
