"""Expected outputs of the drop-in tests (tests/test_dropin_reference_gpu.py) and of the oracle's bit-for-bit check
against the reference (tests/test_oracle_golden.py), stored so that both run from the repository alone.

    python tests/golden/make_golden_dropin.py

Writes `tests/golden/dropin.npz` and `tests/golden/oracle_trials.npz`: the inputs of every case and what the
reference returns for them, computed with oracle/hsc_oracle.py, the NumPy restatement of the reference that
tests/test_oracle_golden.py pins to vectors recorded from the unmodified reference.  Where a copy of the reference is
supplied (HSC_REFERENCE_ROOT or baseline/_ref), the two tests also run the reference itself and check that it returns
exactly these stored values.

    coder_<i>_{mp_nnz,mp_snr,locomp}   ConvolutionalSparseCoder.encode, three shapes (F = 1, 4, 3; float32 and float64),
                                       stop on nbNonzeroCoefs or toleranceSnr=25 (MP) and on nbNonzeroCoefs (LoCOMP)
    hier_*                             HierarchicalConvolutionalSparseCoder.encode of config 3's dictionaries on its signal[:6000]
    ksvd_<method>_*                    ConvolutionalDictionaryLearner(algorithm='ksvd').train, 3 iterations from the
                                       reference's np.random initialisation (seed 5)
    trial<i>_<cmp|locomp>_*            24 small random cases of computeCoefficients (MP and LoCOMP)
"""
import os
import sys

import numpy as np
import scipy.sparse

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
from oracle import hsc_oracle as O  # noqa: E402
from helpers import coo_sorted, load_npz  # noqa: E402

CODER_SHAPES = ((3000, 12, 16, 1, 60, np.float32), (2048, 16, 32, 4, 40, np.float32), (1500, 8, 9, 3, 30, np.float64))
CODER_RUNS = (('mp_nnz', 'cmp', 'nbNonzeroCoefs'), ('mp_snr', 'cmp', 'toleranceSnr'), ('locomp', 'locomp', 'nbNonzeroCoefs'))
HIER_KW = dict(toleranceSnr=10.0, nbBlocks=1, singletonWeight=0.95, returnDistributed=True)
HIER_T = 6000
KSVD = dict(K=6, L=12, T=1500, n=60, seed=5, maxIterations=3, nbNonzeroCoefs=40, toleranceSnr=30.0)


def coder_kwargs(stop, n):
    return dict(nbNonzeroCoefs=n) if stop == 'nbNonzeroCoefs' else dict(toleranceSnr=25.0)


def put_code(d, key, code):
    t, k, v = coo_sorted(code)
    d[key + '_t'], d[key + '_k'], d[key + '_v'] = t, k, v
    d[key + '_shape'] = np.array(code.shape, np.int64)


def coder_cases(d):
    rs = np.random.RandomState(3)
    for i, (T, K, L, F, n, dtype) in enumerate(CODER_SHAPES):
        D = O.normalize(rs.randn(K, L, F)).astype(dtype)
        planted = scipy.sparse.coo_matrix((rs.uniform(0.25, 4.0, n) * rs.choice([-1.0, 1.0], n), (rs.randint(0, T, n), rs.randint(0, K, n))),
                                          shape=(T, K)).tocsc()
        if F == 1:
            D = D[:, :, 0]
        x = O.reconstruct(planted, D).astype(dtype)
        d['coder%d_x' % i], d['coder%d_D' % i], d['coder%d_n' % i] = x, D, np.array(n)
        for tag, method, stop in CODER_RUNS:
            enc = O.mp_encode if method == 'cmp' else O.locomp_encode
            code, res = enc(x, D, **coder_kwargs(stop, n))
            put_code(d, 'coder%d_%s' % (i, tag), code)
            d['coder%d_%s_res' % (i, tag)] = res
            if method == 'cmp':
                d['coder%d_%s_decoded' % (i, tag)] = O.reconstruct(code, D)


def hierarchical_case(d):
    z = load_npz('c3_complex.npz')
    nl = int(z['nb_levels'])
    raw = [z['raw_l%d' % i] for i in range(nl)]
    rep = [z['rep_l%d' % i] for i in range(nl)]
    x = z['x'][:HIER_T]
    codes, res = O.hierarchical_encode(x, raw, z['counts_no_singletons'], rep, method='cmp', **HIER_KW)
    for l, c in enumerate(codes):
        put_code(d, 'hier_l%d' % l, c)
    d['hier_res'] = res


def ksvd_train(x, method, p):
    """_train_ksvd of the reference (hsc/modeling.py:528-641) without initD: the 'noise' initialisation (:554, :320-321),
    then per iteration the encode and the dictionary update, until maxIterations or alpha <= tolerance (0)."""
    np.random.seed(p['seed'])
    D = O.normalize(np.random.uniform(low=np.min(x), high=np.max(x), size=(p['K'], p['L'], 1)))[:, :, 0]
    enc = O.mp_encode if method == 'cmp' else O.locomp_encode
    n, alpha = 0, 1.0
    while n < p['maxIterations'] and alpha > 0.0:
        code, _ = enc(x, D, nbNonzeroCoefs=p['nbNonzeroCoefs'], toleranceSnr=p['toleranceSnr'])
        D, _, alpha = O.ksvd_dictionary_update(code, D)
        n += 1
    return D


def ksvd_cases(d):
    p = KSVD
    rs = np.random.RandomState(8)
    Dt = O.normalize(rs.randn(p['K'], p['L']))
    planted = scipy.sparse.coo_matrix((rs.uniform(0.5, 2.0, p['n']), (rs.randint(0, p['T'], p['n']), rs.randint(0, p['K'], p['n']))),
                                      shape=(p['T'], p['K'])).tocsc()
    x = O.reconstruct(planted, Dt)
    d['ksvd_x'] = x
    for method in ('cmp', 'locomp'):
        d['ksvd_%s_D' % method] = ksvd_train(x, method, p)


def oracle_trials(d):
    rs = np.random.RandomState(31337)
    for trial in range(24):
        T = int(rs.choice([57, 130, 300]))
        L = int(rs.choice([3, 4, 7]))            # edge-dominated tiny cases can cycle forever in the reference
        K = int(rs.choice([3, 8]))
        F = int(rs.choice([1, 2, 5]))
        dtype = rs.choice([np.float32, np.float64])
        x = rs.randn(T, F).astype(dtype)
        D = O.normalize(rs.randn(K, L, F)).astype(dtype)
        if F == 1 and trial % 2 == 0:
            x, D = x[:, 0], D[:, :, 0]
        kw = [dict(nbNonzeroCoefs=12), dict(toleranceSnr=9.0, nbNonzeroCoefs=60), dict(toleranceSnr=6.0, nbBlocks=4, nbNonzeroCoefs=60),
              dict(toleranceResidualScale=0.8, nbNonzeroCoefs=30), dict(toleranceSnr=7.0, nbBlocks="auto", nbNonzeroCoefs=40)][trial % 5]
        if trial % 3 == 0:
            kw['weights'] = np.where(np.arange(K) < max(K // 2, 1), 0.7, 1.0).astype(dtype)
        name = 'trial%d' % trial
        d[name + '_x'], d[name + '_D'] = x, D
        d[name + '_kw'] = np.array(repr({k: (v.tolist() if isinstance(v, np.ndarray) else v) for k, v in kw.items()}))
        for method, fn in (('cmp', O.mp_encode), ('locomp', O.locomp_encode)):
            code, res = fn(x, D, **kw)
            put_code(d, '%s_%s' % (name, method), code)
            d['%s_%s_res' % (name, method)] = res
    d['count'] = np.array(24)


if __name__ == '__main__':
    import warnings
    warnings.simplefilter('ignore')
    d = {}
    coder_cases(d)
    hierarchical_case(d)
    ksvd_cases(d)
    np.savez_compressed(os.path.join(HERE, 'dropin.npz'), **d)
    d = {}
    oracle_trials(d)
    np.savez_compressed(os.path.join(HERE, 'oracle_trials.npz'), **d)
    for f in ('dropin.npz', 'oracle_trials.npz'):
        print('%s: %.0f kB' % (f, os.path.getsize(os.path.join(HERE, f)) / 1e3))
