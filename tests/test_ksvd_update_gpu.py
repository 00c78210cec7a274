"""The K-SVD dictionary update (csrc/ksvd.cuh) against a float64 sweep, at every eigen-solver path, window size and
spectral gap.

  * Eigen-solver contract, through the per-filter sweep API: between `_filter_gram` and `_filter_finish` the caller-owned
    Gram buffer is overwritten with a designed symmetric PSD matrix (what the all-reduce of data-parallel learning does),
    so `_finish` must return its dominant eigenvector: unit norm, <u, d_old> >= 0, ||u - v1|| <= c q eps / g where that
    bound is below 1e-6, and for every spectrum ||C u - (u'Cu) u|| <= c q eps lambda1 and u'Cu >= lambda1 (1 - c q eps).
    The Gram kernel and the projection kernel are compared with float64 on the way.  Which path ran is read from the
    engine's launch counter across `_filter_finish`: 2 launches on the cluster-chained path (q <= 64), 1 + 30 + 1 with the
    separate kernels (30 squaring launches, of which those after the power became rank one return at once).
  * Whole-sweep parity of `Engine.ksvd_update` (the learner's path) on designed codes, with and without PCA and at
    coefficient amplitudes 2^+-200; tolerances follow the reference's per-filter eigenvalue gap.
  * One engine through sweeps of one shape whose code size changes (re-capture of the CUDA graph) and whose PCA switch
    flips, eagerly, from a graph and by default.
  * The sweep API with the internal Gram buffer against `ksvd_update`, `skip`, and the error codes.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import hierarchical_sparse_coding_b200._native as N

EPS = 2.0 ** -52
C_BOUND = 32.0                     # the constant c of the eigen-solver contract
Q_LIST = (1, 2, 15, 16, 17, 63, 64, 65, 128, 256, 891, 892, 1024, 3072)
LF_OF_Q = {1: (1, 1), 2: (2, 1), 15: (5, 3), 16: (4, 4), 17: (17, 1), 63: (21, 3), 64: (16, 4), 65: (65, 1),
           128: (32, 4), 256: (64, 4), 891: (297, 3), 892: (223, 4), 1024: (256, 4), 3072: (768, 4)}
GAPS = (1e-1, 1e-2, 1e-3, 1e-4, 1e-6, 1e-8)
CHAIN_MAX_Q = 64                   # kPowerSmallQ: the cluster-chained eigen-solver serves q <= 64
SEPARATE_FINISH_LAUNCHES = 1 + 30 + 1       # kMaxSquarings squaring launches + power kernel + projection


# ------------------------------------------------------------------ float64 reference of one sweep

def centre_offset(L):
    """Centre tap (include/hsc_b200.h): L/2-1 for even L, L/2 for odd L."""
    return L // 2 - 1 if L % 2 == 0 else L // 2


def decode64(D, sig, pos, idx, coef, S, T):
    """float64 decode of a code of S signals into a buffer padded by L zeros on both sides: [S, T + 2L, F]."""
    K, L, F = D.shape
    off = centre_offset(L)
    R = np.zeros((S, T + 2 * L, F))
    for j in range(L):
        np.add.at(R, (sig, pos - off + j + L), coef[:, None] * D[idx, j])
    R[:, :L] = 0.0
    R[:, L + T:] = 0.0                           # nothing outside the signal
    return R


def windows64(R, sig, pos, L, F):
    """The length-L windows centred at the atoms, zero outside the signal: [n, L*F]."""
    t = pos[:, None] - centre_offset(L) + np.arange(L)[None, :] + L
    return R[sig[:, None], t].reshape(len(sig), L * F)


def ref_sweep(D0, sig, pos, idx, coef0, S, T, use_pca=False):
    """One Gauss-Seidel sweep over the filters with at least one atom: the decode without filter k from scratch, its
    windows (mean-centred with PCA when n >= 2), the dominant right singular vector of W (= eigenvector of W^T W, from
    the SVD of W itself), the sign <u, d_old> >= 0, e_0 for all-zero windows, coefficients W u.  Returns (D, coef,
    alpha, info) with info[k] = dict(lam1, lam2, gap, W) or None for a filter without atoms."""
    D = np.array(D0, np.float64, copy=True)
    coef = np.array(coef0, np.float64, copy=True)
    K, L, F = D.shape
    q = L * F
    info = [None] * K
    for k in range(K):
        sel = np.nonzero(idx == k)[0]
        if len(sel) == 0:
            continue
        o = idx != k
        W = windows64(decode64(D, sig[o], pos[o], idx[o], coef[o], S, T), sig[sel], pos[sel], L, F)
        if use_pca and len(sel) >= 2:
            W = W - W.mean(axis=0)
        _, sv, Vt = np.linalg.svd(W, full_matrices=False)
        lam = sv ** 2
        if lam[0] == 0.0:
            v = np.zeros(q)
            v[0] = 1.0
        else:
            v = Vt[0] if Vt[0] @ D[k].ravel() >= 0 else -Vt[0]
        D[k] = v.reshape(L, F)
        coef[sel] = W @ v
        lam2 = lam[1] if len(lam) > 1 else 0.0
        info[k] = dict(lam1=lam[0], lam2=lam2, gap=(lam[0] - lam2) / lam[0] if lam[0] > 0 else 0.0, W=W)
    return D, coef, float(np.sqrt(np.sum((D - D0) ** 2))), info


def unit_dictionary(rs, K, L, F):
    D = rs.randn(K, L, F)
    return D / np.sqrt(np.sum(D * D, axis=(1, 2), keepdims=True))


def sort_code(sig, pos, idx, coef):
    """Unique (filter, signal, position) entries in that order, the layout the update takes, plus col_ptr."""
    key = (idx.astype(np.int64) * (1 << 20) + sig) * (1 << 24) + pos
    _, first = np.unique(key, return_index=True)
    sig, pos, idx, coef = sig[first], pos[first], idx[first], coef[first]
    order = np.lexsort((pos, sig, idx))
    return sig[order], pos[order], idx[order], coef[order]


def col_ptr_of(idx, K):
    return np.concatenate([[0], np.cumsum(np.bincount(idx, minlength=K))]).astype(np.int64)


# ------------------------------------------------------------------ engine plumbing

@pytest.fixture(scope='module')
def eng():
    import torch
    assert torch.cuda.is_available(), 'gpu tests need a CUDA device'
    from hierarchical_sparse_coding_b200.engine import Engine
    e = Engine(0)
    yield e
    e.close()


def to_dev(eng, sig, pos, idx, coef):
    import torch
    dv = eng.device
    return (torch.from_numpy(np.ascontiguousarray(sig, np.int32)).to(dv), torch.from_numpy(np.ascontiguousarray(pos, np.int32)).to(dv),
            torch.from_numpy(np.ascontiguousarray(idx, np.int32)).to(dv), torch.from_numpy(np.ascontiguousarray(coef, np.float64)).to(dv))


def vp(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def sweep_begin(eng, Dd, cp, code, S, T, gram=None):
    """hsc_b200_ksvd_begin; returns (rc, sweep handle).  cp: numpy int64 [K+1]; code: device (sig, pos, idx, coef)."""
    K, L, F = Dd.shape
    sweep = ctypes.c_void_p()
    cpp = cp.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))
    rc = eng.lib.hsc_b200_ksvd_begin(eng.handle, vp(Dd), K, L, F, cpp, vp(code[0]), vp(code[1]), vp(code[2]), vp(code[3]),
                                     int(S), int(T), vp(gram), eng._stream_ptr(), ctypes.byref(sweep))
    return rc, sweep


def sweep_end(eng, sweep):
    alpha = ctypes.c_double(0.0)
    N.check(eng.lib, eng.handle, eng.lib.hsc_b200_ksvd_end(sweep, ctypes.byref(alpha)))
    return alpha.value


# ------------------------------------------------------------------ 1. eigen-solver contract through the sweep API

def designed_spectra(q, rs):
    """(name, eigenvalues in descending order, relative gap of the top two or None) of the designed Gram matrices."""
    rest = lambda m: np.sort(rs.uniform(0.0, 0.5, m))[::-1]
    out = [('separated', np.concatenate([[1.0], rest(q - 1)]), 0.5 if q > 1 else None)]
    if q >= 2:
        out += [('gap%.0e' % g, np.concatenate([[1.0, 1.0 - g], rest(q - 2)]), g) for g in GAPS]
        out.append(('double', np.concatenate([[1.0, 1.0], rest(q - 2)]), None))
    if q >= 3:
        out.append(('triple', np.concatenate([[1.0, 1.0, 1.0], rest(q - 3)]), None))
    out.append(('rank1', np.concatenate([[1.0], np.zeros(q - 1)]), 1.0 if q > 1 else None))
    out.append(('zero', np.zeros(q), None))
    out.append(('to1e-300', np.logspace(0.0, -300.0, q) if q > 1 else np.ones(1), None))
    sep = out[0][1]
    out.append(('scaled2^400', sep * 2.0 ** 400, 0.5 if q > 1 else None))
    out.append(('scaled2^-400', sep * 2.0 ** -400, 0.5 if q > 1 else None))
    return out


def eigen_contract(eng, q, chain_on, seed=0):
    """Runs every designed spectrum at window size q through begin / gram / (overwrite) / finish / end and checks the
    contract.  Returns a list of report lines."""
    import torch
    rs = np.random.RandomState(1000 + q)
    L, F = LF_OF_Q[q]
    S, T, K = 2, 3 * L + 40, 2
    # filter 1 makes the signal, filter 0 is updated: its windows are the decode of filter 1 (edge atoms included)
    D0 = unit_dictionary(rs, K, L, F)
    n1 = 6
    s1 = rs.randint(0, S, n1)
    p1 = rs.randint(0, T, n1)
    s0 = np.array([0, 0, 1, 1, 0])
    p0 = np.array([0, T - 1, rs.randint(0, L), T - 1 - rs.randint(0, L), T // 2])
    sig, pos, idx, coef = sort_code(np.concatenate([s0, s1]), np.concatenate([p0, p1]), np.concatenate([np.zeros(5, int), np.ones(n1, int)]),
                                    rs.uniform(0.5, 2.0, 5 + n1) * rs.choice([-1.0, 1.0], 5 + n1))
    cp = col_ptr_of(idx, K)
    o = idx != 0
    W_ref = windows64(decode64(D0, sig[o], pos[o], idx[o], coef[o], S, T), sig[~o], pos[~o], L, F)
    # |every atom| on the windows: the engine removes filter 0's atoms from the decode of the whole code, which leaves
    # up to 2 eps of it in each window entry
    W_abs = windows64(decode64(np.abs(D0), sig, pos, idx, np.abs(coef), S, T), sig[~o], pos[~o], L, F)
    nrm_w = np.sqrt(np.sum(W_abs ** 2, axis=1))
    Q, _ = np.linalg.qr(rs.randn(q, q))
    v1 = Q[:, 0]
    code = to_dev(eng, sig, pos, idx, coef)
    gram = torch.empty((q, q), dtype=torch.float64, device=eng.device)
    want_launches = 2 if (chain_on and q <= CHAIN_MAX_Q) else SEPARATE_FINISH_LAUNCHES
    report = []
    launch_counts = set()
    for si, (name, lam, g) in enumerate(designed_spectra(q, rs)):
        C = (Q * lam) @ Q.T
        C = 0.5 * (C + C.T)
        # old filter: along v1, against it, or exactly orthogonal to it
        mode = si % 3
        if mode == 0:
            d_old = v1 + 0.3 * rs.randn(q) / np.sqrt(q)
        elif mode == 1:
            d_old = -v1 + 0.3 * rs.randn(q) / np.sqrt(q)
        else:
            d_old = Q[:, 1] if q > 1 else np.ones(1)
        d_old = d_old / np.linalg.norm(d_old)
        D = D0.copy()
        D[0] = d_old.reshape(L, F)
        Dd = torch.from_numpy(D).to(eng.device)
        cf = code[3].clone()
        rc, sweep = sweep_begin(eng, Dd, cp, (code[0], code[1], code[2], cf), S, T, gram)
        N.check(eng.lib, eng.handle, rc)
        try:
            N.check(eng.lib, eng.handle, eng.lib.hsc_b200_ksvd_filter_gram(sweep, 0, None))
            G = gram.cpu().numpy()
            # Gram kernel: W^T W within (n + 4) eps sum |w_a| |w_b|
            bound = (len(W_ref) + 4) * EPS * (W_abs.T @ W_abs) + 1e-300
            assert np.all(np.abs(G - W_ref.T @ W_ref) <= bound), (q, name, np.max(np.abs(G - W_ref.T @ W_ref) / bound))
            gram.copy_(torch.from_numpy(C))
            l0 = eng.launches
            N.check(eng.lib, eng.handle, eng.lib.hsc_b200_ksvd_filter_finish(sweep, 0, 0))
            launched = eng.launches - l0
        finally:
            sweep_end(eng, sweep)
        launch_counts.add(launched)
        u = Dd.cpu().numpy()[0].ravel()
        c_new = cf.cpu().numpy()[:cp[1]]
        # projection kernel: coefficients = W_ref u within (q + 4) ulp of ||w_i||
        assert np.all(np.abs(c_new - W_ref @ u) <= (q + 4) * EPS * nrm_w + 1e-300), (q, name)
        if name == 'zero':
            want = np.zeros(q)
            want[0] = 1.0
            assert np.array_equal(u, want), (q, u[:4])
            report.append('q=%d %-12s e0' % (q, name))
            continue
        assert abs(np.linalg.norm(u) - 1.0) <= 1e-14, (q, name, np.linalg.norm(u) - 1.0)
        dot = float(u @ d_old)
        assert dot >= (-C_BOUND * q * EPS if mode == 2 else 0.0), (q, name, mode, dot)
        lam1 = float(lam[0])
        Cu = C @ u
        rq = float(u @ Cu)
        res = float(np.linalg.norm(Cu - rq * u))
        assert res <= C_BOUND * q * EPS * lam1, (q, name, res / (q * EPS * lam1))
        assert rq >= lam1 * (1.0 - C_BOUND * q * EPS), (q, name, 1.0 - rq / lam1)
        err = min(np.linalg.norm(u - v1), np.linalg.norm(u + v1))
        line = 'q=%d %-12s residual %.1f q eps lam1, |u-v1| %.2e' % (q, name, res / (q * EPS * lam1), err)
        if g is not None and C_BOUND * q * EPS / g < 1e-6:
            assert err <= C_BOUND * q * EPS / g, (q, name, err, C_BOUND * q * EPS / g)
            line += ' (bound %.1e)' % (C_BOUND * q * EPS / g)
        report.append(line)
    assert launch_counts == {want_launches}, (q, launch_counts, want_launches)       # the eigen-solver path that ran
    return report


@pytest.mark.gpu
@pytest.mark.parametrize('q', Q_LIST)
def test_eigen_solver_contract(eng, q):
    for line in eigen_contract(eng, q, chain_on=True):
        print(line)


_SEPARATE_SCRIPT = r'''
import sys
sys.path.insert(0, %(root)r)
sys.path.insert(0, %(tests)r)
import test_ksvd_update_gpu as t
from hierarchical_sparse_coding_b200.engine import Engine
e = Engine(0)
for q in t.Q_LIST:
    for line in t.eigen_contract(e, q, chain_on=False):
        print(line)
e.close()
print('separate kernels ok')
'''


def run_variant(script, env):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    e = dict(os.environ)
    e.update(env)
    p = subprocess.run([sys.executable, '-c', script % dict(root=root, tests=os.path.join(root, 'tests'))], env=e, timeout=900,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    print(p.stdout[-4000:])
    assert p.returncode == 0, p.stdout[-4000:]


@pytest.mark.gpu
def test_eigen_solver_contract_separate_kernels():
    """The same contract with HSC_KSVD_CHAIN=0 (read once per process): square_kernel + power kernels at every q."""
    run_variant(_SEPARATE_SCRIPT, {'HSC_KSVD_CHAIN': '0'})


# ------------------------------------------------------------------ 2. whole-sweep parity of Engine.ksvd_update

def designed_code(rs, S, T, K, L, F, empty=None, single=None, isolated=False, n_per=None):
    """Random atoms per filter plus: atoms within the first and last L samples of every signal, three adjacent atoms of
    filter 0 in signal 0, filter `empty` without atoms, filter `single` with one.  isolated: non-overlapping atoms only."""
    sig, pos, idx = [], [], []
    live = [k for k in range(K) if k != empty and k != single]
    if isolated:
        for s in range(S):
            p = np.arange(rs.randint(0, L), T, L + 1 + rs.randint(0, 3))
            sig += [s] * len(p)
            pos += list(p)
            idx += list(rs.choice(live, len(p)))
    else:
        n_per = n_per or max(4, (S * T) // (L * K))
        for k in live:
            sig += list(rs.randint(0, S, n_per))
            pos += list(rs.randint(0, T, n_per))
            idx += [k] * n_per
        for s in range(S):
            sig += [s, s, s, s]
            pos += [0, rs.randint(0, L), T - 1, T - 1 - rs.randint(0, L)]
            idx += list(rs.choice(live, 4))
        p0 = rs.randint(L, T - L - 3)
        sig += [0, 0, 0]
        pos += [p0, p0 + 1, p0 + 2]
        idx += [live[0]] * 3
    if single is not None:
        sig.append(rs.randint(0, S))
        pos.append(rs.randint(0, T))
        idx.append(single)
    n = len(sig)
    coef = rs.uniform(0.5, 2.0, n) * rs.choice([-1.0, 1.0], n)
    return sort_code(np.array(sig), np.array(pos), np.array(idx), coef)


def check_sweep(D0, D1, c1, alpha, ref, tag, vec_tol=1e-9):
    """Engine result (D1, c1, alpha) against ref_sweep's.  Filters are compared as vectors while every filter updated
    before them had a relative gap >= 1e-2; after a smaller gap only the Rayleigh quotient is compared."""
    D_ref, c_ref, alpha_ref, info = ref
    K, L, F = D0.shape
    q = L * F
    strict = True
    lo = 0
    gaps = []
    for k in range(K):
        if info[k] is None:
            assert np.array_equal(D1[k], D0[k]), (tag, k)                          # no atoms: the row stays, bit for bit
            continue
        W = info[k]['W']
        n = len(W)
        hi = lo + n
        u = D1[k].ravel()
        if info[k]['lam1'] == 0.0:
            want = np.zeros(q)
            want[0] = 1.0
            assert np.array_equal(u, want) and np.all(c1[lo:hi] == 0.0), (tag, k, u[:4])
            gaps.append('e0')
        else:
            g = info[k]['gap']
            gaps.append('%.2g' % g)
            assert abs(np.linalg.norm(u) - 1.0) <= 1e-14, (tag, k)
            if strict and g >= 1e-2:
                err = np.linalg.norm(u - D_ref[k].ravel())
                assert err <= vec_tol, (tag, k, g, err)
                scale = np.sqrt(np.max(np.sum(W ** 2, axis=1)))
                assert np.all(np.abs(c1[lo:hi] - c_ref[lo:hi]) <= vec_tol * scale), (tag, k, np.abs(c1[lo:hi] - c_ref[lo:hi]).max() / scale)
            else:
                strict = False
                rq = float(np.sum((W @ u) ** 2))
                assert rq >= info[k]['lam1'] * (1.0 - 1e-9), (tag, k, g, 1.0 - rq / info[k]['lam1'])
        lo = hi
    if strict:
        assert abs(alpha - alpha_ref) <= 1e-9 * max(1.0, alpha_ref), (tag, alpha, alpha_ref)
    print('%s gaps %s' % (tag, ' '.join(gaps)))
    return strict


# (name, S, T, K, L, F, empty filter, single-atom filter, isolated atoms)
SWEEP_CASES = (
    ('q64_S1', 1, 700, 5, 16, 4, 3, 4, False),
    ('q65_oddL_S3', 3, 500, 4, 65, 1, None, 2, False),
    ('q63_oddL_S37', 37, 200, 4, 21, 3, 1, None, False),
    ('q128_S37', 37, 260, 3, 32, 4, None, None, False),
    ('q256_S3', 3, 900, 4, 64, 4, 0, 3, False),
    ('q1024_S1', 1, 2600, 3, 256, 4, None, None, False),
    ('q27_K1_isolated', 2, 300, 1, 9, 3, None, None, True),
    ('q96_isolated_S3', 3, 400, 3, 32, 3, None, None, True),
)


@pytest.mark.gpu
@pytest.mark.parametrize('case', SWEEP_CASES, ids=[c[0] for c in SWEEP_CASES])
def test_ksvd_update_matches_float64_sweep(eng, case):
    name, S, T, K, L, F, empty, single, isolated = case
    rs = np.random.RandomState(sum(map(ord, name)))
    D0 = unit_dictionary(rs, K, L, F)
    sig, pos, idx, coef = designed_code(rs, S, T, K, L, F, empty, single, isolated)
    cp = col_ptr_of(idx, K)
    code = to_dev(eng, sig, pos, idx, coef)
    for use_pca in (False, True):
        ref = ref_sweep(D0, sig, pos, idx, coef, S, T, use_pca)
        D1, c1, alpha = eng.ksvd_update(D0, *code, cp, S, T, use_pca=use_pca)
        strict = check_sweep(D0, D1, c1.cpu().numpy(), alpha, ref, '%s pca=%d' % (name, use_pca))
        # coefficient amplitudes 2^+-200: the same filters, the coefficients scaled
        for e2 in (200, -200):
            s2 = 2.0 ** e2
            D2, c2, _ = eng.ksvd_update(D0, code[0], code[1], code[2], code[3] * s2, cp, S, T, use_pca=use_pca)
            if strict:
                assert np.allclose(D2, D1, rtol=0, atol=1e-12), (name, e2, np.abs(D2 - D1).max())
                c1h = c1.cpu().numpy()
                assert np.allclose(c2.cpu().numpy() / s2, c1h, rtol=0, atol=1e-12 * max(1.0, np.abs(c1h).max())), (name, e2)
    eng.lib.hsc_b200_ksvd_set_pca(eng.handle, 0)


@pytest.mark.gpu
def test_ksvd_update_pca_identical_windows(eng):
    """Two signals holding the same two atoms: filter 0's two windows are identical, so their centred windows are zero
    and the PCA variant must give e_0 with zero coefficients; the plain variant gives the normalised window."""
    S, T, K, L, F = 2, 100, 2, 8, 1
    rs = np.random.RandomState(3)
    D0 = unit_dictionary(rs, K, L, F)
    sig, pos, idx, coef = sort_code(np.array([0, 1, 0, 1]), np.array([50, 50, 52, 52]), np.array([0, 0, 1, 1]), np.array([1.0, 1.0, 0.7, 0.7]))
    cp = col_ptr_of(idx, K)
    code = to_dev(eng, sig, pos, idx, coef)
    for use_pca in (True, False):
        ref = ref_sweep(D0, sig, pos, idx, coef, S, T, use_pca)
        if use_pca:
            assert ref[3][0]['lam1'] == 0.0
        D1, c1, alpha = eng.ksvd_update(D0, *code, cp, S, T, use_pca=use_pca)
        check_sweep(D0, D1, c1.cpu().numpy(), alpha, ref, 'identical windows pca=%d' % use_pca)


# ------------------------------------------------------------------ 3. graph replay and engine state

GRAPH_SHAPE = (3, 600, 4, 16, 4)            # S, T, K, L, F
# (atoms, PCA): capacity 400 + 100 + 1024 from the first sweep; a graph from the third; PCA on and off; 2000 > capacity
GRAPH_SEQUENCE = ((400, False), (300, False), (450, False), (500, False), (420, True), (380, False), (2000, False),
                  (350, False), (1800, False), (330, False))


def graph_sequence(eng):
    S, T, K, L, F = GRAPH_SHAPE
    rs = np.random.RandomState(11)
    out = []
    for i, (n, use_pca) in enumerate(GRAPH_SEQUENCE):
        D0 = unit_dictionary(rs, K, L, F)
        sig, pos, idx, coef = sort_code(rs.randint(0, S, 3 * n), rs.randint(0, T, 3 * n), rs.randint(0, K, 3 * n),
                                        rs.uniform(0.5, 2.0, 3 * n) * rs.choice([-1.0, 1.0], 3 * n))
        keep = rs.permutation(len(sig))[:n]
        sig, pos, idx, coef = sort_code(sig[keep], pos[keep], idx[keep], coef[keep])
        cp = col_ptr_of(idx, K)
        D1, c1, alpha = eng.ksvd_update(D0, *to_dev(eng, sig, pos, idx, coef), cp, S, T, use_pca=use_pca)
        ref = ref_sweep(D0, sig, pos, idx, coef, S, T, use_pca)
        out.append(check_sweep(D0, D1, c1.cpu().numpy(), alpha, ref, 'sweep %d n=%d pca=%d' % (i, n, use_pca)))
    eng.lib.hsc_b200_ksvd_set_pca(eng.handle, 0)
    assert all(out), 'a designed sweep had a filter gap below 1e-2'


@pytest.mark.gpu
def test_ksvd_update_graph_and_state(eng):
    graph_sequence(eng)


_GRAPH_SCRIPT = r'''
import sys
sys.path.insert(0, %(root)r)
sys.path.insert(0, %(tests)r)
import test_ksvd_update_gpu as t
from hierarchical_sparse_coding_b200.engine import Engine
e = Engine(0)
t.graph_sequence(e)
e.close()
print('graph sequence ok')
'''


@pytest.mark.gpu
@pytest.mark.parametrize('mode', ['0', '1'])
def test_ksvd_update_graph_modes(mode):
    """The same sequence never (HSC_KSVD_GRAPH=0) and always (=1) from a CUDA graph."""
    run_variant(_GRAPH_SCRIPT, {'HSC_KSVD_GRAPH': mode})


# ------------------------------------------------------------------ 4. sweep API, skip and error codes

@pytest.mark.gpu
def test_sweep_api_matches_update_and_skip(eng):
    import torch
    S, T, K, L, F = 3, 500, 5, 12, 3
    rs = np.random.RandomState(21)
    D0 = unit_dictionary(rs, K, L, F)
    sig, pos, idx, coef = designed_code(rs, S, T, K, L, F, empty=2, single=4)
    cp = col_ptr_of(idx, K)
    code = to_dev(eng, sig, pos, idx, coef)
    D_up, c_up, alpha_up = eng.ksvd_update(D0, *code, cp, S, T)
    # internal Gram buffer, nothing overwritten: the update's result
    Dd = torch.from_numpy(D0.copy()).to(eng.device)
    cf = code[3].clone()
    rc, sweep = sweep_begin(eng, Dd, cp, (code[0], code[1], code[2], cf), S, T, None)
    N.check(eng.lib, eng.handle, rc)
    for k in range(K):
        if cp[k + 1] == cp[k]:
            continue
        N.check(eng.lib, eng.handle, eng.lib.hsc_b200_ksvd_filter_gram(sweep, k, None))
        N.check(eng.lib, eng.handle, eng.lib.hsc_b200_ksvd_filter_finish(sweep, k, 0))
    alpha = sweep_end(eng, sweep)
    assert np.allclose(Dd.cpu().numpy(), D_up, rtol=0, atol=1e-12)
    assert np.allclose(cf.cpu().numpy(), c_up.cpu().numpy(), rtol=0, atol=1e-12 * np.abs(coef).max())
    assert abs(alpha - alpha_up) <= 1e-12
    # skip = 1 on filter 1: D[1] and its coefficients stay bit for bit, the others are updated
    Dd = torch.from_numpy(D0.copy()).to(eng.device)
    cf = code[3].clone()
    rc, sweep = sweep_begin(eng, Dd, cp, (code[0], code[1], code[2], cf), S, T, None)
    N.check(eng.lib, eng.handle, rc)
    n_local = ctypes.c_int64(-1)
    for k in (0, 1):
        N.check(eng.lib, eng.handle, eng.lib.hsc_b200_ksvd_filter_gram(sweep, k, ctypes.byref(n_local)))
        assert n_local.value == cp[k + 1] - cp[k]
        N.check(eng.lib, eng.handle, eng.lib.hsc_b200_ksvd_filter_finish(sweep, k, 1 if k == 1 else 0))
    sweep_end(eng, sweep)
    D_s, c_s = Dd.cpu().numpy(), cf.cpu().numpy()
    assert np.array_equal(D_s[1], D0[1]) and np.array_equal(c_s[cp[1]:cp[2]], coef[cp[1]:cp[2]])
    assert np.allclose(D_s[0], D_up[0], rtol=0, atol=1e-12) and not np.array_equal(D_s[0], D0[0])
    assert np.array_equal(D_s[2:], D0[2:])


@pytest.mark.gpu
def test_ksvd_error_codes(eng):
    import torch
    S, T, K, L, F = 2, 300, 3, 8, 2
    rs = np.random.RandomState(5)
    D0 = unit_dictionary(rs, K, L, F)
    sig, pos, idx, coef = designed_code(rs, S, T, K, L, F)
    cp = col_ptr_of(idx, K)
    code = to_dev(eng, sig, pos, idx, coef)
    Dd = torch.from_numpy(D0.copy()).to(eng.device)
    rc, sweep = sweep_begin(eng, Dd, cp, code, S, T, None)
    N.check(eng.lib, eng.handle, rc)
    try:
        assert eng.lib.hsc_b200_ksvd_filter_finish(sweep, 0, 0) == N.HSC_E_STATE          # no _gram before
        N.check(eng.lib, eng.handle, eng.lib.hsc_b200_ksvd_filter_gram(sweep, 0, None))
        assert eng.lib.hsc_b200_ksvd_filter_gram(sweep, 1, None) == N.HSC_E_STATE         # a filter is open
        assert eng.lib.hsc_b200_ksvd_filter_finish(sweep, 1, 0) == N.HSC_E_STATE          # not the open one
        N.check(eng.lib, eng.handle, eng.lib.hsc_b200_ksvd_filter_finish(sweep, 0, 0))
    finally:
        sweep_end(eng, sweep)
    # PCA set: the sweep API refuses
    N.check(eng.lib, eng.handle, eng.lib.hsc_b200_ksvd_set_pca(eng.handle, 1))
    try:
        rc, _ = sweep_begin(eng, Dd, cp, code, S, T, None)
        assert rc == N.HSC_E_UNSUPPORTED
    finally:
        eng.lib.hsc_b200_ksvd_set_pca(eng.handle, 0)
    # a decreasing col_ptr
    bad = cp.copy()
    bad[1], bad[2] = bad[2], bad[1]
    rc, _ = sweep_begin(eng, Dd, bad, code, S, T, None)
    assert rc == N.HSC_E_INVALID
    with pytest.raises(N.HscError) as ei:
        eng.ksvd_update(D0, *code, bad, S, T)
    assert ei.value.code == N.HSC_E_INVALID
    # q = 3073 is refused, q = 3072 runs and is right
    for (L2, F2), want in (((3073, 1), N.HSC_E_UNSUPPORTED), ((1024, 3), N.HSC_OK)):
        S2, T2, K2 = 1, 3 * L2, 2
        D2 = unit_dictionary(rs, K2, L2, F2)
        s2, p2, i2, c2 = sort_code(np.zeros(8, int), rs.randint(0, T2, 8), np.array([0, 1] * 4), rs.uniform(0.5, 2.0, 8))
        cp2 = col_ptr_of(i2, K2)
        code2 = to_dev(eng, s2, p2, i2, c2)
        rc, sw = sweep_begin(eng, torch.from_numpy(D2).to(eng.device), cp2, code2, S2, T2, None)
        assert rc == want, (L2, F2, rc)
        if rc == N.HSC_OK:
            sweep_end(eng, sw)
            D_new, c_new, alpha = eng.ksvd_update(D2, *code2, cp2, S2, T2)
            assert check_sweep(D2, D_new, c_new.cpu().numpy(), alpha, ref_sweep(D2, s2, p2, i2, c2, S2, T2), 'q=3072')
        else:
            with pytest.raises(N.HscError) as ei:
                eng.ksvd_update(D2, *code2, cp2, S2, T2)
            assert ei.value.code == want
