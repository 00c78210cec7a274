"""Shared helpers of the parity harness (test infrastructure)."""
import ast
import os

import numpy as np
import scipy.sparse

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def load_npz(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


def case_kwargs(z, name):
    kw = ast.literal_eval(str(z[name + '_kw']))
    if 'weights' in kw and kw['weights'] is not None:
        kw['weights'] = np.asarray(kw['weights'], dtype=z[name + '_D'].dtype)
    return kw


def coo_sorted(m):
    c = scipy.sparse.coo_matrix(m)
    c.sum_duplicates()
    order = np.lexsort((c.col, c.row))
    return c.row[order].astype(np.int64), c.col[order].astype(np.int64), c.data[order].astype(np.float64)


def stored_code(z, key):
    """The csc code [T,K] stored under key_t / key_k / key_v / key_shape (tests/golden/make_golden_dropin.py)."""
    return scipy.sparse.coo_matrix((z[key + '_v'], (z[key + '_t'], z[key + '_k'])), shape=tuple(z[key + '_shape'])).tocsc()


def snr_db(x, residual):
    e = float(np.sum(np.square(np.asarray(residual, dtype=np.float64))))
    s = float(np.sum(np.square(np.asarray(x, dtype=np.float64))))
    return np.inf if e == 0.0 else 10.0 * np.log10(s / e)


class TraceComparison(object):
    """Step-wise comparison of two selection traces under the north-star rule: identical (t,k)
    sequence except at documented near-ties (relative correlation gap < tie_tol); after the first
    permitted flip the ORDER may differ, so the accumulated codes are compared instead."""

    def __init__(self, ref_t, ref_k, ref_c, got_t, got_k, got_c):
        self.ref = (np.asarray(ref_t), np.asarray(ref_k), np.asarray(ref_c, dtype=np.float64))
        self.got = (np.asarray(got_t), np.asarray(got_k), np.asarray(got_c, dtype=np.float64))
        n = min(len(self.ref[0]), len(self.got[0]))
        same = (self.ref[0][:n] == self.got[0][:n]) & (self.ref[1][:n] == self.got[1][:n])
        self.common_prefix = int(n if same.all() else np.argmin(same))
        self.n_ref = len(self.ref[0])
        self.n_got = len(self.got[0])

    @property
    def identical_sequence(self):
        return self.common_prefix == self.n_ref == self.n_got

    def prefix_coef_rel_err(self):
        n = self.common_prefix
        if n == 0:
            return 0.0
        r, g = self.ref[2][:n], self.got[2][:n]
        scale = np.maximum(np.abs(r), 1e-3 * np.max(np.abs(r)))
        return float(np.max(np.abs(r - g) / scale))

    def divergence_gap(self):
        """Relative gap between the two candidates at the first divergent step, measured on the
        reference's coefficients: |c_ref(step)| vs the magnitude the other side picked."""
        n = self.common_prefix
        if n >= min(self.n_ref, self.n_got):
            return 0.0
        a, b = abs(self.ref[2][n]), abs(self.got[2][n])
        return float(abs(a - b) / max(a, b, 1e-300))


def oracle_gap(oracle, x, D, kw, cmpx):
    """Relative correlation gap of the first divergent step, measured ON THE ORACLE'S MAP (north star: 'near-tie
    steps below 1e-6 relative correlation gap'): the oracle is replayed to the start of the selection pass that
    produces the divergent event, and the (weighted) scores it holds there for its own pick and for the engine's
    pick are compared.  Returns (gap, score_ref, score_got); gap = 0.0 when the common prefix covers a whole trace."""
    n = cmpx.common_prefix
    if n >= min(cmpx.n_ref, cmpx.n_got):
        return 0.0, None, None
    kw = dict(kw)
    kw.pop('stopCondition', None)
    _, _, tr = oracle.mp_encode(x, D, return_trace=True, snapshot_event=n, **kw)
    snap = tr.snapshot
    assert snap is not None, 'oracle stopped (%s) before event %d' % (tr.stop, n)
    inner = np.abs(snap['inner'])
    w = kw.get('weights')
    if w is not None:
        inner = inner * np.abs(np.asarray(w))[None, :]
    a = float(inner[int(cmpx.ref[0][n]), int(cmpx.ref[1][n])])
    b = float(inner[int(cmpx.got[0][n]), int(cmpx.got[1][n])])
    return abs(a - b) / max(a, b, 1e-300), a, b


def accumulate(t, k, c, shape):
    m = scipy.sparse.coo_matrix((np.asarray(c, dtype=np.float64), (np.asarray(t), np.asarray(k))), shape=shape)
    m = m.tocsc()
    return m


def code_diff(ref, got, rel=1e-5):
    """|delta| <= rel * max(|c_ref|, scale) on the union support (SURVEY 7.3 item 2).  Returns
    (max_violation_ratio, n_support_mismatch)."""
    ref = scipy.sparse.csc_matrix(ref)
    got = scipy.sparse.csc_matrix(got)
    d = (ref - got).tocoo()
    if ref.nnz == 0:
        return (0.0 if got.nnz == 0 else np.inf), got.nnz
    scale = float(np.max(np.abs(ref.data)))
    refd = np.abs(np.asarray(ref[d.row, d.col])).ravel() if d.nnz else np.zeros(0)
    tol = rel * np.maximum(refd, 1e-2 * scale)
    ratio = float(np.max(np.abs(d.data) / tol)) if d.nnz else 0.0
    sr = set(zip(*ref.nonzero()))
    sg = set(zip(*got.nonzero()))
    return ratio, len(sr ^ sg)


# ---- full-length golden traces of the BASELINE shapes (tests/golden/long_traces.npz, make_golden_long.py) ----
LONG_CASES = {
    # name: (bench.py workload, signal seed, index of the signal in the seeded batch, nbNonzeroCoefs)
    'c4_s0': ('c4', 4242, 0, 655),
    'c4_s1': ('c4', 4242, 1, 655),
    'c5_s0': ('c5', 55, 0, 655),
    'c5_s1': ('c5', 55, 1, 655),
    'c2_s0': ('c2', 77, 0, 1200),
}
# the stored config-2 toy input is split into this many consecutive parts so that every file stays under 1 MB
C2TOY_PARTS = 3


def long_case_inputs(name):
    """(x, D, nbNonzeroCoefs) of a long case: the seeded synthetic signals of bench.py (legacy RandomState streams), or
    the stored toy training signal for 'c2toy'."""
    if name == 'c2toy':
        parts = [load_npz('c2_toy_1e6_part%d.npz' % i) for i in range(C2TOY_PARTS)]
        return np.concatenate([z['x'] for z in parts]), parts[0]['D'], 1000
    import bench
    wl, seed, s, n = LONG_CASES[name]
    w = dict(bench.WORKLOADS[wl])
    w['S'] = s + 1
    D = bench.make_dictionary(w)
    x = bench.make_signals(w, D, seed=seed)[s]
    if w['F'] == 1:
        return x[:, 0], D[:, :, 0], n
    return x, D, n
