"""Hierarchical codes that stay on the GPU: the canonical-code kernel (Engine.canonicalize_codes, hsc_b200_canonicalize_codes)
against a float64 replay of the events in selection order, and HierarchicalConvolutionalSparseCoder.encodeBatchDevice against
encodeBatch.  The device path sums duplicate events in selection order; the host path's scipy sum may reorder three or more
events of one (t, k), so values are compared within 1e-12 of the level's largest coefficient and everything else exactly."""
import ctypes

import numpy as np
import pytest
import scipy.sparse

from helpers import load_npz

SETTINGS = (('cmp_b10', 'cmp', 10), ('cmp_b1', 'cmp', 1), ('locomp_b10', 'locomp', 10))
MIN_COEF = 1e-16


@pytest.fixture(scope='module')
def hsc():
    import torch
    assert torch.cuda.is_available(), 'gpu tests need a CUDA device'
    import hierarchical_sparse_coding_b200 as pkg
    return pkg


@pytest.fixture(scope='module')
def c3_mld(hsc):
    z = load_npz('c3_complex.npz')
    nl = int(z['nb_levels'])
    mld = hsc.MultilevelDictionary([z['raw_l%d' % i] for i in range(nl)], [int(v) for v in z['scales']],
                                   [z['rep_l%d' % i] for i in range(nl)], z['counts_no_singletons'], hasSingletonBases=True)
    return z['x'], mld


def _members(x, n_rolls, seed=5):
    rs = np.random.RandomState(seed)
    return [x] + [np.roll(x, int(o)) for o in rs.randint(1, len(x), n_rolls)]


# ---------------------------------------------------------------------------------------------------- kernel vs replay
def _signal_events(rs, n, T, K):
    """n events over a small key set: runs of 2 to 50 duplicates, magnitudes 1e-8..1e8, runs that cancel to exactly 0
    (c then -c) and sums below 1e-16.  Half the filters are below 16, so bounds [4, 12] split the entries."""
    if n == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64), np.zeros(0)
    m = max(1, n // rs.randint(2, 51))
    kt = rs.randint(0, T, m)
    kk = np.where(rs.rand(m) < 0.5, rs.randint(0, 16, m), rs.randint(0, K, m))
    which = rs.randint(0, m, n)
    c = rs.choice([-1.0, 1.0], n) * 10.0 ** rs.uniform(-8, 8, n)
    t, k = kt[which], kk[which]
    if n >= 8:                                         # exact cancellation and sub-threshold sums on keys of their own
        t[:4], k[:4] = T - 1, 3
        c[:4] = [2.5, 7.0, -2.5, -7.0]
        t[4:6], k[4:6] = 0, K - 1
        c[4:6] = [3e-17, 4e-17]
        t[6:8], k[6:8] = 1, 5
        c[6] = 1.25e-3
        c[7] = -c[6]
        order = rs.permutation(n)
        t, k, c = t[order], k[order], c[order]
    return t, k, c


def _replay(offsets, t, k, c, K, bounds):
    """Selection-order float64 sums per (signal, t, k), threshold, ascending (t, k), split by bounds."""
    S = len(offsets) - 1
    L = len(bounds) + 1
    out = [([0], [], [], []) for _ in range(L)]
    for s in range(S):
        acc = {}
        for e in range(offsets[s], offsets[s + 1]):
            key = int(t[e]) * K + int(k[e])
            acc[key] = acc[key] + float(c[e]) if key in acc else float(c[e])
        per = [[] for _ in range(L)]
        for key in sorted(acc):
            v = acc[key]
            if v == 0.0 or abs(v) < MIN_COEF:
                continue
            col = key % K
            j = next((j for j, b in enumerate(bounds) if col < b), L - 1)
            per[j].append((key // K, col, v))
        for j in range(L):
            o, p, i, v = out[j]
            o.append(o[-1] + len(per[j]))
            p.extend(e[0] for e in per[j])
            i.extend(e[1] for e in per[j])
            v.extend(e[2] for e in per[j])
    return [(np.array(o, np.int64), np.array(p, np.int64), np.array(i, np.int64), np.array(v, np.float64)) for (o, p, i, v) in out]


@pytest.mark.gpu
def test_canonicalize_codes_equals_selection_order_replay(hsc):
    import torch
    rs = np.random.RandomState(11)
    T, K = 4096, 1 << 20                               # T*K = 2^32: 64-bit keys
    sizes = [int(v) for v in rs.randint(0, 3001, 300)]
    sizes[3] = 0
    sizes[7] = 1
    sizes[100] = 4096                                  # the largest signal sorted in shared memory
    sizes[101] = 4097                                  # the smallest one sorted in global memory
    sizes.append(200000)                               # a long signal: global-memory path
    parts = [_signal_events(rs, n, T, K) for n in sizes]
    offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    t = np.concatenate([p[0] for p in parts])
    k = np.concatenate([p[1] for p in parts])
    c64 = np.concatenate([p[2] for p in parts])
    S = len(sizes)
    for dt in (np.float32, np.float64):
        c = c64.astype(dt)
        eng = hsc.Engine()
        eng.set_dictionary(np.ones((2, 4, 1)), dtype=dt)
        dev = lambda a, d: torch.from_numpy(np.ascontiguousarray(a, dtype=d)).cuda()
        args = (dev(offsets, np.int64), dev(t, np.int32), dev(k, np.int32), dev(c, dt), S, T, K)
        for bounds in (None, [4, 12]):
            ref = _replay(offsets, t, k, c, K, bounds or [])
            runs = [eng.canonicalize_codes(*args, level_bounds=bounds) for _ in range(2)]
            for run in runs:
                assert len(run) == len(ref)
                for j, (lv, (ro, rp, ri, rv)) in enumerate(zip(run, ref)):
                    n = int(ro[-1])
                    assert np.array_equal(lv['offsets'].cpu().numpy(), ro), (dt, bounds, j)
                    assert np.array_equal(lv['pos'][:n].cpu().numpy(), rp), (dt, bounds, j)
                    assert np.array_equal(lv['idx'][:n].cpu().numpy(), ri), (dt, bounds, j)
                    assert np.array_equal(lv['coef'][:n].cpu().numpy().view(np.int64), rv.view(np.int64)), (dt, bounds, j)
            if bounds:
                assert all(int(r[0][-1]) > 0 for r in ref)          # every level receives entries
        eng.close()


@pytest.mark.gpu
def test_canonicalize_codes_abi_rejects_bad_arguments(hsc):
    from hierarchical_sparse_coding_b200 import _native as N
    lib = N.load_library()
    h = ctypes.c_void_p()
    assert lib.hsc_b200_create(0, ctypes.byref(h)) == N.HSC_OK
    p = ctypes.c_void_p(16)
    b = (ctypes.c_int64 * 3)(4, 12, 20)

    def call(offsets=p, pos=p, capacity=8, S=1, T=10, K=4, bounds=b, n_bounds=2, out_offsets=p, out_pos=p):
        return lib.hsc_b200_canonicalize_codes(h, offsets, pos, p, p, capacity, S, T, K, bounds, n_bounds, 1e-16, out_offsets,
                                               out_pos, p, p, None)
    try:
        assert call() == N.HSC_E_STATE                                          # no dictionary: no coefficient dtype
        D = np.ones((2, 4, 1), dtype=np.float64)
        assert lib.hsc_b200_set_dictionary(h, D.ctypes.data_as(ctypes.c_void_p), N.HSC_F64, 2, 4, 1, None) == N.HSC_OK
        assert call(offsets=None) == N.HSC_E_INVALID
        assert call(out_offsets=None) == N.HSC_E_INVALID
        assert call(pos=None) == N.HSC_E_INVALID
        assert call(out_pos=None) == N.HSC_E_INVALID
        assert call(S=0) == N.HSC_E_INVALID
        assert call(S=65536) == N.HSC_E_INVALID
        assert call(T=0) == N.HSC_E_INVALID
        assert call(T=1 << 31) == N.HSC_E_INVALID
        assert call(K=0) == N.HSC_E_INVALID
        assert call(K=1 << 31) == N.HSC_E_INVALID
        assert call(capacity=-1) == N.HSC_E_INVALID
        assert call(bounds=None) == N.HSC_E_INVALID
        assert call(n_bounds=-1) == N.HSC_E_INVALID
        assert call(n_bounds=16) == N.HSC_E_INVALID
        assert call(bounds=(ctypes.c_int64 * 2)(12, 4)) == N.HSC_E_INVALID       # decreasing
        assert call(bounds=(ctypes.c_int64 * 2)(-1, 4)) == N.HSC_E_INVALID
    finally:
        lib.hsc_b200_destroy(h)


# ---------------------------------------------------------------------------------------------------- encodeBatchDevice
def _assert_matches_host(coder, X, kw, codes_d, res_d):
    """Device codes vs encodeBatch: same pattern at every level, values within 1e-12 max|coef|; the residual and
    reconstructBatchDevice equal the host decoder's on the device codes bit for bit."""
    codes_h, res_h = coder.encodeBatch(X, **kw)
    csc = codes_d.to_csc()
    assert len(csc) == len(codes_h) == codes_d.B
    for b, (cd, ch) in enumerate(zip(csc, codes_h)):
        assert len(cd) == len(ch)
        for l, (a, r) in enumerate(zip(cd, ch)):
            assert a.format == 'csc' and a.dtype == np.float64 and a.shape == r.shape and a.has_canonical_format, (b, l)
            r = r.sorted_indices()
            assert np.array_equal(a.indptr, r.indptr) and np.array_equal(a.indices, r.indices), (b, l)
            if r.nnz:
                assert np.max(np.abs(a.data - r.data)) <= 1e-12 * np.max(np.abs(r.data)), (b, l)
    assert res_d.dtype.is_floating_point and str(res_d.dtype) == 'torch.float64' and res_d.is_cuda
    assert tuple(res_d.shape) == res_h.shape
    if codes_d.B == 0:
        return
    X64 = np.asarray(X, dtype=np.float64).reshape(res_h.shape)
    recon = coder.reconstructBatch(csc)
    assert np.array_equal(res_d.cpu().numpy(), X64 - recon)
    assert np.array_equal(coder.reconstructBatchDevice(codes_d).cpu().numpy(), recon)


def _same_device_result(a, b):
    (ca, ra), (cb, rb) = a, b
    import torch
    assert ca.B == cb.B and ca.T == cb.T and ca.K == cb.K
    for l in range(len(ca.K)):
        for f in ('offsets', 'pos', 'idx', 'coef'):
            assert torch.equal(getattr(ca, f)[l], getattr(cb, f)[l]), (l, f)
    assert torch.equal(ra, rb)


@pytest.mark.gpu
def test_config3_device_codes_match_encode_batch(hsc, c3_mld):
    x, mld = c3_mld
    X = np.stack(_members(x, 4) + [x[::-1].copy()])
    for tag, method, nb in SETTINGS:
        coder = hsc.HierarchicalConvolutionalSparseCoder(mld, hsc.HierarchicalConvolutionalMatchingPursuit(method=method))
        for dist in (True, False):
            kw = dict(toleranceSnr=10.0, nbBlocks=nb, singletonWeight=0.95, returnDistributed=dist)
            codes, res = coder.encodeBatchDevice(X, **kw)
            assert isinstance(codes, hsc.HierarchicalCodes) and codes.K == [4, 12, 28] and codes.T == X.shape[1]
            assert all(t.is_cuda for t in codes.coef)
            if not dist:
                assert all(int(codes.offsets[l][-1]) == 0 for l in range(2))
            _assert_matches_host(coder, X, kw, codes, res)
            _same_device_result((codes, res), coder.encodeBatchDevice(X, **kw))          # deterministic


@pytest.mark.gpu
def test_device_chunk_boundaries_do_not_change_the_result(hsc, c3_mld, monkeypatch):
    x, mld = c3_mld
    X = np.stack(_members(x, 6, seed=9))
    approx = hsc.HierarchicalConvolutionalMatchingPursuit(method='cmp')
    coder = hsc.HierarchicalConvolutionalSparseCoder(mld, approx)
    kw = dict(toleranceSnr=10.0, nbBlocks=10, singletonWeight=0.95)
    one = coder.encodeBatchDevice(X, **kw)
    chunks = []
    orig = type(approx)._forward_chunk
    monkeypatch.setattr(type(approx), '_chunk_size', lambda self, T, specs, cap_scale: 3)
    monkeypatch.setattr(type(approx), '_forward_chunk', lambda self, x, *a: chunks.append(x.shape[0]) or orig(self, x, *a))
    _same_device_result(coder.encodeBatchDevice(X, **kw), one)
    assert chunks == [3, 3, 1]


def _locomp_rerun_input(hsc):
    from oracle import hsc_oracle as O
    rs = np.random.RandomState(77)
    T, K, L = 4096, 6, 32
    D = O.normalize(rs.randn(K, L))
    mld = hsc.MultilevelDictionary([D], [L], [D], [K], hasSingletonBases=True)
    dense = np.zeros(T)
    for p in range(L, T - L, 2):                     # overlapping atoms every 2 samples: large refit groups
        O.overlap_add(dense[:, None], rs.randn() * D[rs.randint(K)][:, None], p)
    sparse = np.zeros(T)
    for p in rs.randint(L, T - L, 20):
        O.overlap_add(sparse[:, None], rs.uniform(1, 2) * D[rs.randint(K)][:, None], p)
    return mld, np.stack([sparse, dense + 1e-3 * rs.randn(T), sparse[::-1].copy()])


@pytest.mark.gpu
def test_device_locomp_capacity_escalation(hsc, monkeypatch):
    """A member that fills the LoCOMP event buffers: its chunk is rerun with 8x the buffers, and the result equals a run
    whose buffers were large enough from the start."""
    mld, X = _locomp_rerun_input(hsc)
    approx = hsc.HierarchicalConvolutionalMatchingPursuit(method='locomp')
    coder = hsc.HierarchicalConvolutionalSparseCoder(mld, approx)
    kw = dict(toleranceSnr=40.0, singletonWeight=0.95)
    scales = []
    orig = type(approx)._encode_pass
    monkeypatch.setattr(type(approx), '_encode_pass', lambda self, x, r, specs, cs, *a: scales.append(cs) or orig(self, x, r, specs, cs, *a))
    rerun = coder.encodeBatchDevice(X, **kw)
    assert max(scales) >= 8, scales
    _assert_matches_host(coder, X, kw, *rerun)
    cap = hsc.Engine.default_capacity
    monkeypatch.setattr(hsc.Engine, 'default_capacity', lambda self, options, T: 64 * cap(self, options, T))
    del scales[:]
    _same_device_result(coder.encodeBatchDevice(X, **kw), rerun)
    assert max(scales) == 1, scales


@pytest.mark.gpu
def test_device_input_variants(hsc, c3_mld):
    import torch
    x, mld = c3_mld
    X = np.stack(_members(x, 2, seed=4))
    coder = hsc.HierarchicalConvolutionalSparseCoder(mld, hsc.HierarchicalConvolutionalMatchingPursuit(method='cmp'))
    kw = dict(toleranceSnr=10.0, nbBlocks=10, singletonWeight=0.95)
    ref = coder.encodeBatchDevice(X, **kw)
    _same_device_result(coder.encodeBatchDevice(torch.from_numpy(X).cuda(), **kw), ref)       # CUDA float32 tensor
    _same_device_result(coder.encodeBatchDevice(torch.from_numpy(X), **kw), ref)              # host tensor
    _same_device_result(coder.encodeBatchDevice(X[:, :, None], **kw), ref)                   # [B,T,1]
    X64 = X.astype(np.float64)
    codes64, res64 = coder.encodeBatchDevice(X64, **kw)
    _assert_matches_host(coder, X64, kw, codes64, res64)
    _same_device_result(coder.encodeBatchDevice(torch.from_numpy(X64).cuda(), **kw), (codes64, res64))
    one = coder.encodeBatchDevice(X[:1], **kw)                                                # B = 1
    _assert_matches_host(coder, X[:1], kw, *one)
    codes0, res0 = coder.encodeBatchDevice(X[:0], **kw)                                       # B = 0
    assert codes0.B == 0 and codes0.to_csc() == [] and tuple(res0.shape) == (0, X.shape[1]) and res0.is_cuda
    assert all(int(o.numel()) == 1 for o in codes0.offsets)
    # one level, three channels
    rs = np.random.RandomState(3)
    T, K, L, F = 1500, 6, 16, 3
    D = hsc.normalize(rs.randn(K, L, F))
    mld1 = hsc.MultilevelDictionary([D], [L], [D], [K], hasSingletonBases=True)
    approx = hsc.HierarchicalConvolutionalMatchingPursuit(method='cmp')
    coder1 = hsc.HierarchicalConvolutionalSparseCoder(mld1, approx)
    X3 = rs.randn(4, T, F)
    kw1 = dict(toleranceSnr=6.0, nbBlocks=1)
    codes3, res3 = coder1.encodeBatchDevice(X3, **kw1)
    assert tuple(res3.shape) == (4, T, F) and codes3.K == [K]
    _assert_matches_host(coder1, X3, kw1, codes3, res3)
    with pytest.raises(AssertionError):
        coder1.encodeBatchDevice(X3[0], **kw1)                     # one sequence: ndim 2 is [B,T], channels then mismatch
    with pytest.raises(AssertionError):
        coder1.encodeBatchDevice(X3[:, :, :, None], **kw1)
    with pytest.raises(AssertionError):
        approx.computeCoefficientsBatchDevice(X3[:, :, :2], mld1, **kw1)    # 2 channels for a 3-channel dictionary


# ---------------------------------------------------------------------------------------------------- host only
def test_hierarchical_codes_to_csc_on_host_tensors():
    import torch
    from hierarchical_sparse_coding_b200 import HierarchicalCodes
    T = 6
    K = [3, 5]
    # level 0: sequence 0 has (1,2), sequence 1 is empty, sequence 2 has (0,0), (4,1); level 1: only sequence 1
    off = [torch.tensor([0, 1, 1, 3]), torch.tensor([0, 0, 2, 2])]
    pos = [torch.tensor([1, 0, 4], dtype=torch.int32), torch.tensor([2, 2], dtype=torch.int32)]
    idx = [torch.tensor([2, 0, 1], dtype=torch.int32), torch.tensor([0, 4], dtype=torch.int32)]
    coef = [torch.tensor([0.5, -1.0, 2.0], dtype=torch.float64), torch.tensor([3.0, -4.0], dtype=torch.float64)]
    codes = HierarchicalCodes(3, T, K, off, pos, idx, coef).to_csc()
    assert len(codes) == 3 and all(len(c) == 2 for c in codes)
    dense = [[np.zeros((T, k)) for k in K] for _ in range(3)]
    dense[0][0][1, 2] = 0.5
    dense[2][0][0, 0] = -1.0
    dense[2][0][4, 1] = 2.0
    dense[1][1][2, 0] = 3.0
    dense[1][1][2, 4] = -4.0
    for b in range(3):
        for l in range(2):
            m = codes[b][l]
            assert m.format == 'csc' and m.dtype == np.float64 and m.shape == (T, K[l]) and m.has_canonical_format
            assert np.array_equal(m.toarray(), dense[b][l]), (b, l)
    assert codes[1][0].nnz == 0 and codes[0][1].nnz == 0
