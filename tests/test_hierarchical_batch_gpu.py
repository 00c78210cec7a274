"""Batched hierarchical encoding (HierarchicalConvolutionalSparseCoder.encodeBatch) and the batched sparse decoder
(Engine.decode_batch, reconstructBatch).  Every member of a batch must get bit for bit the codes and the residual of its
own single call; the single path runs through the same level loop and decoder, so the config-3 member also meets the
reference gate of the single test."""
import numpy as np
import pytest
import scipy.sparse

from helpers import load_npz, snr_db, code_diff

pytestmark = pytest.mark.gpu

SNR_DB = 0.01
COEF_REL = 1e-5
SETTINGS = (('cmp_b10', 'cmp', 10), ('cmp_b1', 'cmp', 1), ('locomp_b10', 'locomp', 10))


@pytest.fixture(scope='module')
def hsc():
    import torch
    assert torch.cuda.is_available(), 'gpu tests need a CUDA device'
    import hierarchical_sparse_coding_b200 as pkg
    return pkg


@pytest.fixture(scope='module')
def c3():
    z = load_npz('c3_complex.npz')
    nl = int(z['nb_levels'])
    raw = [z['raw_l%d' % i] for i in range(nl)]
    rep = [z['rep_l%d' % i] for i in range(nl)]
    return z, raw, rep, z['counts_no_singletons'], [int(v) for v in z['scales']]


@pytest.fixture(scope='module')
def c3_mld(hsc, c3):
    z, raw, rep, cns, scales = c3
    return hsc.MultilevelDictionary(raw, scales, rep, cns, hasSingletonBases=True)


def _members(x, n_rolls, seed=5):
    rs = np.random.RandomState(seed)
    xs = [x] + [np.roll(x, int(o)) for o in rs.randint(1, len(x), n_rolls)]
    return xs


def _assert_same_codes(a, b, where):
    assert len(a) == len(b), where
    for l, (ca, cb) in enumerate(zip(a, b)):
        assert ca.format == 'csc' and cb.format == 'csc' and ca.dtype == np.float64 and ca.shape == cb.shape, (where, l)
        assert (ca != cb).nnz == 0, (where, l)


def test_config3_batch_equals_single_calls(hsc, c3, c3_mld):
    """Six members (x, four rolled copies, x reversed) x three scripted settings x returnDistributed: every member's codes
    and residual equal its own encode's bit for bit; member x also meets the reference gate of the single test."""
    z = c3[0]
    x = z['x']
    xs = _members(x, 4) + [x[::-1].copy()]
    X = np.stack(xs)
    for tag, method, nb in SETTINGS:
        coder = hsc.HierarchicalConvolutionalSparseCoder(c3_mld, hsc.HierarchicalConvolutionalMatchingPursuit(method=method))
        for dist, sfx in ((True, ''), (False, '_nodist')):
            kw = dict(toleranceSnr=10.0, nbBlocks=nb, singletonWeight=0.95, returnDistributed=dist)
            codes, res = coder.encodeBatch(X, **kw)
            assert len(codes) == len(xs) and res.shape == X.shape and res.dtype == np.float64
            for b, xb in enumerate(xs):
                c1, r1 = coder.encode(xb, **kw)
                _assert_same_codes(codes[b], c1, (tag, sfx, b))
                assert np.array_equal(res[b], r1), (tag, sfx, b)
            ref_nnz = [len(z['%s%s_l%d_t' % (tag, sfx, l)]) for l in range(3)]
            assert [c.nnz for c in codes[0]] == ref_nnz, (tag, sfx)
            assert abs(snr_db(x, z['%s%s_res' % (tag, sfx)]) - snr_db(x, res[0])) <= SNR_DB, (tag, sfx)
            # the batched decoder gives what the per-sequence one gives
            xr = coder.reconstructBatch(codes)
            for b in (0, len(xs) - 1):
                assert np.array_equal(xr[b], coder.reconstruct(codes[b])), (tag, sfx, b)


def test_batch_against_the_oracle(hsc, c3):
    """Signals synthesised from seeded sparse level-2 codes through the fixture's representations, plus noise: two members
    against the oracle's hierarchical encoder - same support at every level, coefficients within 1e-5, SNR within 0.01 dB."""
    from oracle import hsc_oracle as O
    z, raw, rep, cns, scales = c3
    mld = hsc.MultilevelDictionary(raw, scales, rep, cns, hasSingletonBases=True)
    rs = np.random.RandomState(2024)
    T, K2 = 6000, rep[2].shape[0]
    xs = []
    for _ in range(4):
        n = 40
        code = scipy.sparse.coo_matrix((rs.uniform(0.5, 2.0, n) * rs.choice([-1.0, 1.0], n),
                                        (rs.randint(0, T, n), rs.randint(0, K2, n))), shape=(T, K2))
        x = O.reconstruct(code.tocsc(), rep[2].astype(np.float64)) + 0.01 * rs.randn(T)
        xs.append(x.astype(np.float32))
    X = np.stack(xs)
    coder = hsc.HierarchicalConvolutionalSparseCoder(mld, hsc.HierarchicalConvolutionalMatchingPursuit(method='cmp'))
    kw = dict(toleranceSnr=10.0, nbBlocks=1, singletonWeight=0.95)
    codes, res = coder.encodeBatch(X, returnDistributed=False, **kw)
    for b in (0, 3):
        c_ref, r_ref = O.hierarchical_encode(xs[b], raw, cns, rep, returnDistributed=False, method='cmp', **kw)
        for l in range(3):
            ratio, mism = code_diff(c_ref[l], codes[b][l], rel=COEF_REL)
            assert mism == 0 and ratio <= 1.0, (b, l, ratio, mism)
        assert abs(snr_db(xs[b], r_ref) - snr_db(xs[b], res[b])) <= SNR_DB, b


def test_chunk_boundaries_do_not_change_the_result(hsc, c3_mld, c3, monkeypatch):
    x = c3[0]['x']
    X = np.stack(_members(x, 6, seed=9))
    approx = hsc.HierarchicalConvolutionalMatchingPursuit(method='cmp')
    coder = hsc.HierarchicalConvolutionalSparseCoder(c3_mld, approx)
    kw = dict(toleranceSnr=10.0, nbBlocks=10, singletonWeight=0.95)
    codes1, res1 = coder.encodeBatch(X, **kw)
    chunks = []
    orig = type(approx)._forward_chunk
    monkeypatch.setattr(type(approx), '_chunk_size', lambda self, T, specs, cap_scale: 3)
    monkeypatch.setattr(type(approx), '_forward_chunk', lambda self, x, *a: chunks.append(x.shape[0]) or orig(self, x, *a))
    codes3, res3 = coder.encodeBatch(X, **kw)
    assert chunks == [3, 3, 1]
    for b in range(len(X)):
        _assert_same_codes(codes3[b], codes1[b], b)
    assert np.array_equal(res3, res1)


def test_locomp_capacity_escalation(hsc, monkeypatch):
    """A member whose LoCOMP run needs more events than the default buffers hold: its chunk is rerun with 8x the buffers,
    and every member still equals its single call."""
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
    X = np.stack([sparse, dense + 1e-3 * rs.randn(T), sparse[::-1].copy()])
    approx = hsc.HierarchicalConvolutionalMatchingPursuit(method='locomp')
    coder = hsc.HierarchicalConvolutionalSparseCoder(mld, approx)
    scales = []
    orig = type(approx)._encode_pass
    monkeypatch.setattr(type(approx), '_encode_pass', lambda self, x, r, specs, cs, *a: scales.append(cs) or orig(self, x, r, specs, cs, *a))
    kw = dict(toleranceSnr=40.0, singletonWeight=0.95)
    codes, res = coder.encodeBatch(X, **kw)
    assert max(scales) >= 8, scales
    for b in range(len(X)):
        c1, r1 = coder.encode(X[b], **kw)
        _assert_same_codes(codes[b], c1, b)
        assert np.array_equal(res[b], r1), b


def test_one_level_multichannel_and_shapes(hsc):
    rs = np.random.RandomState(3)
    T, K, L, F = 1500, 6, 16, 3
    D = hsc.normalize(rs.randn(K, L, F))
    mld = hsc.MultilevelDictionary([D], [L], [D], [K], hasSingletonBases=True)
    approx = hsc.HierarchicalConvolutionalMatchingPursuit(method='cmp')
    coder = hsc.HierarchicalConvolutionalSparseCoder(mld, approx)
    X = rs.randn(4, T, F)
    kw = dict(toleranceSnr=6.0, nbBlocks=1)
    codes, res = coder.encodeBatch(X, **kw)
    assert res.shape == (4, T, F) and len(codes) == 4 and len(codes[0]) == 1
    for b in range(4):
        c1, r1 = coder.encode(X[b], **kw)
        _assert_same_codes(codes[b], c1, b)
        assert np.array_equal(res[b], r1), b
    # B = 1 equals computeCoefficients
    cb, rb = approx.computeCoefficientsBatch(X[:1], mld, **kw)
    c1, r1 = approx.computeCoefficients(X[0], mld, **kw)
    _assert_same_codes(cb[0], c1, 'B=1')
    assert np.array_equal(rb[0], r1)
    xr = coder.reconstructBatch(codes)
    assert xr.shape == (4, T, F)
    assert np.array_equal(xr[2], coder.reconstruct(codes[2]))
    with pytest.raises(AssertionError):
        coder.encodeBatch(X[0])                                  # one sequence: ndim 2 is [B,T], channels then mismatch
    with pytest.raises(AssertionError):
        coder.encodeBatch(X[:, :, :, None])
    with pytest.raises(AssertionError):
        approx.computeCoefficientsBatch(X[:, :, :2], mld, **kw)  # 2 channels for a 3-channel dictionary


def _random_codes(rs, T, K, n_codes, dtype):
    codes = []
    for s in range(n_codes):
        if s == 1:
            codes.append(scipy.sparse.csc_matrix((T, K), dtype=dtype))          # a signal with no atoms
            continue
        n = 30
        t = np.concatenate([[0, 1, T - 1, T - 2], rs.randint(0, T, n)])          # atoms clipped at both ends
        k = rs.randint(0, K, len(t))
        codes.append(scipy.sparse.coo_matrix((rs.randn(len(t)).astype(dtype), (t, k)), shape=(T, K)).tocsc())
    return codes


def test_decoder_batch_equals_single(hsc):
    import ctypes
    import torch
    from hierarchical_sparse_coding_b200 import _native as N
    rs = np.random.RandomState(8)
    T, K, L = 700, 5, 33
    for F in (1, 2):
        D = hsc.normalize(rs.randn(K, L, F))
        for dt in (np.float32, np.float64):
            eng = hsc.Engine()
            eng.set_dictionary(D, dtype=dt)
            codes = _random_codes(rs, T, K, 5, np.float64)
            offsets, pos, idx, coef = [0], [], [], []
            for c in codes:
                cx = c.tocoo()
                pos.append(cx.row); idx.append(cx.col); coef.append(cx.data)
                offsets.append(offsets[-1] + cx.nnz)
            got = eng.decode_batch(np.array(offsets), np.concatenate(pos), np.concatenate(idx), np.concatenate(coef), len(codes), T)
            assert got.shape == (len(codes), T, F) and got.dtype == eng.torch_dtype
            for s, c in enumerate(codes):
                cx = c.tocoo()
                one = eng.decode(cx.row, cx.col, cx.data, T)
                assert torch.equal(got[s], one), (F, dt, s)
                # hsc_b200_decode, the single-signal entry point of the same kernel
                o = np.argsort(cx.row, kind='stable')
                dev = lambda a, t: torch.from_numpy(np.ascontiguousarray(a[o], dtype=t)).cuda()
                p, i, cc = dev(cx.row, np.int32), dev(cx.col, np.int32), dev(cx.data, dt)
                raw = torch.zeros((T, F), dtype=eng.torch_dtype, device='cuda')
                if cx.nnz:
                    N.check(eng.lib, eng.handle, eng.lib.hsc_b200_decode(
                        eng.handle, ctypes.c_void_p(p.data_ptr()), ctypes.c_void_p(i.data_ptr()), ctypes.c_void_p(cc.data_ptr()),
                        cx.nnz, T, ctypes.c_void_p(raw.data_ptr()), eng._stream_ptr()))
                assert torch.equal(got[s], raw), (F, dt, s)
            assert not torch.any(got[1])
            # += into a given buffer
            acc = torch.ones_like(got)
            eng.decode_batch(np.array(offsets), np.concatenate(pos), np.concatenate(idx), np.concatenate(coef), len(codes), T, out=acc)
            if dt == np.float64:
                assert torch.equal(acc, got + 1)
            else:                                        # the kernel adds in float64 and rounds once: a few float32 ulps apart
                assert torch.allclose(acc, got + 1, rtol=0, atol=1e-6 * max(1.0, float(got.abs().max())))
            eng.close()
        for cdt in (np.float32, np.float64):
            coder = hsc.ConvolutionalSparseCoder(D[:, :, 0] if F == 1 else D, hsc.ConvolutionalMatchingPursuit())
            codes = _random_codes(rs, T, K, 4, cdt)
            xr = coder.reconstructBatch(codes)
            assert xr.dtype == coder.reconstruct(codes[0]).dtype == cdt
            assert xr.shape == ((4, T) if F == 1 else (4, T, F))
            for s, c in enumerate(codes):
                assert np.array_equal(xr[s], coder.reconstruct(c)), (F, cdt, s)


def test_decode_batch_abi_rejects_bad_arguments(hsc):
    import ctypes
    from hierarchical_sparse_coding_b200 import _native as N
    lib = N.load_library()
    h = ctypes.c_void_p()
    assert lib.hsc_b200_create(0, ctypes.byref(h)) == N.HSC_OK
    try:
        p = ctypes.c_void_p(16)
        assert lib.hsc_b200_decode_batch(h, p, p, p, p, 1, 10, p, None) == N.HSC_E_STATE          # no dictionary
        D = np.ones((2, 4, 1), dtype=np.float64)
        assert lib.hsc_b200_set_dictionary(h, D.ctypes.data_as(ctypes.c_void_p), N.HSC_F64, 2, 4, 1, None) == N.HSC_OK
        assert lib.hsc_b200_decode_batch(h, None, p, p, p, 1, 10, p, None) == N.HSC_E_INVALID
        assert lib.hsc_b200_decode_batch(h, p, p, p, p, 0, 10, p, None) == N.HSC_E_INVALID
        assert lib.hsc_b200_decode_batch(h, p, p, p, p, 1, 0, p, None) == N.HSC_E_INVALID
        assert lib.hsc_b200_decode_batch(h, p, p, p, p, 1, 10, None, None) == N.HSC_E_INVALID
    finally:
        lib.hsc_b200_destroy(h)
