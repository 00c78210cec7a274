"""Single-level codes that stay on the GPU: ConvolutionalSparseCoder.encodeBatchDevice (Engine.encode_stream_device) against
encodeBatch, on seeded bench.py signals.  The device path sums duplicate events in selection order; the host path's scipy
sum may reorder three or more events of one (t, k), so such values are compared within 1e-12 of the signal's largest
coefficient and everything else - sparsity pattern, entries of one or two events, states, residual - bit for bit.

Bit-equality across different numbers of signals per launch holds at these shapes: for T <= 131072 the K2 and LoCOMP launch
choices in engine.cu do not depend on S (the shared-memory hierarchy fits without the S <= 148 branch, and the S-dependent
next-pick prefetch and third stage ring move data only), and K1 computes every (signal, tile) alike whatever the grid."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


@pytest.fixture(scope='module')
def hsc():
    import torch
    assert torch.cuda.is_available(), 'gpu tests need a CUDA device'
    import hierarchical_sparse_coding_b200 as pkg
    return pkg


def _workload(S, T, F, K, L, atoms, seed):
    import bench
    w = dict(S=S, T=T, F=F, K=K, L=L, atoms=atoms)
    D = bench.make_dictionary(w, seed=seed)
    return D, bench.make_signals(w, D, seed=seed + 1)


@pytest.fixture(scope='module')
def small():
    """6 signals of 4096 x 4 channels, 32 filters of 16 (float32: the tensor-core K1)."""
    return _workload(6, 4096, 4, 32, 16, 40, 7)


def _event_counts(res, b, K):
    """Events per (t, k) key of signal b in an EncodeResult."""
    keys = res.pos[b].astype(np.int64) * K + res.idx[b].astype(np.int64)
    u, n = np.unique(keys, return_counts=True)
    return dict(zip(u.tolist(), n.tolist()))


def _check_against_batch(coder, X, kw, codes, res_d):
    """encodeBatchDevice's result vs encodeBatch on the same input: pattern, values (exact for entries of <= 2 events),
    stats, residual bit for bit; and reconstructBatchDevice vs reconstructBatch on the device codes."""
    codes_h, res_h = coder.encodeBatch(X, **kw)
    host = coder.approximator.last_result
    csc = codes.to_csc()
    assert codes.B == len(codes_h) == len(csc)
    for b, (a, r) in enumerate(zip(csc, codes_h)):
        assert a.format == 'csc' and a.dtype == np.float64 and a.shape == r.shape and a.has_canonical_format, b
        r = r.sorted_indices()
        assert np.array_equal(a.indptr, r.indptr) and np.array_equal(a.indices, r.indices), b
        assert codes.stats(b) == host.stats(b), b
        if r.nnz == 0:
            continue
        counts = _event_counts(host, b, codes.K)
        cols = np.repeat(np.arange(r.shape[1]), np.diff(r.indptr))
        n_ev = np.array([counts[int(t) * codes.K + int(k)] for t, k in zip(r.indices, cols)])
        few = n_ev <= 2
        assert np.array_equal(a.data[few].view(np.int64), r.data[few].view(np.int64)), b
        assert np.max(np.abs(a.data - r.data)) <= 1e-12 * np.max(np.abs(r.data)), b
    if res_d is not None:
        assert res_d.is_cuda and tuple(res_d.shape) == res_h.shape
        assert np.array_equal(res_d.cpu().numpy().astype(res_h.dtype), res_h)
    if codes.B > 0:
        recon = coder.reconstructBatch(csc)
        dev = coder.reconstructBatchDevice(codes)
        assert dev.is_cuda and str(dev.dtype) == 'torch.float64'
        assert np.array_equal(dev.cpu().numpy(), recon)


def _same(a, b):
    import torch
    (ca, ra), (cb, rb) = a, b
    assert (ca.B, ca.T, ca.K) == (cb.B, cb.T, cb.K)
    for f in ('offsets', 'pos', 'idx', 'coef'):
        assert torch.equal(getattr(ca, f), getattr(cb, f)), f
    assert [bytes(s) for s in ca.states] == [bytes(s) for s in cb.states]
    assert (ra is None) == (rb is None)
    if ra is not None:
        assert torch.equal(ra, rb)


def _mp_cases(small):
    D, X = small
    w = np.random.RandomState(3).uniform(0.5, 1.5, D.shape[0]).astype(np.float32)
    return [
        ('nnz', D, X, dict(nbNonzeroCoefs=40)),
        ('snr', D, X, dict(toleranceSnr=20.0)),
        ('blocks10', D, X, dict(nbNonzeroCoefs=40, nbBlocks=10)),
        ('weights', D, X, dict(nbNonzeroCoefs=40, weights=w)),
        ('float64', D.astype(np.float64), X.astype(np.float64), dict(nbNonzeroCoefs=40)),
    ]


@pytest.mark.gpu
@pytest.mark.parametrize('case', ['nnz', 'snr', 'blocks10', 'weights', 'float64'])
def test_mp_matches_encode_batch(hsc, small, case):
    name, D, X, kw = next(c for c in _mp_cases(small) if c[0] == case)
    coder = hsc.ConvolutionalSparseCoder(D, hsc.ConvolutionalMatchingPursuit())
    codes, res = coder.encodeBatchDevice(X, **kw)
    assert isinstance(codes, hsc.SparseCodes) and codes.K == D.shape[0] and codes.T == X.shape[1]
    assert codes.offsets.is_cuda and codes.coef.is_cuda and str(codes.coef.dtype) == 'torch.float64'
    assert str(res.dtype) == ('torch.float64' if X.dtype == np.float64 else 'torch.float32')
    _check_against_batch(coder, X, kw, codes, res)
    _same((codes, res), coder.encodeBatchDevice(X, **kw))                  # deterministic


@pytest.mark.gpu
def test_2d_signals_with_2d_dictionary(hsc):
    D, X = _workload(5, 3000, 1, 12, 24, 30, 21)
    D2, X2 = D[:, :, 0], X[:, :, 0]
    coder = hsc.ConvolutionalSparseCoder(D2, hsc.ConvolutionalMatchingPursuit())
    kw = dict(toleranceSnr=15.0)
    codes, res = coder.encodeBatchDevice(X2, **kw)
    assert tuple(res.shape) == X2.shape
    _check_against_batch(coder, X2, kw, codes, res)
    assert tuple(coder.reconstructBatchDevice(codes).shape) == X2.shape


@pytest.mark.gpu
def test_locomp_config4_like_fast_kernel(hsc):
    """Config 4's filters (256 x 64, 4 channels, float32: the fast LoCOMP kernel) on shorter signals."""
    D, X = _workload(3, 8192, 4, 256, 64, 80, 31)
    coder = hsc.ConvolutionalSparseCoder(D, hsc.LoCOMP())
    kw = dict(nbNonzeroCoefs=80)
    codes, res = coder.encodeBatchDevice(X, **kw)
    _check_against_batch(coder, X, kw, codes, res)


@pytest.mark.gpu
def test_locomp_narrow_float64(hsc):
    D, X = _workload(4, 2048, 1, 8, 16, 25, 41)
    D, X = D.astype(np.float64), X.astype(np.float64)
    coder = hsc.ConvolutionalSparseCoder(D, hsc.LoCOMP())
    kw = dict(toleranceSnr=25.0)
    codes, res = coder.encodeBatchDevice(X, **kw)
    _check_against_batch(coder, X, kw, codes, res)


@pytest.mark.gpu
@pytest.mark.parametrize('chunk', [1, 3])
def test_chunk_boundaries_do_not_change_the_result(hsc, monkeypatch, chunk):
    D, X = _workload(7, 4096, 4, 32, 16, 40, 51)
    coder = hsc.ConvolutionalSparseCoder(D, hsc.ConvolutionalMatchingPursuit())
    kw = dict(toleranceSnr=20.0)
    one = coder.encodeBatchDevice(X, **kw)
    sizes = []
    begin = hsc.engine.EncodeSlot.begin
    monkeypatch.setattr(hsc.Engine, '_stream_chunk_size', lambda self, T, cap, n, opt: chunk)
    monkeypatch.setattr(hsc.engine.EncodeSlot, 'begin', lambda self, xd, *a, **k: sizes.append(int(xd.shape[0])) or begin(self, xd, *a, **k))
    _same(coder.encodeBatchDevice(X, **kw), one)
    assert sizes == ([1] * 7 if chunk == 1 else [2, 2, 3])                 # balanced chunks, the last one uneven
    # the same with the input read in place from the device, and from a pinned host tensor
    import torch
    xd = torch.from_numpy(X).cuda()
    _same(coder.encodeBatchDevice(xd, **kw), one)
    _same(coder.encodeBatchDevice(torch.from_numpy(X).pin_memory(), **kw), one)


def _locomp_rerun_input(hsc):
    from oracle import hsc_oracle as O
    rs = np.random.RandomState(77)
    T, K, L = 4096, 6, 32
    D = O.normalize(rs.randn(K, L))
    dense = np.zeros(T)
    for p in range(L, T - L, 2):                     # overlapping atoms every 2 samples: many events per signal
        O.overlap_add(dense[:, None], rs.randn() * D[rs.randint(K)][:, None], p)
    sparse = np.zeros(T)
    for p in rs.randint(L, T - L, 20):
        O.overlap_add(sparse[:, None], rs.uniform(1, 2) * D[rs.randint(K)][:, None], p)
    return D, np.stack([sparse, dense + 1e-3 * rs.randn(T), sparse[::-1].copy()])


@pytest.mark.gpu
@pytest.mark.parametrize('method', ['mp', 'locomp'])
def test_capacity_rerun(hsc, small, monkeypatch, method):
    """Event buffers too small for some signals: their chunk runs again with 8x the buffers, and the result equals the
    run whose buffers were large enough from the start."""
    if method == 'mp':
        D, X = small
        approx, kw, small_cap = hsc.ConvolutionalMatchingPursuit(), dict(toleranceSnr=20.0), 16
    else:
        D, X = _locomp_rerun_input(hsc)
        approx, kw, small_cap = hsc.LoCOMP(), dict(toleranceSnr=40.0), 512      # LoCOMP's least capacity
    coder = hsc.ConvolutionalSparseCoder(D, approx)
    normal = coder.encodeBatchDevice(X, **kw)
    assert max(normal[0].stats(b)['n_events'] for b in range(len(X))) > small_cap
    caps = []
    pass_ = hsc.Engine._stream_pass
    monkeypatch.setattr(hsc.Engine, 'default_capacity', lambda self, options, T: small_cap)
    monkeypatch.setattr(hsc.Engine, '_stream_pass', lambda self, x, r, o, cap, *a: caps.append(cap) or pass_(self, x, r, o, cap, *a))
    _same(coder.encodeBatchDevice(X, **kw), normal)
    assert caps[0] == small_cap and len(caps) >= 2 and caps[1] == 8 * small_cap, caps


@pytest.mark.gpu
def test_input_variants(hsc, small):
    import torch
    D, X = small
    coder = hsc.ConvolutionalSparseCoder(D, hsc.ConvolutionalMatchingPursuit())
    kw = dict(nbNonzeroCoefs=40)
    ref = coder.encodeBatchDevice(X, **kw)                                          # numpy
    _same(coder.encodeBatchDevice(torch.from_numpy(X), **kw), ref)                  # unpinned host tensor
    _same(coder.encodeBatchDevice(torch.from_numpy(X).pin_memory(), **kw), ref)     # pinned host tensor
    xd = torch.from_numpy(X).cuda()
    keep = xd.clone()
    _same(coder.encodeBatchDevice(xd, **kw), ref)                                   # CUDA tensor, read in place
    assert torch.equal(xd, keep)
    wide = torch.zeros((X.shape[0], X.shape[1], 2 * X.shape[2]), dtype=torch.float32, device='cuda')
    wide[:, :, ::2] = xd
    assert not wide[:, :, ::2].is_contiguous()
    _same(coder.encodeBatchDevice(wide[:, :, ::2], **kw), ref)                      # non-contiguous CUDA tensor
    ref64 = coder.encodeBatchDevice(X.astype(np.float64), **kw)                     # float64 signals: a float64 engine
    _same(coder.encodeBatchDevice(xd.double(), **kw), ref64)                        # CUDA tensor of another dtype
    _check_against_batch(coder, X.astype(np.float64), kw, *ref64)
    one = coder.encodeBatchDevice(X[:1], **kw)                                      # B = 1
    _check_against_batch(coder, X[:1], kw, *one)
    codes0, res0 = coder.encodeBatchDevice(X[:0], **kw)                             # B = 0
    assert codes0.B == 0 and codes0.to_csc() == [] and int(codes0.offsets.numel()) == 1
    assert tuple(res0.shape) == (0,) + X.shape[1:] and res0.is_cuda
    assert tuple(coder.reconstructBatchDevice(codes0).shape) == (0,) + X.shape[1:]
    codes_nr, res_nr = coder.encodeBatchDevice(X, returnResidual=False, **kw)       # no residual
    assert res_nr is None
    _same((codes_nr, None), (ref[0], None))
    with pytest.raises(AssertionError):
        coder.encodeBatchDevice(X[:, :, :2], **kw)                                  # 2 channels for a 4-channel dictionary


@pytest.mark.gpu
@pytest.mark.parametrize('min_coef', [None, 1e-16, 0.5])
def test_min_coefficients(hsc, small, min_coef):
    D, X = small
    coder = hsc.ConvolutionalSparseCoder(D, hsc.ConvolutionalMatchingPursuit())
    kw = dict(nbNonzeroCoefs=40, minCoefficients=min_coef)
    codes, res = coder.encodeBatchDevice(X, **kw)
    _check_against_batch(coder, X, kw, codes, res)
    if min_coef == 0.5:                                # the threshold removes real entries (amplitudes are U(0.25, 4))
        kept = int(codes.offsets[-1])
        full = coder.encodeBatchDevice(X, nbNonzeroCoefs=40)[0]
        assert 0 < kept < int(full.offsets[-1])
        assert float(codes.coef.abs().min()) >= 0.5


# ---------------------------------------------------------------------------------------------------- host only
def test_sparse_codes_to_csc_on_host_tensors():
    import torch
    from hierarchical_sparse_coding_b200 import SparseCodes
    from hierarchical_sparse_coding_b200 import _native as N
    T, K = 6, 5
    # signal 0 has (1,2), signal 1 is empty, signal 2 has (0,0) and (4,1)
    off = torch.tensor([0, 1, 1, 3])
    pos = torch.tensor([1, 0, 4], dtype=torch.int32)
    idx = torch.tensor([2, 0, 1], dtype=torch.int32)
    coef = torch.tensor([0.5, -1.0, 2.0], dtype=torch.float64)
    states = [N.SignalState() for _ in range(3)]
    states[2].status, states[2].n_events, states[2].nnz = N.HSC_STOP_NNZ, 3, 2
    codes = SparseCodes(3, T, K, off, pos, idx, coef, states)
    csc = codes.to_csc()
    dense = [np.zeros((T, K)) for _ in range(3)]
    dense[0][1, 2] = 0.5
    dense[2][0, 0] = -1.0
    dense[2][4, 1] = 2.0
    assert len(csc) == 3
    for b in range(3):
        m = csc[b]
        assert m.format == 'csc' and m.dtype == np.float64 and m.shape == (T, K) and m.has_canonical_format
        assert np.array_equal(m.toarray(), dense[b]), b
    assert csc[1].nnz == 0
    st = codes.stats(2)
    assert st['stop'] == 'nnz' and st['n_events'] == 3 and st['nnz'] == 2
    assert SparseCodes(0, T, K, torch.zeros(1, dtype=torch.int64), pos[:0], idx[:0], coef[:0], []).to_csc() == []
