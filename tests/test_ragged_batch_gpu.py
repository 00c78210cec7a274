"""Ragged batches: ConvolutionalSparseCoder.encodeBatchDevice(X, lengths=...) on a padded batch against encodeBatchDevice of
each signal alone, at its own length, with the same keywords.  Codes, raw states and residual[b, :lengths[b]] must agree bit
for bit, the residual past a signal's length must be 0, and reconstructBatchDevice must give the signal's own
reconstruction with a zero tail.  Both encodes take the same kernel paths at these shapes (T_max <= 131072, T_max*K < 2^31:
see tests/test_encode_batch_device_gpu.py).

The lengths cover the places where a bound changes meaning: 1 and L-1 (every atom an edge atom), 127 / 128 / 129 (the
128-row groups of the argmax hierarchy), 4095 / 4096 / 4097 (blocks of 32 groups), T_max-1, T_max and seeded random ones."""
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


def _lengths(T, L, seed, n_random=3):
    """Boundary lengths that fit in T, then seeded random ones."""
    fixed = [T, 1, L - 1, 127, 128, 129, 4095, 4096, 4097, T - 1]
    out = []
    for n in fixed:
        if 1 <= n <= T and n not in out:
            out.append(n)
    rs = np.random.RandomState(seed)
    out += [int(n) for n in rs.randint(1, T + 1, n_random)]
    return np.array(out, dtype=np.int64)


def _padded(X, lengths, fill=0.0):
    """The signals of X cut to their lengths, padded back to X's length with `fill`."""
    P = X.copy()
    for b, n in enumerate(lengths):
        P[b, n:] = fill
    return P


def _check_ragged(coder, X, lengths, kw, codes, res):
    """Signal by signal against encodeBatchDevice of X[b:b+1, :lengths[b]] alone."""
    import torch
    B, T = X.shape[0], X.shape[1]
    assert codes.B == B and codes.T == T and codes.lengths is not None
    assert codes.lengths.dtype == np.int64 and np.array_equal(codes.lengths, lengths)
    csc = codes.to_csc()
    recon = coder.reconstructBatchDevice(codes)
    assert tuple(recon.shape[:2]) == (B, T)
    res_h = None if res is None else res.cpu().numpy()
    recon_h = recon.cpu().numpy()
    for b, n in enumerate(lengths):
        n = int(n)
        one, one_res = coder.encodeBatchDevice(X[b:b + 1, :n], **kw)
        ref = one.to_csc()[0]
        got = csc[b]
        assert got.shape == (n, codes.K) == ref.shape, b
        assert np.array_equal(got.indptr, ref.indptr) and np.array_equal(got.indices, ref.indices), (b, n)
        assert np.array_equal(got.data.view(np.int64), ref.data.view(np.int64)), (b, n)
        assert bytes(codes.states[b]) == bytes(one.states[0]), (b, n, codes.stats(b), one.stats(0))
        if res_h is not None:
            r1 = one_res.cpu().numpy()[0]
            assert np.array_equal(res_h[b, :n].view(np.uint8), r1.view(np.uint8)), (b, n)
            assert not np.any(res_h[b, n:]), (b, n)
        r_one = coder.reconstructBatchDevice(one).cpu().numpy()[0]
        assert np.array_equal(recon_h[b, :n].view(np.uint8), r_one.view(np.uint8)), (b, n)      # bits: NaN where the code is
        assert not np.any(recon_h[b, n:]), (b, n)
    assert isinstance(recon, torch.Tensor) and recon.is_cuda


def _same(a, b):
    import torch
    (ca, ra), (cb, rb) = a, b
    assert (ca.B, ca.T, ca.K) == (cb.B, cb.T, cb.K)
    for f in ('offsets', 'pos', 'idx', 'coef'):
        assert torch.equal(getattr(ca, f), getattr(cb, f)), f
    assert [bytes(s) for s in ca.states] == [bytes(s) for s in cb.states]
    assert (ra is None) == (rb is None)
    if ra is not None:
        assert torch.equal(ra.contiguous().view(torch.uint8), rb.contiguous().view(torch.uint8))


# ------------------------------------------------------------------------------------------------------------------ MP

@pytest.fixture(scope='module')
def small():
    """16 signals of 8192 x 4 channels, 32 filters of 16 (float32: the tensor-core K1)."""
    return _workload(16, 8192, 4, 32, 16, 60, 101)


def _mp_case(name, small):
    D, X = small
    w = np.random.RandomState(5).uniform(0.5, 1.5, D.shape[0]).astype(np.float32)
    if name == 'nnz':
        return D, X, dict(nbNonzeroCoefs=40)
    if name == 'snr':
        return D, X, dict(toleranceSnr=20.0)
    if name == 'scale':
        return D, X, dict(toleranceResidualScale=0.5, nbNonzeroCoefs=200)
    if name == 'blocks10':
        return D, X, dict(nbNonzeroCoefs=40, nbBlocks=10)
    if name == 'blocks_auto':
        return D, X, dict(toleranceSnr=20.0, nbBlocks='auto')
    if name == 'weights':
        return D, X, dict(nbNonzeroCoefs=40, weights=w)
    if name == 'float64':
        return D.astype(np.float64), X.astype(np.float64), dict(nbNonzeroCoefs=40)
    raise KeyError(name)


@pytest.mark.gpu
@pytest.mark.parametrize('case', ['nnz', 'snr', 'scale', 'blocks10', 'blocks_auto', 'weights', 'float64'])
def test_mp_each_signal_as_if_alone(hsc, small, case):
    D, X, kw = _mp_case(case, small)
    T, L = X.shape[1], D.shape[1]
    lengths = _lengths(T, L, seed=11)
    if case == 'blocks10':
        lengths = lengths[lengths >= 10]            # nbBlocks=10 needs blocks of >= 2 samples in every signal
    X = X[:len(lengths)]
    coder = hsc.ConvolutionalSparseCoder(D, hsc.ConvolutionalMatchingPursuit())
    codes, res = coder.encodeBatchDevice(X, lengths=lengths, **kw)
    _check_ragged(coder, X, lengths, kw, codes, res)


@pytest.mark.gpu
def test_mp_narrow_rows(hsc):
    """K <= 8 floats: the register 'tiny row' window path under the shared-memory hierarchy."""
    D, X = _workload(13, 6000, 1, 8, 16, 40, 121)
    lengths = _lengths(6000, 16, seed=12)
    coder = hsc.ConvolutionalSparseCoder(D, hsc.ConvolutionalMatchingPursuit())
    kw = dict(toleranceSnr=25.0)
    codes, res = coder.encodeBatchDevice(X[:len(lengths)], lengths=lengths, **kw)
    _check_ragged(coder, X[:len(lengths)], lengths, kw, codes, res)


@pytest.mark.gpu
def test_mp_three_channels_simt_k1(hsc):
    """F = 3: the SIMT correlation kernel."""
    D, X = _workload(13, 5000, 3, 24, 12, 40, 131)
    lengths = _lengths(5000, 12, seed=13)
    coder = hsc.ConvolutionalSparseCoder(D, hsc.ConvolutionalMatchingPursuit())
    kw = dict(nbNonzeroCoefs=50)
    codes, res = coder.encodeBatchDevice(X[:len(lengths)], lengths=lengths, **kw)
    _check_ragged(coder, X[:len(lengths)], lengths, kw, codes, res)


@pytest.mark.gpu
def test_mp_config4_filters(hsc):
    """Config 4's filters (256 x 64, 4 channels): shared-memory hierarchy + gram_update_row32."""
    D, X = _workload(13, 8192, 4, 256, 64, 80, 141)
    lengths = _lengths(8192, 64, seed=14)
    coder = hsc.ConvolutionalSparseCoder(D, hsc.ConvolutionalMatchingPursuit())
    kw = dict(toleranceSnr=20.0)
    codes, res = coder.encodeBatchDevice(X[:len(lengths)], lengths=lengths, **kw)
    _check_ragged(coder, X[:len(lengths)], lengths, kw, codes, res)


# ------------------------------------------------------------------------------------------------------------------ LoCOMP

@pytest.mark.gpu
def test_locomp_fast_kernel(hsc):
    D, X = _workload(13, 8192, 4, 256, 64, 80, 151)
    lengths = _lengths(8192, 64, seed=15)
    coder = hsc.ConvolutionalSparseCoder(D, hsc.LoCOMP())
    kw = dict(nbNonzeroCoefs=60)
    codes, res = coder.encodeBatchDevice(X[:len(lengths)], lengths=lengths, **kw)
    _check_ragged(coder, X[:len(lengths)], lengths, kw, codes, res)


@pytest.mark.gpu
def test_locomp_original_kernel_float64_narrow(hsc):
    D, X = _workload(13, 4500, 1, 8, 16, 25, 161)
    D, X = D.astype(np.float64), X.astype(np.float64)
    lengths = _lengths(4500, 16, seed=16)
    coder = hsc.ConvolutionalSparseCoder(D, hsc.LoCOMP())
    kw = dict(toleranceSnr=25.0)
    codes, res = coder.encodeBatchDevice(X[:len(lengths)], lengths=lengths, **kw)
    _check_ragged(coder, X[:len(lengths)], lengths, kw, codes, res)


# ------------------------------------------------------------------------------------------------------------------ padding, uniform, chunking

@pytest.mark.gpu
def test_padding_is_ignored(hsc, small):
    import torch
    D, X = small
    lengths = _lengths(X.shape[1], D.shape[1], seed=17)
    X = X[:len(lengths)]
    coder = hsc.ConvolutionalSparseCoder(D, hsc.ConvolutionalMatchingPursuit())
    kw = dict(toleranceSnr=20.0)
    ref = coder.encodeBatchDevice(_padded(X, lengths, 0.0), lengths=lengths, **kw)
    for fill in (np.nan, 1e30, -1e30):
        _same(coder.encodeBatchDevice(_padded(X, lengths, fill), lengths=lengths, **kw), ref)
    xd = torch.from_numpy(_padded(X, lengths, np.nan)).cuda()
    keep = xd.clone()
    _same(coder.encodeBatchDevice(xd, lengths=lengths, **kw), ref)
    assert torch.equal(xd.view(torch.int32), keep.view(torch.int32))          # the CUDA input, NaN padding included


@pytest.mark.gpu
@pytest.mark.parametrize('method', ['mp', 'locomp'])
def test_full_lengths_equal_uniform(hsc, small, method):
    D, X = small
    coder = hsc.ConvolutionalSparseCoder(D, hsc.ConvolutionalMatchingPursuit() if method == 'mp' else hsc.LoCOMP())
    kw = dict(nbNonzeroCoefs=40)
    uni = coder.encodeBatchDevice(X, **kw)
    assert uni[0].lengths is None
    rag = coder.encodeBatchDevice(X, lengths=[X.shape[1]] * X.shape[0], **kw)
    _same(rag, uni)
    assert [c.shape for c in rag[0].to_csc()] == [c.shape for c in uni[0].to_csc()]
    # a uniform encode on the same engine after a ragged one behaves as before
    _same(coder.encodeBatchDevice(X, **kw), uni)


@pytest.mark.gpu
@pytest.mark.parametrize('chunk', [1, 3])
def test_chunks_do_not_change_the_result(hsc, small, monkeypatch, chunk):
    import torch
    D, X = small
    lengths = _lengths(X.shape[1], D.shape[1], seed=18)
    X = X[:len(lengths)]
    coder = hsc.ConvolutionalSparseCoder(D, hsc.ConvolutionalMatchingPursuit())
    kw = dict(toleranceSnr=20.0)
    one = coder.encodeBatchDevice(X, lengths=lengths, **kw)
    monkeypatch.setattr(hsc.Engine, '_stream_chunk_size', lambda self, T, cap, n, opt: chunk)
    _same(coder.encodeBatchDevice(X, lengths=lengths, **kw), one)
    _same(coder.encodeBatchDevice(torch.from_numpy(X).pin_memory(), lengths=lengths, **kw), one)
    _same(coder.encodeBatchDevice(torch.from_numpy(X).cuda(), lengths=torch.from_numpy(lengths), **kw), one)


@pytest.mark.gpu
@pytest.mark.parametrize('method', ['mp', 'locomp'])
def test_capacity_rerun(hsc, small, monkeypatch, method):
    D, X = small
    lengths = _lengths(X.shape[1], D.shape[1], seed=19)
    X = X[:len(lengths)]
    if method == 'mp':
        approx, kw, small_cap = hsc.ConvolutionalMatchingPursuit(), dict(nbNonzeroCoefs=100), 16
    else:
        approx, kw, small_cap = hsc.LoCOMP(), dict(nbNonzeroCoefs=700), 512      # LoCOMP's least capacity
    coder = hsc.ConvolutionalSparseCoder(D, approx)
    normal = coder.encodeBatchDevice(X, lengths=lengths, **kw)
    caps = []
    pass_ = hsc.Engine._stream_pass
    monkeypatch.setattr(hsc.Engine, 'default_capacity', lambda self, options, T: small_cap)
    monkeypatch.setattr(hsc.Engine, '_stream_pass', lambda self, x, r, o, cap, *a: caps.append(cap) or pass_(self, x, r, o, cap, *a))
    _same(coder.encodeBatchDevice(X, lengths=lengths, **kw), normal)
    assert caps[0] == small_cap and len(caps) >= 2 and caps[1] == 8 * small_cap, caps


@pytest.mark.gpu
def test_2d_input_and_dictionary(hsc):
    D, X = _workload(6, 3000, 1, 12, 24, 30, 171)
    D2, X2 = D[:, :, 0], X[:, :, 0]
    lengths = np.array([3000, 23, 129, 2999, 1000, 1], dtype=np.int64)
    coder = hsc.ConvolutionalSparseCoder(D2, hsc.ConvolutionalMatchingPursuit())
    codes, res = coder.encodeBatchDevice(X2, lengths=lengths, toleranceSnr=15.0)
    assert tuple(res.shape) == X2.shape
    full = hsc.ConvolutionalSparseCoder(D, hsc.ConvolutionalMatchingPursuit())
    _check_ragged(full, X, lengths, dict(toleranceSnr=15.0), *full.encodeBatchDevice(X, lengths=lengths, toleranceSnr=15.0))
    assert np.array_equal(res.cpu().numpy(), full.encodeBatchDevice(X, lengths=lengths, toleranceSnr=15.0)[1].cpu().numpy()[:, :, 0])


# ------------------------------------------------------------------------------------------------------------------ validation

@pytest.mark.parametrize('bad', [[4096, 4096], [4096, 0, 10], [4096, 4097, 10], [4096.0, 100.0, 10.0], [[4096, 1, 1]]])
def test_bad_lengths_raise_without_a_device(bad, monkeypatch):
    import hierarchical_sparse_coding_b200 as hsc
    from hierarchical_sparse_coding_b200 import modeling

    def no_device(*a, **k):
        raise AssertionError('device work before the lengths were checked')
    monkeypatch.setattr(modeling, 'get_engine', no_device)
    monkeypatch.setattr(modeling, 'engine_for_dictionary', no_device)
    D = np.ones((4, 8, 2), np.float32)
    X = np.zeros((3, 4096, 2), np.float32)
    coder = hsc.ConvolutionalSparseCoder(D, hsc.ConvolutionalMatchingPursuit())
    with pytest.raises(ValueError):
        coder.encodeBatchDevice(X, lengths=bad, nbNonzeroCoefs=5)
    with pytest.raises(ValueError):
        hsc.LoCOMP().computeCoefficientsBatchDevice(X, D, lengths=np.array(bad), nbNonzeroCoefs=5)


def test_sparse_codes_lengths_to_csc_on_host():
    import torch
    from hierarchical_sparse_coding_b200.modeling import SparseCodes
    offsets = torch.tensor([0, 2, 2, 3], dtype=torch.int64)
    pos = torch.tensor([0, 4, 6], dtype=torch.int32)
    idx = torch.tensor([1, 0, 2], dtype=torch.int32)
    coef = torch.tensor([1.5, -2.0, 0.25], dtype=torch.float64)
    codes = SparseCodes(3, 10, 3, offsets, pos, idx, coef, [None] * 3, lengths=[5, 1, 7])
    assert codes.lengths.dtype == np.int64 and codes.lengths.tolist() == [5, 1, 7]
    m = codes.to_csc()
    assert [c.shape for c in m] == [(5, 3), (1, 3), (7, 3)]
    assert m[0].toarray()[0, 1] == 1.5 and m[0].toarray()[4, 0] == -2.0 and m[1].nnz == 0 and m[2].toarray()[6, 2] == 0.25
    assert [c.shape for c in SparseCodes(3, 10, 3, offsets, pos, idx, coef, [None] * 3).to_csc()] == [(10, 3)] * 3
    with pytest.raises(ValueError):
        SparseCodes(3, 10, 3, offsets, pos, idx, coef, [None] * 3, lengths=[5, 11, 7])


@pytest.mark.gpu
def test_nb_blocks_too_large_for_one_short_signal(hsc, small):
    D, X = small
    coder = hsc.ConvolutionalSparseCoder(D, hsc.ConvolutionalMatchingPursuit())
    with pytest.raises(hsc.HscError, match='nbBlocks larger than T/2'):
        coder.encodeBatchDevice(X[:1, :9], nbNonzeroCoefs=5, nbBlocks=10)           # the single call
    with pytest.raises(hsc.HscError, match='nbBlocks larger than T/2'):
        coder.encodeBatchDevice(X[:3], lengths=[8192, 9, 4000], nbNonzeroCoefs=5, nbBlocks=10)
