"""Host-side logic of the drop-in layer that needs no GPU: event accumulation into the reference's return type, the
redistribution of the last level's code (hsc/modeling.py:1556-1594), normalize (hsc/utils.py:67-74), option packing,
the tensor-core plan geometry restated from csrc/correlate_tc.cuh."""
import numpy as np
import pytest
import scipy.sparse

from oracle import hsc_oracle as O


def test_encode_result_to_csc_sums_duplicates_and_clips():
    from hierarchical_sparse_coding_b200.engine import EncodeResult
    r = EncodeResult(1, 10, 3)
    r.pos[0] = np.array([2, 5, 2, 7, 7], np.int32)
    r.idx[0] = np.array([1, 0, 1, 2, 2], np.int32)
    r.coef[0] = np.array([1.5, -2.0, 0.25, 1e-20, 1e-20], np.float32)
    m = r.to_csc(0, 1e-16)
    assert m.shape == (10, 3) and m.dtype == np.float64
    assert m.nnz == 2 and m[2, 1] == pytest.approx(1.75) and m[5, 0] == pytest.approx(-2.0)      # (7,2): 2e-20 < 1e-16 dropped (:1171-1177)
    m2 = r.to_csc(0, None)
    assert m2.nnz == 3 and m2[7, 2] == pytest.approx(2e-20, rel=1e-6)                             # minCoefficients=None keeps it
    assert r.total_events() == 5


def test_capacity_escalation_scales_and_limit():
    """The batched encode paths rerun the signal ranges that filled their event buffers with 8x the buffers, up to 4096x."""
    from hierarchical_sparse_coding_b200 import _native as N
    from hierarchical_sparse_coding_b200.engine import escalate_capacity
    seen = []
    with pytest.raises(N.HscError) as e:
        escalate_capacity(lambda ranges, scale: seen.append((ranges, scale)) or ranges, [(0, 4)], 'test')
    assert e.value.code == N.HSC_E_NOMEM and 'event buffers exhausted' in str(e.value)
    assert seen == [([(0, 4)], s) for s in (1, 8, 64, 512, 4096)]
    seen = []
    escalate_capacity(lambda ranges, scale: seen.append((ranges, scale)) or ([(2, 3)] if scale == 1 else []),
                      [(0, 2), (2, 5)], 'test')
    assert seen == [([(0, 2), (2, 5)], 1), ([(2, 3)], 8)]
    escalate_capacity(lambda ranges, scale: pytest.fail('no range to run'), [], 'test')


def test_read_states_classifies_every_status():
    """The per-signal state check of the encode paths, from a ctypes array and from a byte snapshot of one (the pinned
    buffer an asynchronous states copy fills, which may hold more signals than the encode)."""
    import torch
    from hierarchical_sparse_coding_b200 import _native as N
    from hierarchical_sparse_coding_b200.engine import check_refit_groups, read_states
    unfinished = (N.HSC_PAUSE_CAPACITY, N.HSC_PAUSE_PASSES, N.HSC_RUNNING)
    for code in N.STOP_NAMES:
        arr = (N.SignalState * 3)()
        for s in range(3):
            arr[s].status, arr[s].n_events = N.HSC_STOP_SNR, 10 + s
        arr[1].status = code
        snapshot = torch.from_numpy(np.frombuffer(bytes(arr) * 2, np.uint8).copy())
        for src in (arr, snapshot):
            snap, status, paused = read_states(src, 3)
            assert status.dtype == np.int32 and status.tolist() == [N.HSC_STOP_SNR, code, N.HSC_STOP_SNR]
            assert paused == (code in unfinished), N.STOP_NAMES[code]
            assert bytes(snap) == bytes(arr) and [st.n_events for st in snap] == [10, 11, 12]
            assert read_states(src, 1)[1].tolist() == [N.HSC_STOP_SNR] and not read_states(src, 1)[2]
        if code == N.HSC_STOP_GROUP:
            with pytest.raises(NotImplementedError):
                check_refit_groups(status)
        else:
            check_refit_groups(status)
    arr[0].n_events = 99
    assert snap[0].n_events == 10                                                # a private copy


def test_concat_codes_trims_and_rebases():
    import torch
    from hierarchical_sparse_coding_b200.engine import _concat_codes

    def level(offsets, pos):              # canonical codes with room for more entries than they hold (-1: unused room)
        p = torch.tensor(pos, dtype=torch.int32)
        return dict(offsets=torch.tensor(offsets, dtype=torch.int64), pos=p, idx=p + 1, coef=p.double() / 8)
    parts = [(level([0, 2, 3], [10, 11, 12, -1, -1]), 3), (level([0, 0], [-1, -1]), 0), (level([0, 1, 2], [20, 21, -1]), np.int64(2))]
    off, pos, idx, coef = _concat_codes(parts, 'cpu')
    assert off.dtype == torch.int64 and pos.dtype == idx.dtype == torch.int32 and coef.dtype == torch.float64
    assert off.tolist() == [0, 2, 3, 3, 4, 5] and pos.tolist() == [10, 11, 12, 20, 21]
    assert idx.tolist() == [11, 12, 13, 21, 22] and coef.tolist() == [1.25, 1.375, 1.5, 2.5, 2.625]
    off, pos, idx, coef = _concat_codes([], 'cpu')
    assert off.tolist() == [0] and pos.numel() == idx.numel() == coef.numel() == 0
    assert pos.dtype == idx.dtype == torch.int32 and coef.dtype == torch.float64


def test_convert_to_distributed_matches_oracle():
    import hierarchical_sparse_coding_b200.modeling as M
    rs = np.random.RandomState(0)
    T, Ks = 50, (4, 9, 15)
    codes = []
    for K in Ks:
        d = rs.randn(T, K) * (rs.rand(T, K) < 0.1)
        codes.append(scipy.sparse.csc_matrix(d))
    got = M.HierarchicalConvolutionalMatchingPursuit.convertToDistributedCoefficients(None, codes)
    ref = O.distribute_levels(codes)
    assert len(got) == len(ref) == 3
    for g, r in zip(got, ref):
        assert g.shape == r.shape and (g != r).nnz == 0
    assert sum(g.nnz for g in got) == codes[-1].nnz


def test_normalize_matches_reference_semantics():
    import hierarchical_sparse_coding_b200.modeling as M
    rs = np.random.RandomState(1)
    X = rs.randn(5, 7, 3)
    X[2] = 0.0
    n = M.normalize(X)
    assert np.allclose(np.sqrt(np.sum(n[[0, 1, 3, 4]] ** 2, axis=(1, 2))), 1.0) and not n[2].any()       # zero-norm safe
    assert np.allclose(n, O.normalize(X))
    v = rs.randn(9)
    assert np.allclose(M.normalize(v), v / np.linalg.norm(v))                                              # 1-D: whole-vector norm
    assert np.allclose(M.normalize(X, axis=1), O.normalize(X, axis=1))


def test_multilevel_dictionary_holder_and_errors():
    import hierarchical_sparse_coding_b200.modeling as M
    raw = [np.zeros((4, 8)), np.zeros((6, 5, 4))]
    mld = M.MultilevelDictionary(raw, [8, 12], [np.zeros((4, 8)), np.zeros((6, 12))], [4, 2])
    assert mld.getNbLevels() == 2 and mld.getRawDictionary(1).shape == (6, 5, 4) and mld.getBaseDictionary() is raw[0]
    assert M._is_multilevel_dictionary(mld) and not M._is_multilevel_dictionary(object())
    assert mld.withSingletonBases() is mld
    with pytest.raises(AssertionError):
        mld.getRawDictionary(2)
    with pytest.raises(AssertionError):
        M.ConvolutionalSparseCoder(np.zeros(3), None)
    with pytest.raises(Exception):
        M.HierarchicalConvolutionalMatchingPursuit(method='nope')._level_approximator()


def test_learner_samples_and_init_follow_the_reference_random_stream():
    """_train_samples / _init_D consume np.random exactly like the reference (hsc/modeling.py:279-329), so a seeded
    script gets the same initial dictionary."""
    import hierarchical_sparse_coding_b200.modeling as M
    data = np.random.RandomState(3).randn(300)
    np.random.seed(5)
    D = M.ConvolutionalDictionaryLearner(k=6, windowSize=7, algorithm='samples').train(data)
    np.random.seed(5)
    idx = np.random.randint(low=0, high=300 - 7, size=(6,))
    ref = O.normalize(np.stack([data[i:i + 7] for i in idx]))
    assert D.shape == (6, 7) and np.allclose(D, ref)
    np.random.seed(9)
    D0 = M.ConvolutionalDictionaryLearner(k=4, windowSize=5)._init_D(data[:, None], 'noise')
    np.random.seed(9)
    ref0 = O.normalize(np.random.uniform(low=data.min(), high=data.max(), size=(4, 5, 1)))
    assert np.allclose(D0, ref0)
    with pytest.raises(Exception):
        M.ConvolutionalDictionaryLearner(k=4, windowSize=5)._init_D(data, 'bogus')


def test_tensor_core_plan_geometry():
    """The K1 operand geometry documented in DESIGN.md 3 (restated from tc::make_plan): fp16 groups 8/F time steps per
    MMA row, the reduction is padded to a multiple of 16 elements, a slice of NS columns keeps 2*NS*Kd*2 bytes <= 160 KB."""
    def plan(K, L, F, half=True):
        esz = 2 if half else 4
        R = 16 // esz
        if F < 1 or F > R or R % F:
            return None
        kstep = 16 if half else 8
        s = R // F
        Kd = ((L + s - 1) * F + kstep - 1) // kstep * kstep
        npad = (s * K + 31) // 32 * 32
        for ns in (128, 96, 64, 32):
            if npad % ns == 0 and 2 * ns * Kd * esz <= 160 * 1024:
                return dict(s=s, Kd=Kd, Ntot=s * K, NS=ns, nslices=npad // ns)
        return None
    assert plan(256, 64, 4) == dict(s=2, Kd=272, Ntot=512, NS=128, nslices=4)          # config 4
    assert plan(512, 64, 1) == dict(s=8, Kd=80, Ntot=4096, NS=128, nslices=32)         # config 5
    assert plan(16, 32, 1) == dict(s=8, Kd=48, Ntot=128, NS=128, nslices=1)            # config 2
    assert plan(8, 16, 3) is None                                                        # F does not divide 8: SIMT kernel
    assert plan(256, 64, 4, half=False) == dict(s=1, Kd=256, Ntot=256, NS=64, nslices=4)


# The reference's public signatures on the matching-pursuit path (hsc/modeling.py, line numbers in the comments),
# restated so that the test also runs where the reference is not mounted; when it is, the table itself is checked
# against the live reference first.
_REFERENCE_SIGNATURES = {
    ('ConvolutionalDictionaryLearner', '__init__'): [('k', None), ('windowSize', None), ('algorithm', 'kmean'), ('verbose', False)],          # :267
    ('ConvolutionalDictionaryLearner', '_train_samples'): [('data', None), ('avoidSingletons', False)],                                       # :279
    ('ConvolutionalDictionaryLearner', '_train_kmean'): [('data', None), ('nbRandomWindows', None), ('maxIterations', 100), ('tolerance', 0.0),
                                                         ('initMethod', 'random_samples'), ('resetMethod', 'noise'), ('nbAveragedPatches', 8)],  # :420
    ('ConvolutionalDictionaryLearner', '_train_ksvd'): [('data', None), ('method', 'locomp'), ('maxIterations', 100), ('tolerance', 0.0),
                                                        ('nbNonzeroCoefs', None), ('toleranceSnr', 40.0), ('usePCA', False)],                  # :528
    ('ConvolutionalMatchingPursuit', '__init__'): [('verbose', False)],                                                                        # :868
    ('ConvolutionalMatchingPursuit', 'computeCoefficients'): [('sequence', None), ('D', None), ('nbNonzeroCoefs', None), ('toleranceResidualScale', None),
                                                              ('toleranceSnr', None), ('nbBlocks', 1), ('minCoefficients', 1e-16), ('weights', None),
                                                              ('stopCondition', None)],                                                        # :1053
    ('LoCOMP', '__init__'): [('verbose', False)],                                                                                              # :1201
    ('LoCOMP', 'computeCoefficients'): [('sequence', None), ('D', None), ('nbNonzeroCoefs', None), ('toleranceResidualScale', None),
                                        ('toleranceSnr', None), ('nbBlocks', 1), ('minCoefficients', 1e-16), ('weights', None), ('stopCondition', None)],  # :1263
    ('HierarchicalConvolutionalMatchingPursuit', '__init__'): [('method', 'locomp')],                                                          # :1429
    ('HierarchicalConvolutionalMatchingPursuit', 'computeCoefficients'): [
        ('sequence', None), ('multilevelDict', None), ('nbNonzeroCoefs', None), ('toleranceResidualScale', None), ('toleranceSnr', None),
        ('nbBlocks', 1), ('minCoefficients', None), ('singletonWeight', 0.5), ('returnDistributed', True), ('stopCondition', None)],          # :1636
    ('HierarchicalConvolutionalMatchingPursuit', 'computeCoefficientsFromLevel'): [
        ('sequence', None), ('coefficients', None), ('multilevelDict', None), ('nbNonzeroCoefs', None), ('toleranceResidualScale', None),
        ('toleranceSnr', None), ('nbBlocks', 1), ('minCoefficients', None), ('singletonWeight', 0.5), ('stopCondition', None),
        ('returnDistributed', True)],                                                                                                          # :1645
    ('ConvolutionalSparseCoder', '__init__'): [('D', None), ('approximator', None)],                                                           # :1658
    ('HierarchicalConvolutionalSparseCoder', '__init__'): [('multilevelDict', None), ('approximator', None)],                                  # :1673
}


def _params(fn):
    import inspect
    out = []
    for name, p in inspect.signature(fn).parameters.items():
        if name == 'self' or p.kind in (p.VAR_POSITIONAL, p.VAR_KEYWORD):
            continue
        out.append((name, None if p.default is p.empty else p.default))
    return out


def test_drop_in_signatures_match_the_reference():
    """Every reference parameter exists here, in the same order, with the same default (a user who swaps the module gets
    the same behaviour for the same call; ADVICE round 1: the hierarchical default method is 'locomp').  The drop-in may
    append engine-only keywords (device, coef_mode, segmentLength, ...) after the reference's."""
    import os
    import sys
    import hierarchical_sparse_coding_b200.modeling as M
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden'))
    import ref_loader
    if ref_loader.reference_available():
        ref = ref_loader.load_reference().modeling
        for (cls, meth), expected in _REFERENCE_SIGNATURES.items():
            assert _params(getattr(getattr(ref, cls), meth)) == expected, (cls, meth)
    for (cls, meth), expected in _REFERENCE_SIGNATURES.items():
        got = _params(getattr(getattr(M, cls), meth))
        assert got[:len(expected)] == expected, (cls, meth, got)
        for name, default in got[len(expected):]:
            assert default is not None or name in ('device', 'segmentLength', 'initD', 'dtype', 'group'), (cls, meth, name)


def test_event_sparse_converters_match_reference_golden():
    """hsc/dataset.py:798-824 restated in the package (vectorised): same records, same order, same csr matrices as the
    reference produced (tests/golden/converters.npz), and the same as the oracle restatement on random input."""
    import os
    import hierarchical_sparse_coding_b200.dataset as DS
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'converters.npz'), allow_pickle=False)
    T, counts = int(z['T']), [int(c) for c in z['counts']]
    codes = [scipy.sparse.coo_matrix((z['code%d_v' % l], (z['code%d_t' % l], z['code%d_k' % l])), shape=(T, K)).tocsr() for l, K in enumerate(counts)]
    ev = DS.convertSparseMatricesToEvents(codes)
    assert ev.dtype == np.dtype('int32,int32,int32,float32')
    assert np.array_equal(np.stack([ev['f0'], ev['f1'], ev['f2']], axis=1), z['events']) and np.array_equal(ev['f3'], z['events_v'])
    back = DS.convertEventsToSparseMatrices(ev, counts, T)
    for l, m in enumerate(back):
        c = m.tocoo()
        assert m.format == 'csr' and m.shape == (T, counts[l])
        assert np.array_equal(c.row, z['back%d_t' % l]) and np.array_equal(c.col, z['back%d_k' % l]) and np.array_equal(c.data, z['back%d_v' % l])
        assert (m != codes[l]).nnz == 0
    rs = np.random.RandomState(2)
    codes = [scipy.sparse.csc_matrix(rs.randn(80, K) * (rs.rand(80, K) < 0.1)) for K in (3, 5)]
    a, b = DS.convertSparseMatricesToEvents(codes), O.sparse_matrices_to_events(codes)
    assert np.array_equal(a, b)
    assert len(DS.convertSparseMatricesToEvents([])) == 0
    # the engine's per-signal event lists (duplicates allowed) -> the reference's records
    from hierarchical_sparse_coding_b200.engine import EncodeResult
    r = EncodeResult(1, 10, 3)
    r.pos[0], r.idx[0], r.coef[0] = np.array([7, 2, 7], np.int32), np.array([1, 0, 1], np.int32), np.array([1.0, -2.0, 0.5], np.float32)
    e = DS.encodeResultToEvents(r)
    assert [tuple(x) for x in e] == [(2, 0, 0, -2.0), (7, 0, 1, 1.5)]


def test_environment_switches_are_documented():
    """Every HSC_* environment switch the native library or the Python package reads is listed in INTEGRATION.md."""
    import glob
    import os
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    names = set()
    for path in glob.glob(os.path.join(root, 'hierarchical_sparse_coding_b200', 'csrc', '*.cu*')):
        names |= set(re.findall(r'getenv\("(HSC_[A-Z0-9_]+)"\)', open(path).read()))
    for path in glob.glob(os.path.join(root, 'hierarchical_sparse_coding_b200', '*.py')) + [os.path.join(root, 'bench.py')]:
        names |= set(re.findall(r"environ\.get\('(HSC_[A-Z0-9_]+)'", open(path).read()))
    doc = open(os.path.join(root, 'INTEGRATION.md')).read()
    missing = sorted(n for n in names if n not in doc)
    assert names and not missing, missing
