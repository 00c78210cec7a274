"""Host-side mirror of the reference's encoder/decoder API for the matching-pursuit path
(`hsc.modeling`, all citations relative to the reference tree).  Same class names, keyword
arguments, return types and error behaviour; every computation runs in the CUDA engine behind the
C ABI (include/hsc_b200.h).  There is no CPU fallback: constructing an engine without a CUDA
device raises.

    SparseApproximator                         hsc/modeling.py:657-660
    ConvolutionalMatchingPursuit               hsc/modeling.py:866-1186
    HierarchicalConvolutionalMatchingPursuit   hsc/modeling.py:1427-1654
    ConvolutionalSparseCoder                   hsc/modeling.py:1656-1669
    HierarchicalConvolutionalSparseCoder       hsc/modeling.py:1671-1705
    convolve1d / reconstructSignal             hsc/modeling.py:149-188 / :226-263
    ConvolutionalDictionaryLearner (ksvd)      hsc/modeling.py:265-329, :528-655

New entry points (the reference encodes one signal per call, :1664): `computeCoefficientsBatch` /
`encodeBatch` take [B,T,F] and shard nothing themselves - see `distributed.py` for the multi-GPU
partition by independent signals.  The hierarchical coder has them too: one level loop
(`HierarchicalConvolutionalMatchingPursuit._forward_batch`) runs B sequences of one length through every
level at once and `computeCoefficients` is its B = 1 call, so a sequence's codes and residual in a batch
are bit for bit those of its own call.  `reconstructBatch` decodes B codes in one launch
(`Engine.decode_batch`, the kernel behind `Engine.decode` too).  `encodeBatchDevice` runs the same level loop but
keeps the codes (`HierarchicalCodes`) and the residual on the GPU: the last level's events are summed, ordered and
redistributed on the device (`Engine.canonicalize_codes`).
"""
import collections.abc
import copy
import logging

import numpy as np
import scipy.sparse

from .engine import (Engine, get_engine, engine_dtype, engine_for_dictionary, state_stats, read_states, check_refit_groups,
                     escalate_capacity, events_to_csc, _concat_codes)

logger = logging.getLogger(__name__)


class MultilevelDictionary(object):
    """Plain holder with the accessors the hierarchical encoder uses from the reference's
    hsc.dataset.MultilevelDictionary (:110-410): raw per-level dictionaries (singleton bases
    already added), input-level representations, countsNoSingletons.  Any object with the same
    attributes/methods (e.g. the reference's own class) is accepted wherever this one is."""

    def __init__(self, dictionaries, scales, representations, countsNoSingletons, hasSingletonBases=True):
        assert len(dictionaries) > 0 and len(scales) == len(dictionaries)
        self.dictionaries = list(dictionaries)
        self.scales = list(scales)
        self.representations = list(representations)
        self.counts = np.array([d.shape[0] for d in dictionaries], dtype=int)
        self.countsNoSingletons = np.asarray(countsNoSingletons, dtype=int)
        self.hasSingletonBases = hasSingletonBases

    def getNbLevels(self):
        return len(self.scales)

    def getRawDictionary(self, level):
        assert level >= 0 and level < self.getNbLevels()
        return self.dictionaries[level]

    def getBaseDictionary(self):
        return self.dictionaries[0]

    def getMultiscaleDictionaries(self):
        return self.representations

    def withSingletonBases(self):
        if self.hasSingletonBases or self.getNbLevels() == 1:
            return self
        raise NotImplementedError('compose the singleton bases with the reference data model '
                                  '(hsc.dataset.addSingletonBases); it is outside the hot path')


def _codes_to_csc(offsets, pos, idx, coef, T, K):
    """Flat canonical codes of B signals (offsets [B+1], pos, idx, coef tensors) -> B float64 csc matrices [T,K]."""
    off = offsets.cpu().numpy()
    p, i, c = pos.cpu().numpy(), idx.cpu().numpy(), coef.cpu().numpy()
    return [scipy.sparse.csc_matrix((c[a:b].astype(np.float64), (p[a:b], i[a:b])), shape=(T, K)) for a, b in zip(off[:-1], off[1:])]


def _decode_codes_device(eng, offsets, pos, idx, coef, B, T, out):
    """out [B,T,F] (device, float64) += the reconstruction of flat device codes with eng's dictionary, one decoder launch."""
    if B > 0:
        eng.decode_batch_device(*[t.to(eng.device) for t in (offsets, pos, idx, coef)], B, T, out)


class HierarchicalCodes(object):
    """Per-level codes of B sequences of length T, as encodeBatchDevice returns them: level l has K[l] filters and the
    tensors offsets[l] (int64 [B+1], from 0), pos[l], idx[l] (int32) and coef[l] (float64), normally on the GPU.  The
    entries of sequence b are [offsets[l][b], offsets[l][b+1]): one per nonzero (t, k) of its code, in ascending (t, k)
    order, which is the order the batched decoder reads."""

    def __init__(self, B, T, K, offsets, pos, idx, coef):
        self.B, self.T, self.K = int(B), int(T), [int(k) for k in K]
        self.offsets, self.pos, self.idx, self.coef = list(offsets), list(pos), list(idx), list(coef)
        assert len(self.offsets) == len(self.pos) == len(self.idx) == len(self.coef) == len(self.K)

    def to_csc(self):
        """The B lists of per-level float64 csc matrices [T,K_l] (canonical format), the structure encodeBatch returns."""
        levels = [_codes_to_csc(self.offsets[l], self.pos[l], self.idx[l], self.coef[l], self.T, K) for l, K in enumerate(self.K)]
        return [list(b) for b in zip(*levels)]


class SparseCodes(object):
    """Single-level codes of B signals of length T over K filters, as ConvolutionalSparseCoder.encodeBatchDevice returns
    them: offsets (int64 [B+1], from 0), pos, idx (int32) and coef (float64), normally on the GPU.  The entries of signal b
    are [offsets[b], offsets[b+1]): one per nonzero (t, k) of its code, in ascending (t, k) order, which is the order the
    batched decoder reads.  `states` holds the B final per-signal states (host)."""

    def __init__(self, B, T, K, offsets, pos, idx, coef, states):
        self.B, self.T, self.K = int(B), int(T), int(K)
        self.offsets, self.pos, self.idx, self.coef = offsets, pos, idx, coef
        self.states = list(states)
        assert len(self.states) == self.B and int(self.offsets.numel()) == self.B + 1

    def stats(self, b):
        """The dict EncodeResult.stats returns for signal b."""
        return state_stats(self.states[b])

    def to_csc(self):
        """The B float64 csc matrices [T,K] (canonical format) that encodeBatch returns."""
        return _codes_to_csc(self.offsets, self.pos, self.idx, self.coef, self.T, self.K)


def _dict_eps(D):
    """np.finfo(D.dtype).eps (:1057): the energy-stop threshold follows the DICTIONARY's dtype in the reference."""
    dt = np.asarray(D).dtype
    return float(np.finfo(dt).eps) if dt.kind == 'f' else float(np.finfo(np.float64).eps)


def _np_dtype(x):
    """NumPy dtype of an array or a torch tensor."""
    if isinstance(x, np.ndarray):
        return x.dtype
    import torch
    return torch.empty(0, dtype=x.dtype).numpy().dtype


def _is_multilevel_dictionary(obj):
    return all(hasattr(obj, a) for a in ('getNbLevels', 'getRawDictionary', 'getMultiscaleDictionaries',
                                         'countsNoSingletons', 'hasSingletonBases'))


def convolve1d(sequence, filters, padding='valid', device=None):
    """hsc/modeling.py:149-188 on the device: [T] or [T,F] x [K,L] or [K,L,F] -> [T',K] ndarray."""
    sequence = np.asarray(sequence)
    filters = np.asarray(filters)
    x = np.atleast_2d(sequence).reshape((sequence.shape[0], -1))
    L = filters.shape[1]
    F = 1 if filters.ndim == 2 else filters.shape[-1]
    assert F == x.shape[-1]
    if padding not in ('valid', 'same'):
        raise Exception('Padding not supported: %s' % (padding))
    eng = get_engine(device)
    dt = engine_dtype(x, filters)
    eng.set_dictionary(filters, dtype=dt)
    c = eng.correlate(x[None].astype(dt)).cpu().numpy()[0]
    if padding == 'valid':
        off = L // 2 - 1 if L % 2 == 0 else L // 2
        c = c[off:off + x.shape[0] - L + 1]
    return c


def reconstructSignal(coefficients, D, device=None):
    """Sparse decoder (hsc/modeling.py:226-263): float64 like the reference (:238)."""
    assert coefficients.ndim == 1 or coefficients.ndim == 2
    D = np.asarray(D)
    assert D.ndim == 2 or D.ndim == 3
    squeeze = D.ndim == 2
    cx = scipy.sparse.coo_matrix(coefficients)
    eng = get_engine(device)
    out_dtype = cx.dtype if cx.dtype in (np.float32, np.float64) else np.float64
    eng.set_dictionary(D, dtype=np.float64)
    keep = cx.data != 0.0
    sig = eng.decode(cx.row[keep], cx.col[keep], cx.data[keep], cx.shape[0]).cpu().numpy().astype(out_dtype)
    return sig[:, 0] if squeeze else sig


def _decode_codes(eng, codes, T, out):
    """out [S,T,F] (device) += the reconstruction of S codes (csc / any sparse [T,K]) with eng's dictionary, one decoder
    launch.  Each code's atoms are its coo's nonzero entries, the list reconstructSignal decodes."""
    pos, idx, coef = [], [], []
    offsets = np.zeros(len(codes) + 1, dtype=np.int64)
    for s, c in enumerate(codes):
        cx = scipy.sparse.coo_matrix(c)
        assert cx.shape[0] == T, 'every code must have %d rows' % T
        keep = cx.data != 0.0
        pos.append(cx.row[keep])
        idx.append(cx.col[keep])
        coef.append(cx.data[keep])
        offsets[s + 1] = offsets[s] + int(np.count_nonzero(keep))
    cat = lambda a, dt: np.concatenate(a).astype(dt, copy=False) if a else np.zeros(0, dt)
    return eng.decode_batch(offsets, cat(pos, np.int32), cat(idx, np.int32), cat(coef, eng.dtype), len(codes), T, out=out)


def _reconstruct_batch(codes, D, device=None):
    """reconstructSignal for B codes of one shape [T,K] with dictionary D, one decoder launch."""
    D = np.asarray(D)
    assert D.ndim == 2 or D.ndim == 3
    eng = get_engine(device)
    eng.set_dictionary(D, dtype=np.float64)
    dt = np.result_type(*[c.dtype for c in codes])
    out_dtype = dt if dt in (np.float32, np.float64) else np.float64
    sig = _decode_codes(eng, codes, codes[0].shape[0], None).cpu().numpy().astype(out_dtype)
    return sig[:, :, 0] if D.ndim == 2 else sig


def normalize(X, axis=None):
    """hsc/utils.py:67-74: unit L2 norm per leading-axis item (or along `axis`), zero-norm safe.  Host-side
    data preparation (dictionary initialisation), not part of the device path."""
    X = np.asarray(X)
    assert X.ndim >= 1
    if axis is None and X.ndim > 1:
        axis = tuple(range(1, X.ndim))
    l2 = np.sqrt(np.sum(np.square(X), axis=axis, keepdims=True))
    return X / np.where(l2 > 0.0, l2, 1.0)


class ConvolutionalDictionaryLearner(object):
    """Drop-in for the K-SVD path of hsc.modeling.ConvolutionalDictionaryLearner (:265-329, :528-655): the MP /
    LoCOMP inference of every outer iteration and the dictionary-update stage that consumes its codes both run
    on the device (hsc_b200_ksvd_update).  `algorithm='samples'` (random windows of the data, :279-308) is host-side
    initialisation and kept because the reference's scripts build their dictionaries with it; `algorithm='kmean'`
    (convolutional k-means, :420-526, used by scripts/learn_mlcsc_dataset.py to learn the multilevel dictionaries)
    runs its correlation / argmax / cosine-mean step on the device (hsc_b200_kmeans_assign); 'nmf' is a different
    algorithm outside the matching-pursuit path (SURVEY 2, #8) and raises.

    New, beyond the reference (which trains on ONE sequence): `train(X)` also accepts [S,T,F] independent
    sequences, and `segmentLength=` cuts a long sequence into independent segments - the shard BASELINE config 5
    names (a 1e8-sample correlation map does not fit one GPU)."""

    def __init__(self, k, windowSize, algorithm='kmean', verbose=False, device=None, coef_mode=1):
        self.k = k
        self.windowSize = windowSize
        self.algorithm = algorithm
        self.verbose = verbose
        self.fig = None
        self.device = device
        self.coef_mode = coef_mode
        self.history = []          # per outer iteration: dict(alpha, nnz, events, snr_db)

    # -- host-side initialisation, same np.random call sequence as the reference
    def _extract_random_windows(self, data, nbWindows, width):
        assert data.ndim == 1 or data.ndim == 2
        assert nbWindows > 0
        assert width > 0 and width < data.shape[0]
        indices = np.random.randint(low=0, high=data.shape[0] - width, size=(nbWindows,))      # :86-88
        return np.stack([data[i:i + width] for i in indices])

    def _train_samples(self, data, avoidSingletons=False):
        patterns = []
        while len(patterns) < self.k:                                                          # :283-301
            windows = self._extract_random_windows(data, self.k, self.windowSize)
            axes = tuple(range(1, windows.ndim))
            l2norms = np.sqrt(np.sum(np.square(windows), axis=axes))
            if avoidSingletons:
                l0norms = np.sum(windows != 0.0, axis=axes)
                valid = windows[np.where((l2norms > 0.0) & (l0norms > 1))]
            else:
                valid = windows[np.where(l2norms > 0.0)]
            for w in valid:
                patterns.append(w)
                if len(patterns) == self.k:
                    break
        return normalize(np.stack(patterns))

    def _init_D(self, data, initMethod='random_samples'):
        assert data.ndim == 1 or data.ndim == 2
        squeezeOutput = data.ndim == 1
        if squeezeOutput:
            data = data[:, np.newaxis]
        if initMethod == 'noise':                                                              # :320-321
            D = normalize(np.random.uniform(low=np.min(data), high=np.max(data), size=(self.k, self.windowSize, data.shape[-1])))
        elif initMethod == 'random_samples':
            D = normalize(self._extract_random_windows(data, self.k, self.windowSize))
        else:
            raise Exception('Unsupported initialization method: %s' % (initMethod))
        if squeezeOutput:
            D = np.squeeze(D, axis=2)
        return D

    def _train_ksvd(self, data, method='locomp', maxIterations=100, tolerance=0.0, nbNonzeroCoefs=None, toleranceSnr=40.0,
                    usePCA=False, segmentLength=None, initD=None, dtype=None, group=None):
        """hsc/modeling.py:528-641.  `nbNonzeroCoefs` is per sequence / segment.  `dtype=np.float32` runs the
        inference in float32 (tensor-core correlation); the default is the reference's arithmetic, the NumPy
        result type of (data, float64 dictionary) = float64.  The update stage is always float64.
        `group` (a torch.distributed process group, or True for the default one): data-parallel learning - every
        rank passes ITS shard of the sequences / segments; the initial dictionary is rank 0's, the encode is local and
        the update all-reduces one q x q Gram matrix per filter (Engine.ksvd_update), so all ranks return the same D.
        `usePCA=True` (:618-625): first principal component of the mean-centred windows (single process only)."""
        if usePCA and group is not None:
            raise NotImplementedError('usePCA=True under a process group: the window means would have to be shared too')
        if method == 'locomp':
            meth = 1
        elif method == 'cmp':
            meth = 0
        else:
            raise Exception('Unsupported sparse coding method: %s' % (method))
        data = np.asarray(data)
        assert data.ndim in (1, 2, 3)
        squeeze = data.ndim == 1
        if data.ndim == 3:
            x = data
        else:
            x2 = data[:, None] if data.ndim == 1 else data
            if segmentLength is not None:
                nseg = x2.shape[0] // int(segmentLength)
                assert nseg >= 1
                x = x2[:nseg * int(segmentLength)].reshape(nseg, int(segmentLength), x2.shape[-1])
            else:
                x = x2[None]
        S, T, F = x.shape
        if initD is not None:
            D = np.array(initD, dtype=np.float64)
        else:
            D = self._init_D(x.reshape(S * T, F), initMethod='noise')                          # :554
        if D.ndim == 2:
            D = D[:, :, None]
        eng = get_engine(self.device)
        if group is not None:
            import torch
            import torch.distributed as dist
            Dt = torch.from_numpy(np.ascontiguousarray(D, dtype=np.float64)).to(eng.device)
            dist.broadcast(Dt, src=0, group=None if group is True else group)
            D = Dt.cpu().numpy()
        dt = np.dtype(dtype) if dtype is not None else np.dtype(engine_dtype(x, D))
        xe = np.ascontiguousarray(x, dtype=dt)
        energy = float(np.sum(np.square(xe, dtype=np.float64)))
        self.history = []
        n = 0
        alpha = tolerance + 1.0
        import time
        import torch
        xd = resid_buf = resident = None
        while n < maxIterations and alpha > tolerance:
            # coefficient update stage (:580-591)
            t_start = time.perf_counter()
            eng.set_dictionary(D, dtype=dt)
            opt = eng.make_options(nbNonzeroCoefs, None, toleranceSnr, 1, 1e-16, coef_mode=self.coef_mode, method=meth)
            states = None
            if xd is None and resident is None:
                # all sequences resident on the device for the whole training if their maps fit: the events then never
                # leave the device between the encoder and the dictionary update
                resident = S <= eng.max_signals_per_chunk(T)
                if resident:
                    xd = torch.from_numpy(xe).to(eng.device)
                    resid_buf = torch.empty_like(xd)
            if resident:
                cap = eng.default_capacity(opt, T)
                evp, evi, evc, st_arr, _ = eng.encode_device(xd, opt, cap, resid=resid_buf)
                snap, _, unfinished = read_states(st_arr, S)
                # event buffers too small for this stop rule: drain through the host path
                states = None if unfinished else list(snap)
            if states is not None:
                nb = torch.tensor([st.n_buffered for st in states], dtype=torch.int64, device=eng.device)
                mask = torch.arange(evp.shape[1], device=eng.device)[None, :] < nb[:, None]
                sig = torch.arange(S, device=eng.device)[:, None].expand(S, evp.shape[1])[mask]
                pos, idx, coef = evp[mask], evi[mask], evc[mask]
                n_events = int(nb.sum())
            else:
                res = eng.encode_chunked(xe, opt)
                states = res.states
                counts = np.array([len(p) for p in res.pos], dtype=np.int64)
                sig = np.repeat(np.arange(S, dtype=np.int32), counts)
                pos = np.concatenate(res.pos) if S else np.zeros(0, np.int32)
                idx = np.concatenate(res.idx) if S else np.zeros(0, np.int32)
                coef = np.concatenate(res.coef).astype(np.float64) if S else np.zeros(0)
                n_events = int(counts.sum())
            check_refit_groups([st.status for st in states])
            sg, p, ix, c, col_ptr = eng.accumulate_code(sig, pos, idx, coef, S, T, D.shape[0], 1e-16)
            torch.cuda.synchronize(eng.device)
            t_encoded = time.perf_counter()
            # dictionary update stage (:593-633)
            D, c_new, alpha = eng.ksvd_update(D, sg, p, ix, c, col_ptr, S, T, group=group, use_pca=bool(usePCA))
            t_updated = time.perf_counter()
            e_res = float(sum(st.energy_residual for st in states))
            self.history.append(dict(alpha=alpha, nnz=int(c.numel()), events=n_events,
                                     encode_s=t_encoded - t_start, update_s=t_updated - t_encoded,
                                     snr_db=10.0 * np.log10(energy / e_res) if e_res > 0 else float('inf')))
            logger.debug('K-SVD iteration %d: tolerance = %f, sparsity = %f' % (n, alpha, float(c.numel()) / (S * T * D.shape[0])))
            n += 1
        return D[:, :, 0] if squeeze else D


    def _train_kmean(self, data, nbRandomWindows, maxIterations=100, tolerance=0.0, initMethod='random_samples',
                     resetMethod='noise', nbAveragedPatches=8):
        """hsc/modeling.py:420-526 (Dundar et al. 2016, convolutional clustering).  Same np.random call sequence as
        the reference (training windows, initial centroids, resets of empty centroids in filter order); the
        correlation of the windows with the centroids, the per-window argmax and the cosine means run on the device."""
        import torch
        data = np.asarray(data)
        assert data.ndim == 1 or data.ndim == 2
        squeeze = data.ndim == 1
        W = self.windowSize
        windows = self._extract_random_windows(data, nbRandomWindows, 2 * W)                 # :426
        D = self._init_D(data, initMethod)                                                       # :429
        eng = get_engine(self.device)
        w3 = windows[:, :, None] if squeeze else windows
        dt = np.dtype(engine_dtype(w3, D))
        wd = torch.from_numpy(np.ascontiguousarray(w3, dtype=dt)).to(eng.device)
        self.history = []
        n = 0
        alpha = tolerance + 1.0
        while n < maxIterations and alpha > tolerance:
            eng.set_dictionary(D, dtype=dt)
            pos, idx, sums, counts = eng.kmeans_assign(wd)                                       # :455-470
            counts_h = counts.cpu().numpy()
            sums_h = sums.cpu().numpy()
            first_assignment = int(idx[0].item())                                                # centroid of window 0
            pos_h = None
            nbResets = 0
            centroids = []
            out_dtype = w3.dtype            # dtype of the reference's stacked centroids: the windows', float64 once a 'noise' reset joins
            for c in range(D.shape[0]):                                                          # :473-510
                # the reference's empty test is `np.any(np.where(assignments == c))` (:479-481): it looks at the INDICES of
                # the centroid's windows, so a centroid whose only window is window 0 is reset like an empty one
                owns_a_window = counts_h[c] > 1 or (counts_h[c] == 1 and first_assignment != c)
                if owns_a_window:
                    centroid = sums_h[c] / float(counts_h[c])                                    # cosine mean (:480)
                else:
                    if pos_h is None:
                        pos_h = pos.cpu().numpy()
                    patch = lambda b: w3[b, pos_h[b]:pos_h[b] + W]
                    if resetMethod == 'random_samples':
                        centroid = patch(np.random.randint(low=0, high=w3.shape[0])).astype(np.float64)
                    elif resetMethod == 'random_samples_average':
                        indices = np.random.randint(low=0, high=w3.shape[0], size=(nbAveragedPatches,))
                        centroid = np.mean(np.stack([patch(b) for b in indices]), axis=0, dtype=np.float64)
                    elif resetMethod == 'noise':
                        centroid = np.random.uniform(low=-1.0, high=1.0, size=(W,) if squeeze else (W, w3.shape[2]))   # :491
                        out_dtype = np.result_type(out_dtype, np.float64)
                    else:
                        raise Exception('Unsupported reset method: %s' % (resetMethod))
                    nbResets += 1
                centroid = np.asarray(centroid, dtype=np.float64).reshape((W, w3.shape[2]))
                if np.sqrt(np.sum(np.square(centroid))) == 0.0:                                  # :499-502
                    centroid = centroid + 1e-9
                centroids.append(centroid)
            newD = normalize(np.stack(centroids))
            if squeeze:
                newD = newD[:, :, 0]
            newD = newD.astype(out_dtype)
            alpha = float(np.sqrt(np.sum(np.square(D - newD))))                                  # :517
            self.history.append(dict(alpha=alpha, resets=nbResets))
            logger.debug('K-mean iteration %d: tolerance = %f, nb resets = %d' % (n, alpha, nbResets))
            D = newD
            n += 1
        return D

    def train(self, X, *args, **kwargs):
        if self.algorithm == 'samples':
            D = self._train_samples(X, *args, **kwargs)
        elif self.algorithm == 'ksvd':
            D = self._train_ksvd(X, *args, **kwargs)
        elif self.algorithm == 'kmean':
            D = self._train_kmean(X, *args, **kwargs)
        elif self.algorithm in ('nmf',):
            raise NotImplementedError('algorithm %r is outside the matching-pursuit path this engine replaces' % (self.algorithm,))
        else:
            raise Exception('Unknown training algorithm: %s' % (self.algorithm))
        return D


class SparseApproximator(object):

    def computeCoefficients(self, X, D):
        raise NotImplementedError()


class ConvolutionalMatchingPursuit(SparseApproximator):
    """Drop-in for hsc.modeling.ConvolutionalMatchingPursuit (:866-1186) on the B200 engine."""

    _method = 0          # hsc_mp_options.method: 0 = MP, 1 = LoCOMP

    def __init__(self, verbose=False, device=None, coef_mode=1):
        self.verbose = verbose
        self.device = device
        self.coef_mode = coef_mode
        self.last_result = None

    def _engine(self):
        return get_engine(self.device)

    def _encode(self, sequences, D, nbNonzeroCoefs, toleranceResidualScale, toleranceSnr, nbBlocks, minCoefficients,
                weights, stopCondition, max_events_total=0):
        eng = self._engine()
        dt = engine_dtype(sequences, D)
        eng.set_dictionary(D, weights=weights, dtype=dt)
        opt = eng.make_options(nbNonzeroCoefs, toleranceResidualScale, toleranceSnr, nbBlocks, minCoefficients,
                               use_weights=weights is not None, coef_mode=self.coef_mode,
                               max_passes_per_run=1 if stopCondition is not None else 0,
                               max_events_total=max_events_total, method=self._method, energy_eps=_dict_eps(D))
        on_pass = None
        if stopCondition is not None:
            x0 = np.asarray(sequences[0])

            def on_pass(res, states):
                if self._method == 1:       # LoCOMP's callback takes the code only (hsc/modeling.py:1395-1396)
                    return bool(stopCondition(res.to_csc(0, None).tolil()))
                # hsc/modeling.py:1155-1158: stopCondition(sequence, residual, coefficients)
                return bool(stopCondition(x0, res.residual[0].cpu().numpy(), res.to_csc(0, None).tolil()))
        res = eng.encode(np.ascontiguousarray(sequences, dtype=dt), opt, on_pass=on_pass)
        self.last_result = res
        check_refit_groups([st.status for st in res.states])
        return res

    def computeCoefficients(self, sequence, D, nbNonzeroCoefs=None, toleranceResidualScale=None, toleranceSnr=None,
                            nbBlocks=1, minCoefficients=1e-16, weights=None, stopCondition=None):
        sequence = np.asarray(sequence)
        D = np.asarray(D)
        assert sequence.ndim == 1 or sequence.ndim == 2
        assert D.ndim == 2 or D.ndim == 3
        squeezeOutput = sequence.ndim == 1 or D.ndim == 2
        x = sequence[:, None] if sequence.ndim == 1 else sequence
        if weights is not None:
            assert len(weights) == D.shape[0]
        res = self._encode(x[None], D, nbNonzeroCoefs, toleranceResidualScale, toleranceSnr, nbBlocks, minCoefficients,
                           weights, stopCondition)
        st = res.stats(0)
        logger.debug('SNR stop=%s after %d selection iterations; nnz=%d duplicates=%d', st['stop'], st['passes'],
                     st['nnz'], st['duplicates'])
        if st['stop'] == 'empty':
            logger.warning('Selection returned empty set: considering convergence is achieved')
        coefficients = res.to_csc(0, minCoefficients)
        residual = res.residual[0].cpu().numpy().astype(sequence.dtype if sequence.dtype.kind == 'f' else np.float64)
        if squeezeOutput:
            residual = np.squeeze(residual, axis=1)
        return coefficients, residual

    def computeCoefficientsBatch(self, sequences, D, nbNonzeroCoefs=None, toleranceResidualScale=None, toleranceSnr=None,
                                 nbBlocks=1, minCoefficients=1e-16, weights=None):
        """[B,T] or [B,T,F] -> (list of csc_matrix [T,K], residual ndarray like the input)."""
        sequences = np.asarray(sequences)
        D = np.asarray(D)
        assert sequences.ndim == 2 or sequences.ndim == 3
        assert D.ndim == 2 or D.ndim == 3
        x = sequences[:, :, None] if sequences.ndim == 2 else sequences
        eng = self._engine()
        dt = engine_dtype(x, D)
        eng.set_dictionary(D, weights=weights, dtype=dt)
        opt = eng.make_options(nbNonzeroCoefs, toleranceResidualScale, toleranceSnr, nbBlocks, minCoefficients,
                               use_weights=weights is not None, coef_mode=self.coef_mode, method=self._method, energy_eps=_dict_eps(D))
        res = eng.encode_host(np.ascontiguousarray(x, dtype=dt), opt, n_chunks=max(1, min(8, x.shape[0] // 32)))
        self.last_result = res
        codes = [res.to_csc(s, minCoefficients) for s in range(res.S)]
        residual = res.residual.numpy().astype(sequences.dtype if sequences.dtype.kind == 'f' else np.float64)
        if sequences.ndim == 2:
            residual = residual[:, :, 0]
        return codes, residual

    def computeCoefficientsBatchDevice(self, sequences, D, nbNonzeroCoefs=None, toleranceResidualScale=None, toleranceSnr=None,
                                       nbBlocks=1, minCoefficients=1e-16, weights=None, returnResidual=True):
        """computeCoefficientsBatch with the codes and the residual left on the GPU, for batches of any size.  sequences
        [B,T] or [B,T,F]: a numpy array, a host torch tensor (a pinned one of the engine dtype is copied to the device
        without staging) or a CUDA tensor on the coder's device (read in place, never modified, when it is contiguous and of
        the engine dtype).  Keywords and dtype rules are those of computeCoefficientsBatch.  Returns (SparseCodes, residual):
        the residual a CUDA tensor of the engine dtype shaped like computeCoefficientsBatch's ([B,T] for 2-D sequences), or
        None with returnResidual=False.  The signals run in chunks through two encodes in flight (Engine.encode_stream_device);
        the codes are summed, ordered and thresholded on the device (Engine.canonicalize_codes).  Duplicate events are summed
        in selection order, which the host path does not guarantee for three or more events of one (t, k), so such a value
        may differ from computeCoefficientsBatch's in the last bits; sparsity pattern, states and residual are the same."""
        import torch
        if not isinstance(sequences, torch.Tensor):
            sequences = np.asarray(sequences)
        D = np.asarray(D)
        assert sequences.ndim == 2 or sequences.ndim == 3
        assert D.ndim == 2 or D.ndim == 3
        x = sequences[:, :, None] if sequences.ndim == 2 else sequences
        eng = self._engine()
        dt = engine_dtype(np.zeros(0, _np_dtype(x)), D)
        eng.set_dictionary(D, weights=weights, dtype=dt)
        opt = eng.make_options(nbNonzeroCoefs, toleranceResidualScale, toleranceSnr, nbBlocks, minCoefficients,
                               use_weights=weights is not None, coef_mode=self.coef_mode, method=self._method, energy_eps=_dict_eps(D))
        offsets, pos, idx, coef, states, residual = eng.encode_stream_device(x, opt, min_coefficients=minCoefficients,
                                                                             want_residual=returnResidual)
        codes = SparseCodes(x.shape[0], x.shape[1], eng.K, offsets, pos, idx, coef, states)
        if residual is not None and sequences.ndim == 2:
            residual = residual[:, :, 0]
        return codes, residual

    def reconstructBatchDevice(self, codes, D):
        """The float64 reconstruction of SparseCodes on the device, one decoder launch: [B,T] for a 2-D dictionary, else
        [B,T,F]; equal to ConvolutionalSparseCoder.reconstructBatch(codes.to_csc()) bit for bit."""
        import torch
        D = np.asarray(D)
        assert D.ndim == 2 or D.ndim == 3
        eng = engine_for_dictionary(D, None, np.float64, self.device)
        recon = torch.zeros((codes.B, codes.T, eng.F), dtype=torch.float64, device=eng.device)
        _decode_codes_device(eng, codes.offsets, codes.pos, codes.idx, codes.coef, codes.B, codes.T, recon)
        return recon[:, :, 0] if D.ndim == 2 else recon


class LoCOMP(ConvolutionalMatchingPursuit):
    """Drop-in for hsc.modeling.LoCOMP (:1191-1425): MP plus a local least-squares refit of the selected atom and
    the already-selected atoms sharing its support, on the device (csrc/locomp.cuh)."""
    _method = 1

    def __init__(self, verbose=False, device=None, coef_mode=1):
        super(LoCOMP, self).__init__(verbose, device, coef_mode)


class HierarchicalConvolutionalMatchingPursuit(SparseApproximator):
    """Drop-in for hsc.modeling.HierarchicalConvolutionalMatchingPursuit (:1427-1654): the level loop
    (each level's input is the previous level's dense code map, :1489), singleton weights
    (:1448-1450), redistribution (:1556-1594) and the input-level residual (:1596-1611)."""

    def __init__(self, method='locomp', device=None, coef_mode=1):          # the reference's default (:1429)
        self.method = method
        self.device = device
        self.coef_mode = coef_mode

    def _level_approximator(self):
        if self.method == 'cmp':
            return ConvolutionalMatchingPursuit(device=self.device, coef_mode=self.coef_mode)
        if self.method == 'locomp':
            return LoCOMP(device=self.device, coef_mode=self.coef_mode)
        raise Exception('Unsupported sparse coding method: %s' % (self.method))

    def _forward(self, sequence, coefficients, multilevelDict, toleranceSnr, nbBlocks, singletonWeight):
        """The forward phase (:1432-1492 / :1494-1554) of one sequence: the B = 1 call of _forward_batch.  With given
        `coefficients` (computeCoefficientsFromLevel) the loop starts at the next level, its input the dense map of the last
        given level (:1498)."""
        given = list(coefficients)
        x0 = np.asarray(sequence) if len(given) == 0 else np.asarray(given[-1].todense())
        x0 = x0[:, None] if x0.ndim == 1 else x0
        return self._forward_batch(x0[None], given, multilevelDict, toleranceSnr, nbBlocks, singletonWeight)[0]

    def _forward_batch(self, x, given, multilevelDict, toleranceSnr, nbBlocks, singletonWeight, bounds=None):
        """The forward phase of B independent sequences x [B,T,F] (the input of level len(given)) with the level hand-off ON
        THE DEVICE: level l's events stay in device memory, hsc_b200_mp_events_to_dense turns them into the dense float64
        code map that is level l+1's K_l-channel input (:1489), and every level's dictionary lives in its own native engine,
        so nothing is uploaded twice.  The signals run in chunks that fit the device (_encode_pass); per chunk the host reads
        every level's events once, at the end, and builds the csc matrices the reference returns.  Returns one list per
        sequence: the given codes followed by one csc [T,K_l] per encoded level.  x may also be a torch tensor.  With
        `bounds` (the device path, see _forward_chunk) returns instead a dict: first signal of each chunk -> what
        _forward_chunk returns for it."""
        if self.method == 'cmp':
            meth = 0
        elif self.method == 'locomp':
            meth = 1
        else:
            raise Exception('Unsupported sparse coding method: %s' % (self.method))
        B, T = x.shape[0], x.shape[1]
        out = [list(given) for _ in range(B)] if bounds is None else {}
        if len(given) >= multilevelDict.getNbLevels() or B == 0:
            return out
        specs = []               # (D, weights, engine dtype, options, K, level) per encoded level
        for level in range(len(given), multilevelDict.getNbLevels()):
            if toleranceSnr is not None and isinstance(toleranceSnr, collections.abc.Iterable):
                targetSnr = toleranceSnr[level]
            else:
                targetSnr = toleranceSnr
            D = np.asarray(multilevelDict.getRawDictionary(level))
            assert D.ndim == 2 or D.ndim == 3
            nbSingletons = D.shape[0] - multilevelDict.countsNoSingletons[level]
            weights = np.ones((D.shape[0],), dtype=D.dtype)                     # :1448-1450
            weights[:nbSingletons] = singletonWeight
            # the first level encodes the input; later levels the dense code map, which is float64 (:1489)
            dt = engine_dtype(np.zeros(0, _np_dtype(x)), D) if not specs else engine_dtype(np.zeros(0, np.float64), D)
            eng = engine_for_dictionary(D, weights, dt, self.device)
            opt = eng.make_options(None, None, targetSnr, nbBlocks, 1e-16, use_weights=True, coef_mode=self.coef_mode, method=meth,
                                   energy_eps=_dict_eps(D))
            specs.append((D, weights, dt, opt, D.shape[0], level))
        escalate_capacity(lambda ranges, scale: self._encode_pass(x, ranges, specs, scale, out, bounds), [(0, B)],
                          'hierarchical encode')
        for (D, weights, dt, _, _, _) in specs:
            eng = engine_for_dictionary(D, weights, dt, self.device)
            ws = getattr(eng, '_ws_cache', None)
            if ws is not None and ws.numel() > (256 << 20):      # the per-level engines outlive the call: do not pin large maps
                eng._ws_cache = eng._last_workspace = None
        return out

    def _chunk_size(self, T, specs, cap_scale):
        """Signals per chunk: every level's workspace, its input and residual, the dense hand-off [S,T,K_l] float64 and the
        event buffers (padded and compacted) of all levels, and the device path's canonical codes of the last level (one
        set of float64 buffers per level, plus the sort scratch) fit 80 % of the free device memory; at most 65535 signals
        (hsc_b200_mp_begin)."""
        per = 0
        eng = None
        for (D, weights, dt, opt, K, _) in specs:
            eng = engine_for_dictionary(D, weights, dt, self.device)
            cap = eng.default_capacity(opt, T) * cap_scale
            per += eng.workspace_bytes(1, T) + 2 * T * eng.F * eng.dtype.itemsize + T * K * 8 + 2 * cap * (8 + eng.dtype.itemsize)
        per += cap * (16 * len(specs) + 12)
        return int(max(1, min(65535, int(eng._free_device_bytes() * 0.8) // per)))

    def _encode_pass(self, x, ranges, specs, cap_scale, out, bounds):
        """One pass of the level loop over the signal ranges [a, b), in chunks of _chunk_size signals, with cap_scale times the
        default event buffers.  Finished chunks go to `out` (see _forward_batch); returns the ranges of the chunks in which a
        level wrote more events than its buffers hold (LoCOMP emits one event per refitted group atom): the later levels saw
        a truncated code, so their forward phase must be repeated with larger buffers."""
        T = x.shape[1]
        n = self._chunk_size(T, specs, cap_scale)
        rerun = []
        for lo, hi in ranges:
            for a in range(lo, hi, n):
                b = min(hi, a + n)
                levels = self._forward_chunk(x[a:b], specs, cap_scale, bounds)
                if levels is None:
                    rerun.append((a, b))
                elif bounds is not None:
                    out[a] = levels
                else:
                    for (K, off, p, i, c) in levels:
                        for s in range(b - a):
                            out[a + s].append(events_to_csc(p[off[s]:off[s + 1]], i[off[s]:off[s + 1]], c[off[s]:off[s + 1]], T, K))
        return rerun

    def _forward_chunk(self, x, specs, cap_scale, bounds=None):
        """All levels of S <= 65535 signals x [S,T,F] (numpy, or a torch tensor, used in place when it is a contiguous device
        tensor of the first level's engine dtype).  Right after a level's run, on the same stream, its events are compacted
        into buffers this call owns and its states copied to pinned memory, so that a later level cannot overwrite them even
        when two levels share one cached engine.  One synchronisation after the last level; then one read per level of the
        offsets and the flat event arrays.  Returns (K, offsets, pos, idx, coef) host arrays per level.
        With `bounds` (the device path) only the last level's events are compacted; they are canonicalized on the device,
        split into levels by `bounds`, and nothing but the states and the per-level entry counts is read back.  Returns
        (per-level dicts of device tensors from Engine.canonicalize_codes, host array of their entry counts).
        Returns None when a level's event buffers filled up before its stop rule fired."""
        import torch
        S, T = x.shape[0], x.shape[1]
        xd = None
        pending = []
        for li, (D, weights, dt, opt, K, level) in enumerate(specs):
            eng = engine_for_dictionary(D, weights, dt, self.device)
            last = li + 1 == len(specs)
            if xd is None:
                if isinstance(x, np.ndarray):
                    xd = torch.from_numpy(np.ascontiguousarray(x, dtype=dt)).to(eng.device)
                else:
                    xd = x.to(device=eng.device, dtype=eng.torch_dtype).contiguous()
            assert xd.shape[2] == eng.F, 'level %d: the dictionary has %d channels, its input %d' % (level, eng.F, xd.shape[2])
            cap = eng.default_capacity(opt, T) * cap_scale
            evp, evi, evc, _, _ = eng.encode_device(xd, opt, cap, sync_states=False)
            flat = eng.compact_events(evp, evi, evc) if bounds is None or last else None
            hstate, states = eng._pinned_states(S)
            eng._states_async(states)
            pending.append((K, flat, hstate))
            if not last:
                xd = eng.events_to_dense(evp, evi, evc, 1e-16)
            elif bounds is not None:
                canon = eng.canonicalize_codes(flat['offsets'], flat['pos'], flat['idx'], flat['coef'], S, T, K, bounds, 1e-16)
                counts = torch.empty((len(canon),), dtype=torch.int64, pin_memory=True)
                counts.copy_(torch.stack([lv['offsets'][S] for lv in canon]), non_blocking=True)
        torch.cuda.current_stream(xd.device).synchronize()
        levels = []
        for (K, flat, hstate) in pending:
            _, status, unfinished = read_states(hstate, S)
            check_refit_groups(status)
            if unfinished:
                return None
            if bounds is not None:
                continue
            off = flat['offsets'].cpu().numpy()
            n = int(off[S])
            levels.append((K, off, flat['pos'][:n].cpu().numpy(), flat['idx'][:n].cpu().numpy(),
                           flat['coef'][:n].cpu().numpy()))
        if bounds is not None:
            return canon, counts.numpy().copy()
        return levels

    def convertToDistributedCoefficients(self, coefficients):
        """:1556-1594.  The singleton (pass-through) columns [0, K_l) of the LAST level's code are the events of level l: they
        are cut out level by level, so that the total number of nonzeros is conserved (:1592).  Done on the (row, column,
        value) triples of the last level's code - a few hundred entries - instead of slicing / stacking sparse matrices."""
        last = scipy.sparse.coo_matrix(coefficients[-1])
        row, col, val = last.row, last.col, last.data
        keep = val != 0.0
        row, col, val = row[keep], col[keep], val[keep]
        T = last.shape[0]
        taken = np.zeros(len(val), dtype=bool)
        out = []
        for level in range(len(coefficients)):
            if level < len(coefficients) - 1:
                nf = coefficients[level].shape[1]
                m = (col < nf) & ~taken
                taken |= m
                lvl = scipy.sparse.csc_matrix((val[m], (row[m], col[m])), shape=(T, nf), dtype=last.dtype)
            else:
                m = ~taken
                lvl = scipy.sparse.csc_matrix((val[m], (row[m], col[m])), shape=last.shape, dtype=last.dtype)
            out.append(lvl)
        assert len(out) == len(coefficients)
        assert np.sum([c.nnz for c in out]) == len(val)
        return out

    def _calculateResidual(self, sequence, coefficients, multilevelDict):
        """:1596-1611 for one sequence: the B = 1 call of _calculateResidualBatch."""
        T = coefficients[0].shape[0]
        return self._calculateResidualBatch(np.asarray(sequence).reshape(1, T, -1), [coefficients], multilevelDict)[0]

    def _calculateResidualBatch(self, sequences, codes, multilevelDict):
        """:1596-1611 for B sequences [B,T,F] and their codes (one list of per-level csc per sequence): sequence - sum over
        the levels of decode(code_l, input-level representations of level l).  Per level, the codes of all sequences go
        into one decoder launch (each level's representations live in their own engine) that accumulates into ONE float64
        device buffer [B,T,F]; the input is subtracted on the device and read back once.  Float64 [B,T] if the base
        dictionary is 2-D, else [B,T,F]."""
        import torch
        baseDict = multilevelDict.getBaseDictionary()
        B = len(codes)
        T = codes[0][0].shape[0]
        representations = multilevelDict.getMultiscaleDictionaries()
        recon = None
        for level in range(multilevelDict.getNbLevels()):
            eng = engine_for_dictionary(representations[level], None, np.float64, self.device)
            if recon is None:
                recon = torch.zeros((B, T, eng.F), dtype=torch.float64, device=eng.device)
            _decode_codes(eng, [c[level] for c in codes], T, recon)
        xd = torch.from_numpy(np.ascontiguousarray(np.asarray(sequences).reshape(B, T, -1), dtype=np.float64)).to(recon.device)
        residual = (xd - recon).cpu().numpy()
        return residual[:, :, 0] if baseDict.ndim == 2 else residual

    def _postprocessCoefficients(self, coefficients, multilevelDict, returnDistributed=True):
        if returnDistributed:
            return self.convertToDistributedCoefficients(coefficients)
        out = []
        for level in range(multilevelDict.getNbLevels()):
            c = coefficients[level]
            if level < multilevelDict.getNbLevels() - 1:
                c = scipy.sparse.csc_matrix(c.shape, dtype=c.dtype)
            out.append(c)
        return out

    def computeCoefficients(self, sequence, multilevelDict, nbNonzeroCoefs=None, toleranceResidualScale=None,
                            toleranceSnr=None, nbBlocks=1, minCoefficients=None, singletonWeight=0.5,
                            returnDistributed=True, stopCondition=None):
        assert _is_multilevel_dictionary(multilevelDict)
        coefficients = self._forward(np.asarray(sequence), [], multilevelDict, toleranceSnr, nbBlocks, singletonWeight)
        coefficients = self._postprocessCoefficients(coefficients, multilevelDict, returnDistributed)
        residual = self._calculateResidual(np.asarray(sequence), coefficients, multilevelDict)
        return coefficients, residual

    def computeCoefficientsBatch(self, sequences, multilevelDict, nbNonzeroCoefs=None, toleranceResidualScale=None,
                                 toleranceSnr=None, nbBlocks=1, minCoefficients=None, singletonWeight=0.5, returnDistributed=True):
        """computeCoefficients for B independent sequences [B,T] or [B,T,F] of one length: returns a list of B per-level lists
        of float64 csc matrices and the float64 residual [B,T] or [B,T,F] (the shape rule of computeCoefficients).  Every
        argument means what it means there (nbNonzeroCoefs, toleranceResidualScale and minCoefficients are ignored there
        too).  Each sequence gets bit for bit the codes and residual of its own computeCoefficients call: the levels run on
        all sequences of a chunk at once, the pursuit one CTA per sequence."""
        assert _is_multilevel_dictionary(multilevelDict)
        sequences = np.asarray(sequences)
        assert sequences.ndim == 2 or sequences.ndim == 3
        x = sequences[:, :, None] if sequences.ndim == 2 else sequences
        codes = self._forward_batch(x, [], multilevelDict, toleranceSnr, nbBlocks, singletonWeight)
        codes = [self._postprocessCoefficients(c, multilevelDict, returnDistributed) for c in codes]
        if len(codes) == 0:
            F = np.asarray(multilevelDict.getBaseDictionary()).shape[2:]
            return codes, np.zeros((0, x.shape[1]) + F, dtype=np.float64)
        residual = self._calculateResidualBatch(x, codes, multilevelDict)
        return codes, residual

    def computeCoefficientsBatchDevice(self, sequences, multilevelDict, toleranceSnr=None, nbBlocks=1, singletonWeight=0.5,
                                       returnDistributed=True):
        """computeCoefficientsBatch with the codes and the residual left on the GPU: sequences [B,T] or [B,T,F], a numpy
        array or a torch tensor (a contiguous CUDA tensor on the coder's device, of the first level's engine dtype, is read
        in place); the dtype rules are those of computeCoefficientsBatch.  Returns (HierarchicalCodes, residual), the
        residual a float64 CUDA tensor [B,T] or [B,T,F] (the shape rule of computeCoefficientsBatch).
        The level loop is the one of computeCoefficientsBatch; only the last level's events are kept, and per chunk they are
        summed, ordered and redistributed on the device (Engine.canonicalize_codes).  Duplicate events are summed in
        selection order, which the host path does not guarantee for three or more events of one (t, k), so a value may
        differ from computeCoefficientsBatch's in the last bits; the sparsity pattern is the same."""
        import torch
        assert _is_multilevel_dictionary(multilevelDict)
        if not isinstance(sequences, torch.Tensor):
            sequences = np.asarray(sequences)
        assert sequences.ndim == 2 or sequences.ndim == 3
        x = sequences[:, :, None] if sequences.ndim == 2 else sequences
        B, T = x.shape[0], x.shape[1]
        nl = multilevelDict.getNbLevels()
        K = [np.asarray(multilevelDict.getRawDictionary(l)).shape[0] for l in range(nl)]
        device = engine_for_dictionary(multilevelDict.getMultiscaleDictionaries()[0], None, np.float64, self.device).device
        if isinstance(x, np.ndarray):            # one upload, read by the first level and by the residual
            x = torch.from_numpy(np.ascontiguousarray(x)).to(device)
        # redistribution (:1556-1594): columns [0, K_l) of the last level's code are level l's events; bounds of 0 leave
        # the lower levels empty
        done = self._forward_batch(x, [], multilevelDict, toleranceSnr, nbBlocks, singletonWeight,
                                   K[:-1] if returnDistributed else [0] * (nl - 1))
        chunks = [done[a] for a in sorted(done)]
        levels = [_concat_codes([(canon[l], counts[l]) for canon, counts in chunks], device) for l in range(nl)]
        codes = HierarchicalCodes(B, T, K, *zip(*levels))
        recon = self.reconstructBatchDevice(codes, multilevelDict)
        return codes, x.to(device=device, dtype=torch.float64).reshape(recon.shape) - recon

    def reconstructBatchDevice(self, codes, multilevelDict):
        """The input-level reconstruction of HierarchicalCodes (:1596-1611 without the subtraction), on the device: per level,
        one decoder launch over all sequences with that level's representations (float64 engine), accumulating into one
        float64 buffer [B,T,F] in level order.  Returns a float64 CUDA tensor [B,T] if the base dictionary is 2-D, else
        [B,T,F]."""
        import torch
        representations = multilevelDict.getMultiscaleDictionaries()
        assert len(codes.K) == multilevelDict.getNbLevels()
        recon = None
        for level in range(multilevelDict.getNbLevels()):
            eng = engine_for_dictionary(representations[level], None, np.float64, self.device)
            if recon is None:
                recon = torch.zeros((codes.B, codes.T, eng.F), dtype=torch.float64, device=eng.device)
            _decode_codes_device(eng, codes.offsets[level], codes.pos[level], codes.idx[level], codes.coef[level], codes.B, codes.T,
                                 recon)
        return recon[:, :, 0] if np.asarray(multilevelDict.getBaseDictionary()).ndim == 2 else recon

    def computeCoefficientsFromLevel(self, sequence, coefficients, multilevelDict, nbNonzeroCoefs=None,
                                     toleranceResidualScale=None, toleranceSnr=None, nbBlocks=1, minCoefficients=None,
                                     singletonWeight=0.5, stopCondition=None, returnDistributed=True):
        assert _is_multilevel_dictionary(multilevelDict)
        coefficients = copy.deepcopy(coefficients)
        coefficients = self._forward(np.asarray(sequence), coefficients, multilevelDict, toleranceSnr, nbBlocks, singletonWeight)
        return self._postprocessCoefficients(coefficients, multilevelDict, returnDistributed)


class ConvolutionalSparseCoder(object):
    """hsc/modeling.py:1656-1669."""

    def __init__(self, D, approximator):
        assert D.ndim == 2 or D.ndim == 3
        self.D = D
        self.approximator = approximator

    def encode(self, X, *args, **kwargs):
        assert X.ndim == 1 or X.ndim == 2
        return self.approximator.computeCoefficients(X, self.D, *args, **kwargs)

    def encodeBatch(self, X, *args, **kwargs):
        assert X.ndim == 2 or X.ndim == 3
        return self.approximator.computeCoefficientsBatch(X, self.D, *args, **kwargs)

    def encodeBatchDevice(self, X, *args, **kwargs):
        """encodeBatch with the codes and the residual left on the GPU, for batches of any size: (SparseCodes, CUDA residual
        of the engine dtype, or None with returnResidual=False); X [B,T] or [B,T,F], numpy or torch (see
        ConvolutionalMatchingPursuit.computeCoefficientsBatchDevice)."""
        assert X.ndim == 2 or X.ndim == 3
        return self.approximator.computeCoefficientsBatchDevice(X, self.D, *args, **kwargs)

    def reconstructBatchDevice(self, codes):
        """The float64 reconstruction of SparseCodes on the device: [B,T] (2-D dictionary) or [B,T,F]; equal to
        reconstructBatch(codes.to_csc())."""
        return self.approximator.reconstructBatchDevice(codes, self.D)

    def reconstruct(self, coefficients):
        assert coefficients.ndim == 1 or coefficients.ndim == 2
        return reconstructSignal(coefficients, self.D, device=getattr(self.approximator, 'device', None))

    def reconstructBatch(self, codes):
        """reconstruct for B codes of one shape [T,K] in one decoder launch: [B,T] (2-D dictionary) or [B,T,F], each row
        bit for bit reconstruct(codes[b]), in the dtype reconstruct gives (the codes' float dtype, else float64)."""
        assert len(codes) > 0 and all(c.ndim == 2 and c.shape == codes[0].shape for c in codes)
        return _reconstruct_batch(codes, self.D, getattr(self.approximator, 'device', None))


class HierarchicalConvolutionalSparseCoder(object):
    """hsc/modeling.py:1671-1705."""

    def __init__(self, multilevelDict, approximator):
        assert _is_multilevel_dictionary(multilevelDict)
        if not multilevelDict.hasSingletonBases:
            multilevelDict = multilevelDict.withSingletonBases()
        self.multilevelDict = multilevelDict
        self.approximator = approximator

    def encode(self, sequence, *args, **kwargs):
        assert sequence.ndim == 1 or sequence.ndim == 2
        return self.approximator.computeCoefficients(sequence, self.multilevelDict, *args, **kwargs)

    def encodeBatch(self, X, *args, **kwargs):
        assert X.ndim == 2 or X.ndim == 3
        return self.approximator.computeCoefficientsBatch(X, self.multilevelDict, *args, **kwargs)

    def encodeBatchDevice(self, X, **kwargs):
        """encodeBatch with the codes and the residual left on the GPU: (HierarchicalCodes, float64 CUDA residual); X [B,T]
        or [B,T,F], numpy or torch (see HierarchicalConvolutionalMatchingPursuit.computeCoefficientsBatchDevice)."""
        assert X.ndim == 2 or X.ndim == 3
        return self.approximator.computeCoefficientsBatchDevice(X, self.multilevelDict, **kwargs)

    def reconstructBatchDevice(self, codes):
        """The float64 reconstruction of HierarchicalCodes on the device: [B,T] (2-D base dictionary) or [B,T,F]; equal to
        reconstructBatch(codes.to_csc())."""
        return self.approximator.reconstructBatchDevice(codes, self.multilevelDict)

    def encodeFromLevel(self, sequence, coefficients, *args, **kwargs):
        assert len(coefficients) > 0
        return self.approximator.computeCoefficientsFromLevel(sequence, coefficients, self.multilevelDict, *args, **kwargs)

    def reconstruct(self, coefficients):
        assert len(coefficients) > 0
        baseDict = self.multilevelDict.getBaseDictionary()
        shape = (coefficients[0].shape[0],) if baseDict.ndim == 2 else (coefficients[0].shape[0], baseDict.shape[-1])
        signal = np.zeros(shape, dtype=coefficients[0].dtype)
        representations = self.multilevelDict.getMultiscaleDictionaries()
        for level in range(self.multilevelDict.getNbLevels()):
            signal += reconstructSignal(coefficients[level], representations[level],
                                        device=getattr(self.approximator, 'device', None))
        return signal

    def reconstructBatch(self, codes):
        """reconstruct for B sequences' per-level codes (as encodeBatch returns them): one decoder launch per level, the
        levels summed on the host in level order like reconstruct, so each row is bit for bit reconstruct(codes[b])."""
        assert len(codes) > 0 and all(len(c) == self.multilevelDict.getNbLevels() for c in codes)
        representations = self.multilevelDict.getMultiscaleDictionaries()
        signal = None
        for level in range(self.multilevelDict.getNbLevels()):
            lvl = _reconstruct_batch([c[level] for c in codes], representations[level], getattr(self.approximator, 'device', None))
            if signal is None:
                signal = np.zeros(lvl.shape, dtype=codes[0][0].dtype)
            signal += lvl
        return signal
