"""Python host side of the engine: owns a native `hsc_engine` handle and uses PyTorch only for
device memory, pinned host buffers and streams.  Every number is produced by the CUDA kernels
behind the C ABI (include/hsc_b200.h); there is no CPU path in this module.
"""
import ctypes
import math

import numpy as np

from . import _native as N


def _torch():
    import torch
    return torch


def _np_dtype(code):
    return np.float32 if code == N.HSC_F32 else np.float64


def engine_dtype(*arrays):
    """Arithmetic type of the path: the NumPy result type of (signal, dictionary), as np.dot gives the
    reference (hsc/modeling.py:186-187): float32 only if everything is float32."""
    rt = np.result_type(*[np.asarray(a).dtype for a in arrays])
    return np.float32 if rt == np.float32 else np.float64


def state_stats(st):
    """The final state of one signal (N.SignalState) as the dict EncodeResult.stats returns."""
    return dict(energy_signal=st.energy_signal, energy_residual=st.energy_residual, n_events=st.n_events, nnz=st.nnz,
                duplicates=st.duplicates, passes=st.passes, reranked=st.reranked,
                stop=N.STOP_NAMES.get(st.status, str(st.status)))


_STATE_DTYPE = np.dtype(N.SignalState)


def read_states(states, n):
    """The first n per-signal states of a ctypes SignalState array, or of the pinned uint8 tensor an asynchronous states
    copy fills: returns (a private copy as a SignalState array, its status column int32 [n], whether any signal is paused
    or still running - its encode has to be run again)."""
    raw = states.numpy() if hasattr(states, 'numpy') else bytes(states)
    snap = (N.SignalState * n).from_buffer_copy(raw[:n * _STATE_DTYPE.itemsize])
    status = np.frombuffer(snap, _STATE_DTYPE)['status']
    return snap, status, bool((status[:, None] == (N.HSC_PAUSE_CAPACITY, N.HSC_PAUSE_PASSES, N.HSC_RUNNING)).any())


def check_refit_groups(status):
    """Raises when a signal stopped because a LoCOMP selection had more common-support atoms than the device refit holds:
    such an encode has no result to return."""
    if np.any(np.asarray(status) == N.HSC_STOP_GROUP):
        raise NotImplementedError('LoCOMP: a selection has more than 255 common-support atoms; the device refit holds groups '
                                  'of at most 256')


def escalate_capacity(run_pass, ranges, what):
    """Runs run_pass(ranges, scale) with scale 1, 8, 64, ... 4096 (times the default event buffers) until it returns no
    signal range to run again; signals are independent, so a range that filled its buffers is rerun on its own."""
    scale = 1
    while ranges:
        if scale > 4096:
            raise N.HscError(N.HSC_E_NOMEM, '%s: event buffers exhausted' % what)
        ranges = run_pass(ranges, scale)
        scale *= 8


def _concat_codes(parts, device):
    """(offsets int64 [B+1], pos, idx int32, coef float64) device tensors of the canonical codes `parts`, pairs (one level's
    dict from Engine.canonicalize_codes, its entry count) in signal order: each trimmed to its count, the offsets rebased."""
    torch = _torch()
    offsets, pos, idx, coef = [torch.zeros((1,), dtype=torch.int64, device=device)], [], [], []
    base = 0
    for lv, n in parts:
        n = int(n)
        offsets.append(lv['offsets'][1:] + base)
        pos.append(lv['pos'][:n])
        idx.append(lv['idx'][:n])
        coef.append(lv['coef'][:n])
        base += n
    cat = lambda a, dt: torch.cat(a) if a else torch.zeros((0,), dtype=dt, device=device)
    return torch.cat(offsets), cat(pos, torch.int32), cat(idx, torch.int32), cat(coef, torch.float64)


def events_to_csc(pos, idx, coef, T, K, min_coefficients=1e-16):
    """One signal's events (selection order, duplicates allowed) -> the reference's return type: csc_matrix [T,K] float64,
    duplicates summed (`+=`, hsc/modeling.py:992), |c| < min_coefficients dropped (:1171-1177; None: none), zeros
    eliminated (:1180-1181)."""
    import scipy.sparse
    m = scipy.sparse.coo_matrix((coef.astype(np.float64), (pos.astype(np.int64), idx.astype(np.int64))), shape=(T, K)).tocsc()
    m.sum_duplicates()
    if min_coefficients is not None:
        m.data[np.abs(m.data) < min_coefficients] = 0.0
    m.eliminate_zeros()
    return m


class EncodeResult(object):
    """Events of S signals in selection order, plus the final states and (optionally) residuals."""

    def __init__(self, S, T, K):
        self.S, self.T, self.K = S, T, K
        self.pos = [np.zeros(0, np.int32) for _ in range(S)]
        self.idx = [np.zeros(0, np.int32) for _ in range(S)]
        self.coef = [None] * S
        self.states = None
        self.residual = None
        self.counts = None          # events per signal (host pipeline; also set when the event lists stay on the device)
        self.gathered = None        # what the on_device_events hook of the host pipeline returned (multi-GPU gather)
        self.batch_index = None

    def stats(self, s=0):
        return state_stats(self.states[s])

    def total_events(self):
        if self.counts is not None:
            return int(np.sum(self.counts))
        return int(sum(len(p) for p in self.pos))

    def to_csc(self, s=0, min_coefficients=1e-16):
        """The events of signal s as the reference's csc_matrix [T,K] float64 (events_to_csc)."""
        return events_to_csc(self.pos[s], self.idx[s], self.coef[s], self.T, self.K, min_coefficients)


def _with_stream(fn):
    """A `stream=` argument becomes torch's CURRENT stream for the duration of the call, so that the tensor allocations, the
    non-blocking host-to-device copies and the torch.distributed collectives inside are ordered with the native launches
    (which go to the same stream through _stream_ptr) instead of racing them from the default stream."""
    import functools

    @functools.wraps(fn)
    def wrapper(self, *args, **kw):
        stream = kw.get('stream')
        if stream is None:
            return fn(self, *args, **kw)
        with _torch().cuda.stream(stream):
            return fn(self, *args, **kw)
    return wrapper


class Engine(object):
    """One native engine on one CUDA device."""

    def __init__(self, device=None):
        torch = _torch()
        if not torch.cuda.is_available():
            raise RuntimeError('hierarchical_sparse_coding_b200 needs a CUDA device (no CPU fallback)')
        self.lib = N.load_library()
        if device is None:
            device = torch.cuda.current_device()
        self.device = torch.device('cuda', int(device) if not isinstance(device, torch.device) else device.index or 0)
        h = ctypes.c_void_p()
        N.check(self.lib, None, self.lib.hsc_b200_create(self.device.index, ctypes.byref(h)))
        self.handle = h
        self.dtype = None
        self.K = self.L = self.F = None
        self._D_host = None
        self._w_host = None

    def close(self):
        self._pipe_cache = self._host_cache = self._ws_cache = self._last_workspace = None    # device + pinned staging buffers
        self._stream_stage = None
        for h in getattr(self, '_views', []):
            self.lib.hsc_b200_destroy(h)
        self._views = []
        if getattr(self, 'handle', None):
            self.lib.hsc_b200_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launches(self):
        return int(self.lib.hsc_b200_launch_count(self.handle))

    # ------------------------------------------------------------------ dictionary
    def set_dictionary(self, D, weights=None, dtype=None):
        D = np.asarray(D)
        assert D.ndim == 2 or D.ndim == 3
        if D.ndim == 2:
            D = D[:, :, None]
        dt = np.dtype(dtype) if dtype is not None else np.dtype(engine_dtype(D))
        assert dt in (np.dtype(np.float32), np.dtype(np.float64))
        Dh = np.ascontiguousarray(D, dtype=dt)
        wh = None
        if weights is not None:
            wh = np.ascontiguousarray(np.asarray(weights), dtype=dt)
            assert wh.shape == (Dh.shape[0],)
        # the same dictionary again (every encode of a coder re-sends it): keep the uploaded D, Gram tensor and K1 operand
        if (self._D_host is not None and self.dtype == dt and self._D_host.shape == Dh.shape and np.array_equal(self._D_host, Dh)
                and ((wh is None and self._w_host is None) or
                     (wh is not None and self._w_host is not None and np.array_equal(self._w_host, wh)))):
            return self
        code = N.HSC_F32 if dt == np.dtype(np.float32) else N.HSC_F64
        with _torch().cuda.device(self.device):
            N.check(self.lib, self.handle, self.lib.hsc_b200_set_dictionary(
                self.handle, Dh.ctypes.data_as(ctypes.c_void_p), code, Dh.shape[0], Dh.shape[1], Dh.shape[2],
                wh.ctypes.data_as(ctypes.c_void_p) if wh is not None else None))
        self.dtype = dt
        self.K, self.L, self.F = Dh.shape
        self._dict_version = getattr(self, '_dict_version', 0) + 1
        self._D_host, self._w_host = Dh.copy(), (None if wh is None else wh.copy())
        return self

    @property
    def torch_dtype(self):
        torch = _torch()
        return torch.float32 if self.dtype == np.dtype(np.float32) else torch.float64

    def _to_host(self, ptr, shape):
        out = np.empty(shape, dtype=self.dtype)
        N.check(self.lib, self.handle, self.lib.hsc_b200_copy_to_host(
            self.handle, ctypes.c_void_p(ptr), out.ctypes.data_as(ctypes.c_void_p), out.nbytes))
        return out

    def gram(self):
        """Copy of the device Gram tensor G[K][2L-1][K] (tests)."""
        return self._to_host(self.lib.hsc_b200_gram_dev(self.handle), (self.K, 2 * self.L - 1, self.K))

    # ------------------------------------------------------------------ helpers
    def _stream_ptr(self, stream=None):
        torch = _torch()
        s = stream if stream is not None else torch.cuda.current_stream(self.device)
        return ctypes.c_void_p(s.cuda_stream)

    def _as_device_batch(self, x, stream=None):
        """x: numpy [S,T,F] / torch tensor (host or device) -> contiguous device tensor of the engine dtype."""
        torch = _torch()
        if isinstance(x, np.ndarray):
            x = torch.from_numpy(np.ascontiguousarray(x, dtype=self.dtype))
        x = x.to(device=self.device, dtype=self.torch_dtype, non_blocking=True).contiguous()
        assert x.dim() == 3 and x.shape[2] == self.F, 'signals must be [S,T,F=%d]' % self.F
        return x

    def make_options(self, nbNonzeroCoefs=None, toleranceResidualScale=None, toleranceSnr=None, nbBlocks=1,
                     minCoefficients=1e-16, use_weights=False, coef_mode=1, max_passes_per_run=0, max_events_total=0,
                     method=0, rerank_tolerance=-1.0, energy_eps=None):
        o = N.MpOptions()
        o.nb_nonzero_coefs = -1 if nbNonzeroCoefs is None else int(nbNonzeroCoefs)
        o.tolerance_snr = float('nan') if toleranceSnr is None else float(toleranceSnr)
        o.tolerance_residual_scale = float('nan') if toleranceResidualScale is None else float(toleranceResidualScale)
        o.min_coefficients = -1.0 if minCoefficients is None else float(minCoefficients)
        o.nb_blocks = -1 if nbBlocks == 'auto' else int(nbBlocks)
        o.use_weights = 1 if use_weights else 0
        o.coef_mode = int(coef_mode)
        o.max_passes_per_run = int(max_passes_per_run)
        o.max_events_total = int(max_events_total)
        o.method = int(method)
        o.rerank_tolerance = float(rerank_tolerance)       # < 0: the engine's default near-tie window (include/hsc_b200.h)
        o.energy_eps = 0.0 if energy_eps is None else float(energy_eps)     # np.finfo(D.dtype).eps of the caller's dictionary (:1057)
        return o

    # ------------------------------------------------------------------ correlation (K1)
    @_with_stream
    def correlate(self, x, stream=None):
        """convolve1d(x, D, 'same') for a batch: returns the device map [S,T,K]."""
        torch = _torch()
        with torch.cuda.device(self.device):
            xd = self._as_device_batch(x)
            S, T, _ = xd.shape
            out = torch.empty((S, T, self.K), dtype=self.torch_dtype, device=self.device)
            N.check(self.lib, self.handle, self.lib.hsc_b200_correlate(
                self.handle, ctypes.c_void_p(xd.data_ptr()), S, T, ctypes.c_void_p(out.data_ptr()), self._stream_ptr(stream)))
        return out

    # ------------------------------------------------------------------ pursuit (K1 + K2)
    def workspace_bytes(self, S, T):
        return int(self.lib.hsc_b200_workspace_bytes(self.handle, S, T))

    def _free_device_bytes(self):
        torch = _torch()
        free, _ = torch.cuda.mem_get_info(self.device)
        # blocks torch's caching allocator holds but has not handed out are reusable too
        return free + torch.cuda.memory_reserved(self.device) - torch.cuda.memory_allocated(self.device)

    def _event_buffers(self, S, cap):
        """The [S,cap] event buffers mp_run fills: positions, filter indices (int32) and coefficients (engine dtype)."""
        torch = _torch()
        return (torch.empty((S, cap), dtype=torch.int32, device=self.device),
                torch.empty((S, cap), dtype=torch.int32, device=self.device),
                torch.empty((S, cap), dtype=self.torch_dtype, device=self.device))

    def _compact_buffers(self, S, cap):
        """compact_events' output for S signals of `cap` events each: offsets int64 [S+1], flat pos, idx, coef."""
        torch = _torch()
        return dict(offsets=torch.empty((S + 1,), dtype=torch.int64, device=self.device),
                    pos=torch.empty((S * cap,), dtype=torch.int32, device=self.device),
                    idx=torch.empty((S * cap,), dtype=torch.int32, device=self.device),
                    coef=torch.empty((S * cap,), dtype=self.torch_dtype, device=self.device))

    def _pinned_states(self, S):
        """A pinned buffer for S per-signal states and its ctypes view (the target of _states_async)."""
        torch = _torch()
        hstate = torch.empty((S * _STATE_DTYPE.itemsize,), dtype=torch.uint8, pin_memory=True)
        return hstate, (N.SignalState * S).from_address(hstate.data_ptr())

    def _states_async(self, states, stream=None, handle=None):
        """Enqueues the copy of the states of the encode in flight on `handle` (default: this engine's) into `states`."""
        h = self.handle if handle is None else handle
        N.check(self.lib, h, self.lib.hsc_b200_mp_states_async(h, states, self._stream_ptr(stream)))

    def _workspace(self, S, T):
        """The workspace of an encode of S signals of length T: kept on the engine and grown when too small."""
        torch = _torch()
        wsb = self.workspace_bytes(S, T)
        ws = getattr(self, '_ws_cache', None)
        if ws is None or ws.numel() < wsb:
            self._ws_cache = None
            ws = self._ws_cache = torch.empty((wsb,), dtype=torch.uint8, device=self.device)
        return ws, wsb

    def max_signals_per_chunk(self, T, budget_bytes=None, extra_per_signal=0):
        if budget_bytes is None:
            budget_bytes = int(self._free_device_bytes() * 0.8)
        per = self.workspace_bytes(1, T) + 2 * T * self.F * self.dtype.itemsize + int(extra_per_signal)
        return max(1, int(budget_bytes // per))

    def default_capacity(self, options, T):
        if options.method == 1:       # LoCOMP emits one event per refitted group atom (<= 64 per selection)
            base = int(options.nb_nonzero_coefs * 4) if options.nb_nonzero_coefs >= 0 else int(max(1024, T // 8))
            return int(min(max(2048, base + 1024), 1 << 20))
        if options.max_events_total > 0:
            return int(options.max_events_total)
        if options.nb_nonzero_coefs >= 0:
            return int(options.nb_nonzero_coefs * 1.5) + 64
        return int(min(max(1024, T // 8), 1 << 20))

    @_with_stream
    def encode(self, x, options, capacity=None, return_residual=True, residual_inplace=False, stream=None,
               on_pass=None):
        """Matching pursuit of S independent signals.

        x: [S,T,F] numpy array, host tensor (ideally pinned) or device tensor.
        Returns EncodeResult with numpy event lists; `residual` is a device tensor [S,T,F] when
        return_residual (D2H is the caller's choice: .cpu()).
        on_pass(result_so_far, states) -> bool, if given, is called between launches
        (options.max_passes_per_run should be 1 then); returning True stops the encode."""
        torch = _torch()
        with torch.cuda.device(self.device):
            xd = self._as_device_batch(x)
            S, T, _ = xd.shape
            res = EncodeResult(S, T, self.K)
            if S == 0:
                return res
            cap = int(capacity) if capacity is not None else self.default_capacity(options, T)
            wsb = self.workspace_bytes(S, T)
            ws = torch.empty((wsb,), dtype=torch.uint8, device=self.device)
            resid = xd if residual_inplace else torch.empty_like(xd)
            evp, evi, evc = self._event_buffers(S, cap)
            sp = self._stream_ptr(stream)
            N.check(self.lib, self.handle, self.lib.hsc_b200_mp_begin(
                self.handle, ctypes.c_void_p(xd.data_ptr()), ctypes.c_void_p(resid.data_ptr()), S, T,
                ctypes.c_void_p(ws.data_ptr()), wsb, ctypes.byref(options), sp))
            states = (N.SignalState * S)()
            chunks_p = [[] for _ in range(S)]
            chunks_i = [[] for _ in range(S)]
            chunks_c = [[] for _ in range(S)]
            while True:
                N.check(self.lib, self.handle, self.lib.hsc_b200_mp_run(
                    self.handle, ctypes.c_void_p(evp.data_ptr()), ctypes.c_void_p(evi.data_ptr()),
                    ctypes.c_void_p(evc.data_ptr()), cap, states, sp))
                nb = np.array([states[s].n_buffered for s in range(S)], dtype=np.int64)
                m = int(nb.max())
                if m > 0:
                    hp = evp[:, :m].cpu().numpy()
                    hi = evi[:, :m].cpu().numpy()
                    hc = evc[:, :m].cpu().numpy()
                    for s in range(S):
                        if nb[s] > 0:
                            chunks_p[s].append(hp[s, :nb[s]].copy())
                            chunks_i[s].append(hi[s, :nb[s]].copy())
                            chunks_c[s].append(hc[s, :nb[s]].copy())
                if not read_states(states, S)[2]:
                    break
                if on_pass is not None:
                    self._fill(res, chunks_p, chunks_i, chunks_c, states)
                    res.residual = resid
                    if on_pass(res, states):
                        break
            self._fill(res, chunks_p, chunks_i, chunks_c, states)
            res.residual = resid if return_residual else None
            self._last_workspace = ws   # keeps the map alive for map_snapshot()
            self._last_shape = (S, T)
        return res

    @_with_stream
    def encode_device(self, xd, options, capacity, resid=None, stream=None, sync_states=True):
        """Lean path for resident data: xd is a device tensor [S,T,F] of the engine dtype; runs K1 + one
        K2 launch and returns (ev_pos, ev_idx, ev_coef, states, residual) with the events still on the
        device ([S,capacity] each).  `states` is None when sync_states is False (fully asynchronous)."""
        if resid is None:
            resid = _torch().empty_like(xd)
        self.begin_only(xd, options, resid, stream=stream)
        evp, evi, evc = self._event_buffers(xd.shape[0], capacity)
        states = self.run_only(evp, evi, evc, capacity, sync_states, stream=stream)
        return evp, evi, evc, states, resid

    @_with_stream
    def begin_only(self, xd, options, resid, stream=None):
        """K1 + state reset only (bench: times the correlation separately from the pursuit)."""
        torch = _torch()
        S, T, _ = xd.shape
        with torch.cuda.device(self.device):
            ws, wsb = self._workspace(S, T)
            N.check(self.lib, self.handle, self.lib.hsc_b200_mp_begin(
                self.handle, ctypes.c_void_p(xd.data_ptr()), ctypes.c_void_p(resid.data_ptr()), S, T,
                ctypes.c_void_p(ws.data_ptr()), wsb, ctypes.byref(options), self._stream_ptr(stream)))
            self._last_workspace = ws
            self._last_shape = (S, T)

    @_with_stream
    def run_only(self, evp, evi, evc, capacity, sync_states=True, stream=None):
        S = self._last_shape[0]
        states = (N.SignalState * S)() if sync_states else None
        with _torch().cuda.device(self.device):
            N.check(self.lib, self.handle, self.lib.hsc_b200_mp_run(
                self.handle, ctypes.c_void_p(evp.data_ptr()), ctypes.c_void_p(evi.data_ptr()),
                ctypes.c_void_p(evc.data_ptr()), capacity, states, self._stream_ptr(stream)))
        return states

    @_with_stream
    def events_to_dense(self, evp, evi, evc, min_coefficients=1e-16, stream=None):
        """Level hand-off of the hierarchical encoder on the device (hsc/modeling.py:1489): the accumulated code of the
        encode in flight as a dense float64 device tensor [S,T,K] - the next level's K-channel input."""
        torch = _torch()
        S, T = self._last_shape
        with torch.cuda.device(self.device):
            out = torch.empty((S, T, self.K), dtype=torch.float64, device=self.device)
            N.check(self.lib, self.handle, self.lib.hsc_b200_mp_events_to_dense(
                self.handle, ctypes.c_void_p(evp.data_ptr()), ctypes.c_void_p(evi.data_ptr()), ctypes.c_void_p(evc.data_ptr()),
                int(evp.shape[1]), -1.0 if min_coefficients is None else float(min_coefficients), ctypes.c_void_p(out.data_ptr()),
                self._stream_ptr(stream)))
        return out

    # ------------------------------------------------------------------ resident pipeline (several encodes in flight)
    def make_slots(self, n, S, T, capacity, own_residual=True):
        """n independent encode slots on this engine's dictionary (native views: own workspace, event buffers, residual,
        pinned states), so that the correlation of one batch can run - on its own stream - while the pursuit of the
        previous one is still going, and the pursuit CTAs of the next batch move into the SMs the previous batch's tail
        frees.  own_residual=False: the caller passes the residual buffer to every begin().  See EncodeSlot."""
        views = self._views_for(n)
        return [EncodeSlot(self, views[i], S, T, capacity, own_residual) for i in range(n)]

    @_with_stream
    def compact_events(self, evp, evi, evc, out=None, stream=None, handle=None):
        """Compacts the [S,capacity] event buffers of the encode in flight (after run_only / encode_device) on the device:
        returns dict(offsets=int64[S+1], pos, idx, coef flat device tensors of S*capacity entries); the atoms of signal s are
        [offsets[s], offsets[s+1]).  `out`: a dict from an earlier call to reuse its buffers (they may be larger).
        `handle`: the native handle whose encode is in flight (default: this engine's).  Asynchronous."""
        torch = _torch()
        S, cap = evp.shape
        h = self.handle if handle is None else handle
        with torch.cuda.device(self.device):
            if out is None or out['pos'].numel() < S * cap or out['offsets'].numel() < S + 1:
                out = self._compact_buffers(S, cap)
            N.check(self.lib, h, self.lib.hsc_b200_mp_compact_events(
                h, ctypes.c_void_p(evp.data_ptr()), ctypes.c_void_p(evi.data_ptr()), ctypes.c_void_p(evc.data_ptr()), cap,
                ctypes.c_void_p(out['offsets'].data_ptr()), ctypes.c_void_p(out['pos'].data_ptr()), ctypes.c_void_p(out['idx'].data_ptr()),
                ctypes.c_void_p(out['coef'].data_ptr()), S * cap, self._stream_ptr(stream)))
        return out

    # ------------------------------------------------------------------ host pipeline (public batched path)
    def _views_for(self, n):
        """n extra native handles sharing this engine's device dictionary, one per in-flight chunk."""
        ver = getattr(self, '_dict_version', 0)
        if getattr(self, '_views_version', None) != ver or len(getattr(self, '_views', [])) < n:
            for h in getattr(self, '_views', []):
                self.lib.hsc_b200_destroy(h)
            self._views = []
            for _ in range(n):
                h = ctypes.c_void_p()
                N.check(self.lib, self.handle, self.lib.hsc_b200_create_view(self.handle, ctypes.byref(h)))
                self._views.append(h)
            self._views_version = ver
            self._chunk_cache = {}
        return self._views[:n]

    def encode_host(self, x_host, options, capacity=None, n_chunks=4, residual_out=None, want_residual=True):
        """Matching pursuit of S independent signals that live in HOST memory (ideally a pinned torch tensor
        [S,T,F] of the engine dtype).  The host-to-device copy is cut into `n_chunks` chunks on a copy stream;
        the correlation (K1) of a chunk starts as soon as its copy has landed (hsc_b200_mp_begin_part), so the
        PCIe transfer hides under K1.  The select/update loop (K2) then runs once over the whole batch - it
        needs every signal resident to fill the GPU - and codes + residuals are copied back.
        Residuals land in `residual_out` (host tensor like x; allocated, pinned if x is, when None and wanted).
        Returns EncodeResult (events as numpy arrays, residual = the host tensor)."""
        torch = _torch()
        if isinstance(x_host, np.ndarray):
            x_host = torch.from_numpy(np.ascontiguousarray(x_host, dtype=self.dtype))
        assert x_host.dim() == 3 and x_host.shape[2] == self.F and x_host.dtype == self.torch_dtype
        S, T, _ = x_host.shape
        res = EncodeResult(S, T, self.K)
        if S == 0:
            return res
        cap = int(capacity) if capacity is not None else self.default_capacity(options, T)
        n_chunks = max(1, min(int(n_chunks), S))
        if want_residual and residual_out is None:
            residual_out = torch.empty_like(x_host).pin_memory() if x_host.is_pinned() else torch.empty_like(x_host)
        with torch.cuda.device(self.device):
            key = (S, T, cap, self.F, str(self.dtype))
            cache = getattr(self, '_host_cache', None)
            if cache is None or cache['key'] != key:
                self._host_cache = None
                wsb = self.workspace_bytes(S, T)
                cache = dict(key=key, wsb=wsb, copy_stream=torch.cuda.Stream(device=self.device),
                             ws=torch.empty((wsb,), dtype=torch.uint8, device=self.device),
                             xd=torch.empty((S, T, self.F), dtype=self.torch_dtype, device=self.device),
                             hp=torch.empty((S, cap), dtype=torch.int32).pin_memory(),
                             hi=torch.empty((S, cap), dtype=torch.int32).pin_memory(),
                             hc=torch.empty((S, cap), dtype=self.torch_dtype).pin_memory(),
                             states=(N.SignalState * S)())
                cache['evp'], cache['evi'], cache['evc'] = self._event_buffers(S, cap)
                self._host_cache = cache
            cur = torch.cuda.current_stream(self.device)
            cs = cache['copy_stream']
            cs.wait_stream(cur)                       # the staging buffer may still be read by earlier work
            sp = ctypes.c_void_p(cur.cuda_stream)
            xp = ctypes.c_void_p(cache['xd'].data_ptr())
            wsp = ctypes.c_void_p(cache['ws'].data_ptr())
            for c in range(n_chunks):
                lo, hi = S * c // n_chunks, S * (c + 1) // n_chunks
                with torch.cuda.stream(cs):
                    cache['xd'][lo:hi].copy_(x_host[lo:hi], non_blocking=True)
                    ev = torch.cuda.Event()
                    ev.record(cs)
                cur.wait_event(ev)
                N.check(self.lib, self.handle, self.lib.hsc_b200_mp_begin_part(
                    self.handle, xp, xp, S, T, wsp, cache['wsb'], ctypes.byref(options), lo, hi - lo, sp))
            stt = cache['states']
            pp, ip, cp_ = (ctypes.c_void_p(cache['evp'].data_ptr()), ctypes.c_void_p(cache['evi'].data_ptr()),
                           ctypes.c_void_p(cache['evc'].data_ptr()))
            chunks_p = [[] for _ in range(S)]
            chunks_i = [[] for _ in range(S)]
            chunks_c = [[] for _ in range(S)]
            while True:
                N.check(self.lib, self.handle, self.lib.hsc_b200_mp_run(self.handle, pp, ip, cp_, cap, None, sp))
                self._states_async(stt, cur)
                cache['hp'].copy_(cache['evp'], non_blocking=True)
                cache['hi'].copy_(cache['evi'], non_blocking=True)
                cache['hc'].copy_(cache['evc'], non_blocking=True)
                cur.synchronize()
                hp, hi_, hc = cache['hp'].numpy(), cache['hi'].numpy(), cache['hc'].numpy()
                for s in range(S):
                    nb = stt[s].n_buffered
                    if nb > 0:
                        chunks_p[s].append(hp[s, :nb].copy())
                        chunks_i[s].append(hi_[s, :nb].copy())
                        chunks_c[s].append(hc[s, :nb].copy())
                if not read_states(stt, S)[2]:
                    break
            if want_residual:
                residual_out.copy_(cache['xd'], non_blocking=True)
                cur.synchronize()
            self._fill(res, chunks_p, chunks_i, chunks_c, stt)
            res.residual = residual_out if want_residual else None
            self._last_workspace = cache['ws']
            self._last_shape = (S, T)
        return res

    # ------------------------------------------------------------------ streamed encode, codes left on the device
    def encode_stream_device(self, x, options, capacity=None, min_coefficients=1e-16, want_residual=True):
        """Matching pursuit of B independent signals x [B,T,F], any B, with the canonical codes and the residual left on the
        device.  The signals run in chunks (_stream_chunk_size) through two encode slots (EncodeSlot): the correlation (K1)
        of chunk i+1 runs on its own stream while the pursuit (K2) of chunk i is still in its tail.  Per chunk, on its slot's
        stream: K2, the states to pinned memory, the compaction of the events and their canonical code (canonicalize_codes:
        duplicates summed in float64 in selection order, zero sums and |sum| < min_coefficients (None: none) dropped, entries
        in ascending (t, k) order) plus its entry count to pinned memory.  The host reads a chunk's states only after the next
        chunk has been enqueued.  A chunk in which a signal filled its event buffers is run again at the end with 8x the
        buffers (up to 4096x).

        x: a CUDA tensor on this engine's device - read in place when it is contiguous and of the engine dtype, never
        written -, a pinned host tensor of the engine dtype (copied to the device on a copy stream), or any other host
        tensor or numpy array, which first goes through a pinned staging buffer: its throughput is bounded by that host copy.
        Returns (offsets int64 [B+1], pos int32, idx int32, coef float64: device tensors, the entries of signal b being
        [offsets[b], offsets[b+1]); the B final SignalStates; the residual [B,T,F] of the engine dtype on the device, or None
        when not want_residual)."""
        torch = _torch()
        if isinstance(x, np.ndarray):
            x = torch.from_numpy(np.ascontiguousarray(x))
        assert x.dim() == 3 and x.shape[2] == self.F, 'signals must be [B,T,F=%d]' % self.F
        assert not x.is_cuda or x.device == self.device, 'a CUDA input must be on the engine device %s' % self.device
        B, T = int(x.shape[0]), int(x.shape[1])
        cap = int(capacity) if capacity is not None else self.default_capacity(options, T)
        with torch.cuda.device(self.device):
            cur = torch.cuda.current_stream(self.device)
            resid = torch.empty((B, T, self.F), dtype=self.torch_dtype, device=self.device) if want_residual else None
            done = {}                       # first signal of a finished chunk -> (canonical code, entries, states)
            escalate_capacity(lambda ranges, scale: self._stream_pass(x, ranges, options, cap * scale, min_coefficients, resid, done),
                              [(0, B)] if B > 0 else [], 'encode_stream_device')
            chunks = [done[a] for a in sorted(done)]
            offsets, pos, idx, coef = _concat_codes([(canon, n) for canon, n, _ in chunks], self.device)
            return offsets, pos, idx, coef, [st for _, _, states in chunks for st in states], resid

    def _stream_chunk_size(self, T, capacity, n_signals, options):
        """Signals per chunk of encode_stream_device: two chunks in flight - each with its workspace, an input staging and a
        residual buffer (max_signals_per_chunk), its event buffers and their compaction, its canonical-code buffers and sort
        scratch, and LoCOMP's refit scratch - plus the canonical codes of all n_signals kept until the end, within 80 % of the
        free device memory (the output residual is already allocated).  At most 65535 signals (hsc_b200_mp_begin)."""
        it = self.dtype.itemsize
        extra = capacity * (2 * (8 + it) + 16 + 12)
        if options.method == 1:
            extra += (256 * 257 + 2 * 256) * 8             # kLocompScratchStride doubles per signal
        budget = int(self._free_device_bytes() * 0.8) - n_signals * capacity * 16
        return int(min(65535, self.max_signals_per_chunk(T, budget // 2, extra)))

    def _stream_pass(self, x, ranges, options, cap, min_coefficients, resid, done):
        """One pass of encode_stream_device over the signal ranges [a, b) with event buffers of `cap` per signal.  Finished
        chunks go to `done`; returns the ranges of the chunks that must be run again with larger buffers."""
        torch = _torch()
        T, F = int(x.shape[1]), self.F
        total = sum(b - a for a, b in ranges)
        per = max(1, min(self._stream_chunk_size(T, cap, total, options), max(b - a for a, b in ranges)))
        chunks = []
        for a, b in ranges:
            nc = -(-(b - a) // per)                        # balanced: the last chunk is not a small remainder
            chunks += [(a + (b - a) * c // nc, a + (b - a) * (c + 1) // nc) for c in range(nc)]
        n = max(b - a for a, b in chunks)
        in_place = x.is_cuda and x.dtype == self.torch_dtype and x.is_contiguous()
        direct_h2d = not x.is_cuda and x.is_pinned() and x.dtype == self.torch_dtype and x.is_contiguous()
        slots = self.make_slots(2, n, T, cap, own_residual=resid is None)
        xst = None if in_place else [torch.empty((n, T, F), dtype=self.torch_dtype, device=self.device) for _ in range(2)]
        hst = None
        if not in_place and not direct_h2d and not x.is_cuda:
            # pinned staging of host input, kept on the engine between calls: pinning costs tens of milliseconds per GB
            st_ = getattr(self, '_stream_stage', None)
            if st_ is None or st_[0].shape[0] < n or tuple(st_[0].shape[1:]) != (T, F) or st_[0].dtype != self.torch_dtype:
                self._stream_stage = None
                self._stream_stage = [torch.empty((n, T, F), dtype=self.torch_dtype).pin_memory() for _ in range(2)]
            hst = self._stream_stage
        ctx = getattr(self, '_stream_ctx', None)
        if ctx is None:
            # K1 on the higher-priority stream: its CTAs are placed before waiting K2 CTAs as the previous chunk's tail
            # frees SMs (the pipeline of bench.py)
            ctx = self._stream_ctx = dict(k1=torch.cuda.Stream(device=self.device, priority=-1),
                                          k2=[torch.cuda.Stream(device=self.device) for _ in range(2)],
                                          copy=torch.cuda.Stream(device=self.device))
        s_k1, s_k2, cs = ctx['k1'], ctx['k2'], ctx['copy']
        cur = torch.cuda.current_stream(self.device)
        count = [torch.empty((1,), dtype=torch.int64).pin_memory() for _ in range(2)]
        compacted = [None, None]
        slot_free = [None, None]        # per slot: the last work of its previous chunk
        h2d = [None, None]              # per slot: the copy out of its pinned staging buffer
        rerun = []

        def finish(a, b, k, canon):
            slot_free[k].synchronize()
            snap, status, unfinished = read_states(slots[k].hstate, b - a)
            check_refit_groups(status)
            if unfinished:
                rerun.append((a, b))
                return
            done[a] = (canon, int(count[k][0]), list(snap))

        for st_ in [s_k1, cs] + s_k2:
            st_.wait_stream(cur)                          # the input and the residual may come from work queued on cur
        try:
            pending = None
            for ci, (a, b) in enumerate(chunks):
                k, m = ci & 1, b - a
                sl, s2 = slots[k], s_k2[k]
                if slot_free[k] is not None:
                    s_k1.wait_event(slot_free[k])         # workspace, event buffers, staging: chunk ci-2 is done with them
                if in_place:
                    xd = x[a:b]
                else:
                    src = x[a:b]
                    if hst is not None:
                        if h2d[k] is not None:
                            h2d[k].synchronize()          # chunk ci-2 has left the pinned staging buffer
                        hst[k][:m].copy_(src)
                        src = hst[k][:m]
                    with torch.cuda.stream(cs):
                        if slot_free[k] is not None:
                            cs.wait_event(slot_free[k])
                        xst[k][:m].copy_(src, non_blocking=True)
                        h2d[k] = torch.cuda.Event()
                        h2d[k].record(cs)
                    s_k1.wait_event(h2d[k])
                    xd = xst[k][:m]
                sl.begin(xd, options, s_k1, resid=None if resid is None else resid[a:b])
                k1_done = torch.cuda.Event()
                k1_done.record(s_k1)
                s2.wait_event(k1_done)
                sl.run(s2)
                compacted[k] = sl.compact(compacted[k], s2)
                c = compacted[k]
                canon = self.canonicalize_codes(c['offsets'][:m + 1], c['pos'][:m * cap], c['idx'][:m * cap], c['coef'][:m * cap],
                                                m, T, self.K, None, min_coefficients, stream=s2, handle=sl.handle)[0]
                with torch.cuda.stream(s2):
                    count[k].copy_(canon['offsets'][m:], non_blocking=True)
                slot_free[k] = torch.cuda.Event()
                slot_free[k].record(s2)
                if pending is not None:
                    finish(*pending)
                pending = (a, b, k, canon)
            if pending is not None:
                finish(*pending)
        finally:
            for st_ in [s_k1, cs] + s_k2:
                cur.wait_stream(st_)
            for ev in h2d:
                if ev is not None:
                    ev.synchronize()
        return rerun

    # ------------------------------------------------------------------ K-SVD dictionary update
    def accumulate_code(self, sig, pos, idx, coef, S, T, K, min_coefficients=1e-16):
        """Event lists (selection order, duplicates allowed) -> the accumulated code the reference returns
        (`+=` per (t,k), hsc/modeling.py:992; |c| < minCoefficients dropped, :1171-1177; zeros eliminated, :1181),
        as device tensors sorted by (filter, signal, position) plus the per-filter column pointer (host, [K+1]).
        Sorting / compaction is torch tensor plumbing; the arithmetic on the code happens in the engine."""
        torch = _torch()
        with torch.cuda.device(self.device):
            to = lambda a, dt: (a if torch.is_tensor(a) else torch.from_numpy(np.ascontiguousarray(a))).to(self.device, dt)
            sig, pos, idx, coef = to(sig, torch.int64), to(pos, torch.int64), to(idx, torch.int64), to(coef, torch.float64)
            key = (idx * int(S) + sig) * int(T) + pos
            key, order = torch.sort(key, stable=True)
            uniq, inv = torch.unique_consecutive(key, return_inverse=True)
            c = torch.zeros(uniq.numel(), dtype=torch.float64, device=self.device).index_add_(0, inv, coef[order])
            keep = c != 0.0
            if min_coefficients is not None:
                keep &= c.abs() >= float(min_coefficients)
            uniq, c = uniq[keep], c[keep].contiguous()
            p = (uniq % int(T)).to(torch.int32).contiguous()
            rest = uniq // int(T)
            sg = (rest % int(S)).to(torch.int32).contiguous()
            ix = (rest // int(S)).to(torch.int32).contiguous()
            counts = torch.bincount(ix.long(), minlength=int(K)).cpu().numpy().astype(np.int64)
            col_ptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
        return sg, p, ix, c, col_ptr

    @_with_stream
    def ksvd_update(self, D, sig, pos, idx, coef, col_ptr, S, T, stream=None, group=None, use_pca=False):
        """One dictionary-update stage (hsc/modeling.py:593-636) on the device, float64.  D: numpy [K,L,F];
        (sig, pos, idx, coef, col_ptr) as accumulate_code returns them.  Returns (D_new numpy float64,
        coef_new device tensor, alpha).

        `group`: a torch.distributed process group (or True for the default group) when every rank holds the code of
        its own signals and the same D: per filter the q x q window Gram matrices are summed over the ranks
        (all_reduce, the one exchange the dictionary update needs, SURVEY 8e) and every rank derives the same filter.
        `use_pca`: the usePCA=True variant (:618-625): first principal component of the mean-centred windows."""
        torch = _torch()
        if use_pca and group is not None:
            raise NotImplementedError('usePCA=True under a process group: the window means would have to be shared too')
        N.check(self.lib, self.handle, self.lib.hsc_b200_ksvd_set_pca(self.handle, 1 if use_pca else 0))
        D = np.ascontiguousarray(D, dtype=np.float64)
        K, L, F = D.shape
        with torch.cuda.device(self.device):
            Dd = torch.from_numpy(D).to(self.device)
            coef = coef.clone()
            cp = np.ascontiguousarray(col_ptr, dtype=np.int64)
            assert cp.shape == (K + 1,) and int(cp[-1]) == int(coef.numel())
            alpha = ctypes.c_double(0.0)
            cpp = cp.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))
            args = (ctypes.c_void_p(Dd.data_ptr()), K, L, F, cpp, ctypes.c_void_p(sig.data_ptr()), ctypes.c_void_p(pos.data_ptr()),
                    ctypes.c_void_p(idx.data_ptr()), ctypes.c_void_p(coef.data_ptr()), int(S), int(T))
            if group is None:
                N.check(self.lib, self.handle, self.lib.hsc_b200_ksvd_update(self.handle, *args, ctypes.byref(alpha), self._stream_ptr(stream)))
                return Dd.cpu().numpy(), coef, float(alpha.value)
            import torch.distributed as dist
            pg = None if group is True else group
            counts = torch.from_numpy(np.diff(cp)).to(self.device)
            dist.all_reduce(counts, group=pg)                      # which filters have an atom on ANY rank (:598-599)
            counts = counts.cpu().numpy()
            C = torch.empty((L * F, L * F), dtype=torch.float64, device=self.device)
            sweep = ctypes.c_void_p()
            N.check(self.lib, self.handle, self.lib.hsc_b200_ksvd_begin(
                self.handle, *args, ctypes.c_void_p(C.data_ptr()), self._stream_ptr(stream), ctypes.byref(sweep)))
            try:
                for k in range(K):
                    if counts[k] == 0:
                        continue
                    N.check(self.lib, self.handle, self.lib.hsc_b200_ksvd_filter_gram(sweep, k, None))
                    dist.all_reduce(C, group=pg)                   # sum of the ranks' window Gram matrices
                    N.check(self.lib, self.handle, self.lib.hsc_b200_ksvd_filter_finish(sweep, k, 0))
            finally:
                rc = self.lib.hsc_b200_ksvd_end(sweep, ctypes.byref(alpha))
            N.check(self.lib, self.handle, rc)
            return Dd.cpu().numpy(), coef, float(alpha.value)

    def encode_chunked(self, x, options, capacity=None, budget_bytes=None):
        """encode() over as many signals at a time as the correlation maps fit in free HBM.  x: numpy [S,T,F].
        Returns one EncodeResult for all S signals (no residual)."""
        S, T, _ = x.shape
        per = self.max_signals_per_chunk(T, budget_bytes)
        out = EncodeResult(S, T, self.K)
        out.states = []
        for lo in range(0, S, per):
            r = self.encode(x[lo:lo + per], options, capacity=capacity, return_residual=False)
            n = r.S
            out.pos[lo:lo + n], out.idx[lo:lo + n], out.coef[lo:lo + n] = r.pos, r.idx, r.coef
            out.states.extend(r.states)
            self._last_workspace = None
        return out

    # ------------------------------------------------------------------ convolutional k-means assignment step
    @_with_stream
    def kmeans_assign(self, windows, stream=None):
        """Assignment step of the convolutional k-means learner (hsc/modeling.py:455-480) with the centroids set as
        the dictionary.  windows: device tensor [B,Tw,F] of the engine dtype.  Returns (pos[B] int32 = first sample
        of each window's best patch, idx[B] int32 = its centroid, sums[K,L,F] float64 = sum of the L2-normalised
        assigned patches, counts[K] int32), all device tensors."""
        torch = _torch()
        B, Tw, _ = windows.shape
        with torch.cuda.device(self.device):
            scratch = torch.empty((B, Tw, self.K), dtype=self.torch_dtype, device=self.device)
            pos = torch.empty((B,), dtype=torch.int32, device=self.device)
            idx = torch.empty((B,), dtype=torch.int32, device=self.device)
            sums = torch.empty((self.K, self.L, self.F), dtype=torch.float64, device=self.device)
            counts = torch.empty((self.K,), dtype=torch.int32, device=self.device)
            N.check(self.lib, self.handle, self.lib.hsc_b200_kmeans_assign(
                self.handle, ctypes.c_void_p(windows.data_ptr()), int(B), int(Tw), ctypes.c_void_p(scratch.data_ptr()),
                ctypes.c_void_p(pos.data_ptr()), ctypes.c_void_p(idx.data_ptr()), ctypes.c_void_p(sums.data_ptr()),
                ctypes.c_void_p(counts.data_ptr()), self._stream_ptr(stream)))
        return pos, idx, sums, counts

    def encode_host_pipelined(self, batches, options, capacity=None, n_chunks=8, want_residual=False, residual_outs=None,
                              host_events=True, on_device_events=None, two_workspaces=True):
        """Generator over EncodeResult, one per batch of `batches` (an iterable of host tensors [S,T,F] of the engine
        dtype, ideally pinned, all the same shape).  Per batch: chunked host-to-device copy hidden under the correlation
        (hsc_b200_mp_begin_part), the select/update loop, compaction of the event buffers on the device
        (hsc_b200_mp_compact_events) and the device-to-host read of the codes - exactly 12-16 bytes per atom.  Two sets of
        staging buffers let the copies out of batch i (their own stream) overlap the copy in and the correlation of batch
        i+1 (PCIe is full duplex), and the host-side unpacking of batch i overlaps the GPU work of batch i+1.

        want_residual: also copy the residual [S,T,F] back (as large as the input; off by default - the codes are the
          result, the residual is x - decode(codes)).  `residual_outs`: one host tensor per batch to receive it.
        host_events=False: skip the device-to-host read of the codes (ranks that only feed a gather); the result then
          carries the per-signal counts / states only.
        on_device_events(batch_index, dev): called when a batch is finished, under the code-copy stream, with dev =
          dict(offsets=int64[S+1], pos=int32[..], idx=int32[..], coef=[..], total=n) - the compacted codes still on the
          device (valid until the hook's stream work is done): the hook for the NCCL gather of the sparse codes
          (distributed.gather_device_events); its return value becomes result.gathered.
        two_workspaces: keep one workspace per staging slot when device memory allows (2 x the correlation maps), so that
          the correlation of batch i+1 overlaps the tail of batch i's pursuit.
        A batch whose event buffers overflow (`capacity`) raises: use encode_host for open-ended stop rules."""
        torch = _torch()
        it = iter(batches)
        # staging buffers (device + pinned host) and streams are kept on the engine between calls: pinned allocations
        # cost tens of milliseconds
        cache = getattr(self, '_pipe_cache', None)
        if cache is None:
            cache = self._pipe_cache = dict(slots=[None, None], ctx=dict(copy_in=None, copy_out=None))
        slots, ctx = cache['slots'], cache['ctx']
        for sl_ in slots:                     # an abandoned earlier call may have left copies in flight
            if sl_ is not None and sl_['d2h_done'] is not None:
                sl_['d2h_done'].synchronize()
                sl_['d2h_done'] = None
        ctx['states_copied'] = None
        pending = None          # (slot index, EncodeResult shell, residual_out)

        def make_slot(S, T, cap):
            n_max = S * cap
            d = dict(xd=torch.empty((S, T, self.F), dtype=self.torch_dtype, device=self.device),
                     compact=self._compact_buffers(S, cap),
                     hoff=torch.empty((S + 1,), dtype=torch.int64).pin_memory(),
                     hp=torch.empty((n_max,), dtype=torch.int32).pin_memory(),
                     hi=torch.empty((n_max,), dtype=torch.int32).pin_memory(),
                     hc=torch.empty((n_max,), dtype=self.torch_dtype).pin_memory(),
                     d2h_done=None)
            d['evp'], d['evi'], d['evc'] = self._event_buffers(S, cap)
            d['hstate'], d['states'] = self._pinned_states(S)
            return d

        def finish(p):
            k, res, residual_out = p
            sl = slots[k]
            dev = sl['compact']
            cout = ctx['copy_codes']                  # its own stream: copy_out already holds the next batch's (waiting) work
            sl['small_done'].synchronize()            # states + offsets are on the host
            S = res.S
            # one private copy of the S states, then vectorised unpacking (a Python loop over 512 signals with three
            # array copies each costs several milliseconds per batch)
            snap, _, unfinished = read_states(sl['hstate'], S)
            if unfinished:
                sl['d2h_done'].synchronize()
                raise N.HscError(N.HSC_E_NOMEM, 'encode_host_pipelined: event capacity exhausted before the stop rule fired')
            sl['d2h_done'].synchronize()              # residual (if wanted) and the gather hook's reads of this slot
            off = sl['hoff'].numpy().copy()
            total = int(off[-1])
            res.counts = np.diff(off)
            if on_device_events is not None:
                # the sparse codes are still on the device, compacted: the hook gathers them over the ranks (NCCL)
                with torch.cuda.stream(cout):
                    res.gathered = on_device_events(res.batch_index, dict(dev, total=total))
            if host_events:
                # the codes: exactly `total` atoms cross the bus
                with torch.cuda.stream(cout):
                    sl['hp'][:total].copy_(dev['pos'][:total], non_blocking=True)
                    sl['hi'][:total].copy_(dev['idx'][:total], non_blocking=True)
                    sl['hc'][:total].copy_(dev['coef'][:total], non_blocking=True)
                    done = torch.cuda.Event()
                    done.record(cout)
                sl['d2h_done'] = done
                done.synchronize()
                cuts = off[1:-1]
                res.pos = np.split(sl['hp'].numpy()[:total].copy(), cuts)
                res.idx = np.split(sl['hi'].numpy()[:total].copy(), cuts)
                res.coef = np.split(sl['hc'].numpy()[:total].copy(), cuts)
            res.states = [snap[i] for i in range(S)]
            res.residual = residual_out
            return res

        with torch.cuda.device(self.device):
            cur = torch.cuda.current_stream(self.device)
            for bi, x_host in enumerate(it):
                if isinstance(x_host, np.ndarray):
                    x_host = torch.from_numpy(np.ascontiguousarray(x_host, dtype=self.dtype))
                assert x_host.dim() == 3 and x_host.shape[2] == self.F and x_host.dtype == self.torch_dtype
                S, T, _ = x_host.shape
                cap = int(capacity) if capacity is not None else self.default_capacity(options, T)
                k = bi & 1
                if slots[k] is None or slots[k]['xd'].shape != (S, T, self.F) or slots[k]['evp'].shape[1] != cap:
                    slots[k] = make_slot(S, T, cap)
                wsb = self.workspace_bytes(S, T)
                if ctx.get('copy_in') is None:
                    ctx['copy_in'] = torch.cuda.Stream(device=self.device)
                    ctx['copy_out'] = torch.cuda.Stream(device=self.device)
                    ctx['copy_codes'] = torch.cuda.Stream(device=self.device)
                    ctx['k1'] = torch.cuda.Stream(device=self.device, priority=-1)
                    ctx['k2'] = [torch.cuda.Stream(device=self.device), torch.cuda.Stream(device=self.device)]
                    ctx['wss'] = [None, None]
                # Two workspaces (one per staging slot) when they fit: the correlation of batch i+1 - on its own stream,
                # under the chunks of its copy in - then starts while the pursuit of batch i is still in its tail, and the
                # pursuit of batch i+1 moves into the SMs that tail frees.  One shared workspace otherwise: the correlation
                # of batch i+1 waits for the pursuit of batch i.
                if ctx['wss'][k] is None or ctx['wss'][k].numel() < wsb:
                    ctx['wss'][k] = None
                    other = ctx['wss'][k ^ 1]
                    if two_workspaces and (other is None or other.numel() < wsb or self._free_device_bytes() > wsb + (4 << 30)):
                        ctx['wss'][k] = torch.empty((wsb,), dtype=torch.uint8, device=self.device)
                    else:
                        if other is None or other.numel() < wsb:
                            ctx['wss'][k ^ 1] = other = torch.empty((wsb,), dtype=torch.uint8, device=self.device)
                        ctx['wss'][k] = other                       # shared
                shared_ws = ctx['wss'][0] is ctx['wss'][1]
                handles = [self.handle, self.handle] if shared_ws else self._views_for(2)
                sl, ws, cin, cout = slots[k], ctx['wss'][k], ctx['copy_in'], ctx['copy_out']
                s_k1, s_k2, hk = ctx['k1'], ctx['k2'][k], handles[k]
                if bi == 0:
                    for st_ in (cin, s_k1, ctx['k2'][0], ctx['k2'][1]):
                        st_.wait_stream(cur)                        # work queued by the caller before this call
                residual_out = None
                if want_residual:
                    residual_out = residual_outs[bi] if residual_outs is not None else (
                        torch.empty_like(x_host).pin_memory() if x_host.is_pinned() else torch.empty_like(x_host))
                # this slot's staging buffers (and its workspace) are free once the copies of batch bi-2 have left them;
                # a shared workspace also waits for the pursuit and the compaction of batch bi-1
                if sl['d2h_done'] is not None:
                    cin.wait_event(sl['d2h_done'])
                    s_k1.wait_event(sl['d2h_done'])
                if shared_ws and ctx.get('states_copied') is not None:
                    s_k1.wait_event(ctx['states_copied'])
                xp, wsp = ctypes.c_void_p(sl['xd'].data_ptr()), ctypes.c_void_p(ws.data_ptr())
                k1p = ctypes.c_void_p(s_k1.cuda_stream)
                nch = max(1, min(int(n_chunks), S))
                for c in range(nch):
                    lo, hi = S * c // nch, S * (c + 1) // nch
                    with torch.cuda.stream(cin):
                        sl['xd'][lo:hi].copy_(x_host[lo:hi], non_blocking=True)
                        ev = torch.cuda.Event()
                        ev.record(cin)
                    s_k1.wait_event(ev)
                    N.check(self.lib, hk, self.lib.hsc_b200_mp_begin_part(
                        hk, xp, xp, S, T, wsp, wsb, ctypes.byref(options), lo, hi - lo, k1p))
                k1_done = torch.cuda.Event()
                k1_done.record(s_k1)
                s_k2.wait_event(k1_done)
                N.check(self.lib, hk, self.lib.hsc_b200_mp_run(
                    hk, ctypes.c_void_p(sl['evp'].data_ptr()), ctypes.c_void_p(sl['evi'].data_ptr()),
                    ctypes.c_void_p(sl['evc'].data_ptr()), cap, None, ctypes.c_void_p(s_k2.cuda_stream)))
                k2_done = torch.cuda.Event()
                k2_done.record(s_k2)
                if shared_ws:
                    s_k1.wait_event(k2_done)                        # the next correlation overwrites this map
                with torch.cuda.stream(cout):
                    cout.wait_event(k2_done)
                    self._states_async(sl['states'], cout, hk)
                    self.compact_events(sl['evp'], sl['evi'], sl['evc'], out=sl['compact'], stream=cout, handle=hk)
                    ctx['states_copied'] = torch.cuda.Event()       # a shared workspace's states may be reset by the next batch
                    ctx['states_copied'].record(cout)
                    sl['hoff'].copy_(sl['compact']['offsets'], non_blocking=True)
                    small = torch.cuda.Event()
                    small.record(cout)
                    sl['small_done'] = small
                    if want_residual:
                        residual_out.copy_(sl['xd'], non_blocking=True)
                    done = torch.cuda.Event()
                    done.record(cout)
                sl['d2h_done'] = done
                self._last_workspace, self._last_shape = ws, (S, T)
                shell = EncodeResult(S, T, self.K)
                shell.batch_index = bi
                if pending is not None:
                    yield finish(pending)
                pending = (k, shell, residual_out)
            if pending is not None:
                yield finish(pending)
            for st_ in (ctx['copy_out'], ctx['copy_codes']):
                cur.wait_stream(st_)

    def _fill(self, res, cp, ci, cc, states):
        for s in range(res.S):
            res.pos[s] = np.concatenate(cp[s]) if cp[s] else np.zeros(0, np.int32)
            res.idx[s] = np.concatenate(ci[s]) if ci[s] else np.zeros(0, np.int32)
            res.coef[s] = np.concatenate(cc[s]) if cc[s] else np.zeros(0, self.dtype)
        res.states = [N.SignalState.from_buffer_copy(bytes(states[s])) for s in range(res.S)]

    def map_snapshot(self):
        """Copy of the correlation map of the last encode [S,T,K] (tests / diagnostics)."""
        S, T = self._last_shape
        return self._to_host(self.lib.hsc_b200_mp_map_dev(self.handle), (S, T, self.K))

    # ------------------------------------------------------------------ decoder
    @_with_stream
    def decode(self, pos, idx, coef, T, out=None, stream=None):
        """reconstructSignal for one signal: returns the device tensor [T,F] (+= into `out` if given).  The S = 1 case of
        decode_batch."""
        torch = _torch()
        T = int(T)
        with torch.cuda.device(self.device):
            if out is None:
                out = torch.zeros((T, self.F), dtype=self.torch_dtype, device=self.device)
            n = len(np.asarray(pos))
            self.decode_batch(np.array([0, n], dtype=np.int64), pos, idx, coef, 1, T, out=out.view(1, T, self.F))
        return out

    @_with_stream
    def decode_batch(self, offsets, pos, idx, coef, S, T, out=None, stream=None):
        """reconstructSignal for S signals of length T in one launch: returns the device tensor [S,T,F] (+= into `out` if
        given).  The atoms of signal s are entries [offsets[s], offsets[s+1]) of the flat host arrays pos / idx / coef
        (offsets: S+1 integers from 0, the layout compact_events returns).  Each signal's atoms are put in the order decode()
        uses (stable sort by position), so signal s gets bit for bit what decode() gives for its atoms alone."""
        torch = _torch()
        S, T = int(S), int(T)
        offsets = np.asarray(offsets, dtype=np.int64)
        pos = np.asarray(pos, dtype=np.int32)
        assert offsets.shape == (S + 1,) and offsets[0] == 0 and np.all(np.diff(offsets) >= 0) and offsets[S] == len(pos)
        assert len(idx) == len(pos) and len(coef) == len(pos)
        with torch.cuda.device(self.device):
            if out is None:
                out = torch.zeros((S, T, self.F), dtype=self.torch_dtype, device=self.device)
            if len(pos) == 0:
                assert out.shape == (S, T, self.F) and out.dtype == self.torch_dtype and out.is_contiguous()
                return out
            # stable within each signal: the segments are already in signal order, lexsort keeps equal positions in list order
            order = np.lexsort((pos, np.repeat(np.arange(S, dtype=np.int64), np.diff(offsets))))
            o = torch.from_numpy(offsets).to(self.device)
            p = torch.from_numpy(np.ascontiguousarray(pos[order])).to(self.device)
            i = torch.from_numpy(np.ascontiguousarray(np.asarray(idx, dtype=np.int32)[order])).to(self.device)
            c = torch.from_numpy(np.ascontiguousarray(np.asarray(coef, dtype=self.dtype)[order])).to(self.device)
            return self.decode_batch_device(o, p, i, c, S, T, out)

    @_with_stream
    def decode_batch_device(self, offsets, pos, idx, coef, S, T, out, stream=None):
        """decode_batch for atoms already on the device and in decode order: out [S,T,F] (device, engine dtype) += the
        reconstruction of S signals whose atoms are entries [offsets[s], offsets[s+1]) of the device tensors pos / idx
        (int32) / coef (engine dtype), sorted by position within each signal (the order canonicalize_codes writes).  One
        launch, no host work on the atoms.  Asynchronous; returns out."""
        torch = _torch()
        S, T = int(S), int(T)
        assert out.shape == (S, T, self.F) and out.dtype == self.torch_dtype and out.is_contiguous() and out.device == self.device
        assert offsets.shape == (S + 1,) and offsets.dtype == torch.int64 and offsets.device == self.device
        assert pos.dtype == torch.int32 and idx.dtype == torch.int32 and coef.dtype == self.torch_dtype
        assert all(t.device == self.device and t.is_contiguous() for t in (pos, idx, coef))
        if pos.numel() == 0:
            return out
        with torch.cuda.device(self.device):
            N.check(self.lib, self.handle, self.lib.hsc_b200_decode_batch(
                self.handle, ctypes.c_void_p(offsets.data_ptr()), ctypes.c_void_p(pos.data_ptr()), ctypes.c_void_p(idx.data_ptr()),
                ctypes.c_void_p(coef.data_ptr()), S, T, ctypes.c_void_p(out.data_ptr()), self._stream_ptr(stream)))
        return out

    @_with_stream
    def canonicalize_codes(self, offsets, pos, idx, coef, S, T, K, level_bounds=None, min_coefficients=1e-16, stream=None,
                           handle=None):
        """Canonical codes of S signals from their flat, selection-ordered events on the device (the layout compact_events
        returns: offsets int64 [S+1], pos / idx int32, coef of the engine dtype; the events of signal s are
        [offsets[s], offsets[s+1])).  Every signal gets one entry per distinct (t, k), the float64 sum of its events in
        selection order, without zero sums and sums below min_coefficients (None = keep all), in ascending (t, k) order.
        With level_bounds [b_0 <= ... <= b_{L-2}], an entry with filter k goes to the first level j with k < b_j, else to the
        last one (convertToDistributedCoefficients); without, there is one level.  Returns one dict per level: offsets int64
        [S+1] (from 0) and pos / idx int32, coef float64 device tensors with room for every event (len(pos) entries); level
        j's entries are the first offsets[S] of them.  Asynchronous: nothing is read back.  `handle`: the native handle whose
        sort scratch the launch uses (default: this engine's; an EncodeSlot's when several chunks are in flight)."""
        torch = _torch()
        S, T, K = int(S), int(T), int(K)
        bounds = np.ascontiguousarray([] if level_bounds is None else level_bounds, dtype=np.int64)
        assert bounds.ndim == 1
        n_levels = len(bounds) + 1
        assert offsets.shape == (S + 1,) and offsets.dtype == torch.int64
        assert pos.dtype == torch.int32 and idx.dtype == torch.int32 and coef.dtype == self.torch_dtype
        assert pos.numel() == idx.numel() == coef.numel()
        assert all(t.device == self.device and t.is_contiguous() for t in (offsets, pos, idx, coef))
        cap = pos.numel()
        with torch.cuda.device(self.device):
            off = torch.empty((n_levels, S + 1), dtype=torch.int64, device=self.device)
            p = torch.empty((n_levels, cap), dtype=torch.int32, device=self.device)
            i = torch.empty((n_levels, cap), dtype=torch.int32, device=self.device)
            c = torch.empty((n_levels, cap), dtype=torch.float64, device=self.device)
            ptr = lambda t: ctypes.c_void_p(t.data_ptr())
            h = self.handle if handle is None else handle
            N.check(self.lib, h, self.lib.hsc_b200_canonicalize_codes(
                h, ptr(offsets), ptr(pos), ptr(idx), ptr(coef), cap, S, T, K,
                bounds.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), len(bounds),
                -1.0 if min_coefficients is None else float(min_coefficients), ptr(off), ptr(p), ptr(i), ptr(c),
                self._stream_ptr(stream)))
        return [dict(offsets=off[j], pos=p[j], idx=i[j], coef=c[j]) for j in range(n_levels)]


class EncodeSlot(object):
    """One encode in flight: a native view of the engine's dictionary with its own workspace (correlation map, argmax
    hierarchy, states), event buffers and residual.  begin() = K1 + state reset, run() = K2, both asynchronous on the
    stream given; states_async() copies the per-signal states to the slot's pinned buffer.  An encode may hold fewer
    signals than the slot was made for (the last chunk of a stream): begin() takes them from xd, and run() / compact()
    work on that many."""

    def __init__(self, eng, handle, S, T, capacity, own_residual=True):
        torch = _torch()
        self.eng, self.handle = eng, handle
        self.S, self.T, self.cap = int(S), int(T), int(capacity)
        self.n = self.S                 # signals of the encode in flight
        dev = eng.device
        with torch.cuda.device(dev):
            self.wsb = eng.workspace_bytes(S, T)
            self.ws = torch.empty((self.wsb,), dtype=torch.uint8, device=dev)
            self.resid = torch.empty((S, T, eng.F), dtype=eng.torch_dtype, device=dev) if own_residual else None
            self.evp, self.evi, self.evc = eng._event_buffers(S, capacity)
            self.hstate, self.states = eng._pinned_states(S)
        self.k2_done = None

    def begin(self, xd, options, stream, resid=None):
        """K1 + state reset of the xd.shape[0] <= S signals xd (device, engine dtype, contiguous); the residual goes to
        `resid` (same shape; default: the slot's own buffer)."""
        e = self.eng
        n = int(xd.shape[0])
        assert 0 < n <= self.S and tuple(xd.shape) == (n, self.T, e.F) and xd.dtype == e.torch_dtype and xd.is_contiguous()
        if resid is None:
            resid = self.resid[:n]
        assert resid.shape == xd.shape and resid.dtype == xd.dtype and resid.is_contiguous() and resid.device == xd.device
        N.check(e.lib, self.handle, e.lib.hsc_b200_mp_begin(
            self.handle, ctypes.c_void_p(xd.data_ptr()), ctypes.c_void_p(resid.data_ptr()), n, self.T,
            ctypes.c_void_p(self.ws.data_ptr()), self.wsb, ctypes.byref(options), ctypes.c_void_p(stream.cuda_stream)))
        self.n = n

    def run(self, stream):
        e = self.eng
        N.check(e.lib, self.handle, e.lib.hsc_b200_mp_run(
            self.handle, ctypes.c_void_p(self.evp.data_ptr()), ctypes.c_void_p(self.evi.data_ptr()),
            ctypes.c_void_p(self.evc.data_ptr()), self.cap, None, ctypes.c_void_p(stream.cuda_stream)))
        e._states_async(self.states, stream, self.handle)

    def compact(self, out, stream):
        n, e = self.n, self.eng
        if out is None:
            out = e._compact_buffers(self.S, self.cap)       # room for a full slot, allocated in the caller's stream context
        return e.compact_events(self.evp[:n], self.evi[:n], self.evc[:n], out=out, stream=stream, handle=self.handle)

    def launches(self):
        return int(self.eng.lib.hsc_b200_launch_count(self.handle))


_engines = {}
_dict_engines = {}


def engine_for_dictionary(D, weights=None, dtype=None, device=None, max_entries=16):
    """An engine that already holds dictionary D (weights, dtype): callers that alternate between a few dictionaries - the
    levels of a multilevel dictionary, their input-level representations for decoding - get one native engine per
    dictionary (D, Gram tensor and K1 operand stay on the device between calls) instead of re-uploading on every switch.
    Small LRU per (process, device), keyed by the dictionary's bytes."""
    import os
    torch = _torch()
    if not torch.cuda.is_available():
        raise RuntimeError('hierarchical_sparse_coding_b200 needs a CUDA device (no CPU fallback)')
    idx = torch.cuda.current_device() if device is None else int(torch.device(device).index or 0) if not isinstance(device, int) else device
    D = np.asarray(D)
    dt = np.dtype(dtype) if dtype is not None else np.dtype(engine_dtype(D))
    Dc = np.ascontiguousarray(D if D.ndim == 3 else D[:, :, None], dtype=dt)
    wc = None if weights is None else np.ascontiguousarray(np.asarray(weights), dtype=dt)
    key = (os.getpid(), idx, str(dt), Dc.shape, hash(Dc.tobytes()), None if wc is None else hash(wc.tobytes()))
    cache = _dict_engines
    eng = cache.pop(key, None)
    if eng is None:
        eng = Engine(idx)
        eng.set_dictionary(Dc, weights=wc, dtype=dt)
        while len(cache) >= max_entries:
            old = cache.pop(next(iter(cache)))
            old.close()
    cache[key] = eng            # most recently used last
    return eng


def get_engine(device=None):
    """Process-wide engine per device (created lazily, after fork: the reference's Pool fan-out,
    scripts/scale_weight_effect_mlcsc.py:165, must not inherit a CUDA context)."""
    import os
    torch = _torch()
    if not torch.cuda.is_available():
        raise RuntimeError('hierarchical_sparse_coding_b200 needs a CUDA device (no CPU fallback)')
    idx = torch.cuda.current_device() if device is None else int(torch.device(device).index or 0) if not isinstance(device, int) else device
    key = (os.getpid(), idx)
    if key not in _engines:
        _engines[key] = Engine(idx)
    return _engines[key]
