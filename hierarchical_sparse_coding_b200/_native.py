"""ctypes binding of the engine's C ABI (include/hsc_b200.h).

The library is the product: there is no CPU fallback.  `load_library()` raises if the shared
object has not been built (`python -m hierarchical_sparse_coding_b200.build`), and creating an
engine raises if no CUDA device is present.
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('HSC_B200_LIB') or os.path.join(HERE, 'libhsc_b200.so')

HSC_F32, HSC_F64 = 0, 1

HSC_OK = 0
HSC_E_INVALID, HSC_E_CUDA, HSC_E_UNSUPPORTED, HSC_E_STATE, HSC_E_NOMEM = -1, -2, -3, -4, -5

(HSC_RUNNING, HSC_STOP_ENERGY, HSC_STOP_NNZ, HSC_STOP_SNR, HSC_STOP_SCALE, HSC_STOP_EMPTY,
 HSC_PAUSE_CAPACITY, HSC_PAUSE_PASSES, HSC_STOP_MAX_EVENTS, HSC_STOP_STALL, HSC_STOP_GROUP) = range(11)

STOP_NAMES = {HSC_RUNNING: 'running', HSC_STOP_ENERGY: 'energy', HSC_STOP_NNZ: 'nnz', HSC_STOP_SNR: 'snr',
              HSC_STOP_SCALE: 'scale', HSC_STOP_EMPTY: 'empty', HSC_PAUSE_CAPACITY: 'capacity',
              HSC_PAUSE_PASSES: 'passes', HSC_STOP_MAX_EVENTS: 'max_events', HSC_STOP_STALL: 'stall',
              HSC_STOP_GROUP: 'group_too_large'}

# every symbol include/hsc_b200.h declares (checked by tests/test_abi.py without a GPU)
EXPORTED_SYMBOLS = [
    'hsc_b200_create', 'hsc_b200_destroy', 'hsc_b200_last_error', 'hsc_b200_abi_version',
    'hsc_b200_set_dictionary', 'hsc_b200_dictionary_dev', 'hsc_b200_gram_dev', 'hsc_b200_correlate',
    'hsc_b200_workspace_bytes', 'hsc_b200_mp_begin', 'hsc_b200_mp_run', 'hsc_b200_mp_states',
    'hsc_b200_mp_map_dev', 'hsc_b200_decode', 'hsc_b200_mp_encode_host', 'hsc_b200_launch_count', 'hsc_b200_copy_to_host', 'hsc_b200_create_view',
    'hsc_b200_mp_states_async', 'hsc_b200_mp_begin_part', 'hsc_b200_ksvd_update', 'hsc_b200_ksvd_set_pca', 'hsc_b200_kmeans_assign',
    'hsc_b200_ksvd_begin', 'hsc_b200_ksvd_filter_gram', 'hsc_b200_ksvd_filter_finish', 'hsc_b200_ksvd_end',
    'hsc_b200_mp_compact_events', 'hsc_b200_mp_events_to_dense', 'hsc_b200_decode_batch', 'hsc_b200_canonicalize_codes',
]


class MpOptions(ctypes.Structure):
    _fields_ = [('nb_nonzero_coefs', ctypes.c_int64),
                ('tolerance_snr', ctypes.c_double),
                ('tolerance_residual_scale', ctypes.c_double),
                ('min_coefficients', ctypes.c_double),
                ('nb_blocks', ctypes.c_int32),
                ('use_weights', ctypes.c_int32),
                ('coef_mode', ctypes.c_int32),
                ('method', ctypes.c_int32),
                ('max_passes_per_run', ctypes.c_int64),
                ('max_events_total', ctypes.c_int64),
                ('rerank_tolerance', ctypes.c_double),
                ('energy_eps', ctypes.c_double)]


class SignalState(ctypes.Structure):
    _fields_ = [('energy_signal', ctypes.c_double),
                ('energy_residual', ctypes.c_double),
                ('n_events', ctypes.c_int64),
                ('n_buffered', ctypes.c_int64),
                ('nnz', ctypes.c_int64),
                ('duplicates', ctypes.c_int64),
                ('passes', ctypes.c_int64),
                ('status', ctypes.c_int32),
                ('offset_flag', ctypes.c_int32),
                ('initialised', ctypes.c_int32),
                ('pass_count', ctypes.c_int32),
                ('pass_cursor', ctypes.c_int32),
                ('reserved', ctypes.c_int32),
                ('reranked', ctypes.c_int64),
                ('edge_written', ctypes.c_uint64 * 2)]


class HscError(RuntimeError):
    def __init__(self, code, text):
        RuntimeError.__init__(self, 'hsc_b200 error %d: %s' % (code, text))
        self.code = code


_lib = None


def load_library():
    """dlopen()s libhsc_b200.so and declares the prototypes.  Raises if it was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError('libhsc_b200.so is not built (%s); run `python -m hierarchical_sparse_coding_b200.build`. '
                          'There is no CPU fallback.' % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    vp, i32, i64, sz = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_size_t
    lib.hsc_b200_abi_version.restype = ctypes.c_int
    lib.hsc_b200_abi_version.argtypes = []
    lib.hsc_b200_create.restype = ctypes.c_int
    lib.hsc_b200_create.argtypes = [ctypes.c_int, ctypes.POINTER(vp)]
    lib.hsc_b200_destroy.restype = ctypes.c_int
    lib.hsc_b200_destroy.argtypes = [vp]
    lib.hsc_b200_last_error.restype = ctypes.c_char_p
    lib.hsc_b200_last_error.argtypes = [vp]
    lib.hsc_b200_launch_count.restype = i64
    lib.hsc_b200_launch_count.argtypes = [vp]
    lib.hsc_b200_set_dictionary.restype = ctypes.c_int
    lib.hsc_b200_set_dictionary.argtypes = [vp, vp, ctypes.c_int, i64, i64, i64, vp]
    lib.hsc_b200_dictionary_dev.restype = vp
    lib.hsc_b200_dictionary_dev.argtypes = [vp]
    lib.hsc_b200_gram_dev.restype = vp
    lib.hsc_b200_gram_dev.argtypes = [vp]
    lib.hsc_b200_correlate.restype = ctypes.c_int
    lib.hsc_b200_correlate.argtypes = [vp, vp, i64, i64, vp, vp]
    lib.hsc_b200_workspace_bytes.restype = sz
    lib.hsc_b200_workspace_bytes.argtypes = [vp, i64, i64]
    lib.hsc_b200_mp_begin.restype = ctypes.c_int
    lib.hsc_b200_mp_begin.argtypes = [vp, vp, vp, i64, i64, vp, sz, ctypes.POINTER(MpOptions), vp]
    lib.hsc_b200_mp_begin_part.restype = ctypes.c_int
    lib.hsc_b200_mp_begin_part.argtypes = [vp, vp, vp, i64, i64, vp, sz, ctypes.POINTER(MpOptions), i64, i64, vp]
    lib.hsc_b200_mp_run.restype = ctypes.c_int
    lib.hsc_b200_mp_run.argtypes = [vp, vp, vp, vp, i64, ctypes.POINTER(SignalState), vp]
    lib.hsc_b200_mp_states.restype = ctypes.c_int
    lib.hsc_b200_mp_states.argtypes = [vp, ctypes.POINTER(SignalState), vp]
    lib.hsc_b200_mp_compact_events.restype = ctypes.c_int
    lib.hsc_b200_mp_compact_events.argtypes = [vp, vp, vp, vp, i64, vp, vp, vp, vp, i64, vp]
    lib.hsc_b200_mp_events_to_dense.restype = ctypes.c_int
    lib.hsc_b200_mp_events_to_dense.argtypes = [vp, vp, vp, vp, i64, ctypes.c_double, vp, vp]
    lib.hsc_b200_mp_map_dev.restype = vp
    lib.hsc_b200_mp_map_dev.argtypes = [vp]
    lib.hsc_b200_decode.restype = ctypes.c_int
    lib.hsc_b200_decode.argtypes = [vp, vp, vp, vp, i64, i64, vp, vp]
    lib.hsc_b200_decode_batch.restype = ctypes.c_int
    lib.hsc_b200_decode_batch.argtypes = [vp, vp, vp, vp, vp, i64, i64, vp, vp]
    lib.hsc_b200_canonicalize_codes.restype = ctypes.c_int
    lib.hsc_b200_canonicalize_codes.argtypes = [vp, vp, vp, vp, vp, i64, i64, i64, i64, ctypes.POINTER(i64), i64, ctypes.c_double,
                                                vp, vp, vp, vp, vp]
    lib.hsc_b200_mp_encode_host.restype = ctypes.c_int
    lib.hsc_b200_mp_encode_host.argtypes = [vp, vp, i64, i64, ctypes.POINTER(MpOptions), vp, vp, vp, i64, vp, vp,
                                            ctypes.POINTER(SignalState)]
    lib.hsc_b200_create_view.restype = ctypes.c_int
    lib.hsc_b200_create_view.argtypes = [vp, ctypes.POINTER(vp)]
    lib.hsc_b200_mp_states_async.restype = ctypes.c_int
    lib.hsc_b200_mp_states_async.argtypes = [vp, ctypes.POINTER(SignalState), vp]
    lib.hsc_b200_ksvd_update.restype = ctypes.c_int
    lib.hsc_b200_ksvd_update.argtypes = [vp, vp, i64, i64, i64, ctypes.POINTER(i64), vp, vp, vp, vp, i64, i64,
                                         ctypes.POINTER(ctypes.c_double), vp]
    lib.hsc_b200_ksvd_set_pca.restype = ctypes.c_int
    lib.hsc_b200_ksvd_set_pca.argtypes = [vp, ctypes.c_int]
    lib.hsc_b200_ksvd_begin.restype = ctypes.c_int
    lib.hsc_b200_ksvd_begin.argtypes = [vp, vp, i64, i64, i64, ctypes.POINTER(i64), vp, vp, vp, vp, i64, i64, vp, vp, ctypes.POINTER(vp)]
    lib.hsc_b200_ksvd_filter_gram.restype = ctypes.c_int
    lib.hsc_b200_ksvd_filter_gram.argtypes = [vp, i64, ctypes.POINTER(i64)]
    lib.hsc_b200_ksvd_filter_finish.restype = ctypes.c_int
    lib.hsc_b200_ksvd_filter_finish.argtypes = [vp, i64, ctypes.c_int]
    lib.hsc_b200_ksvd_end.restype = ctypes.c_int
    lib.hsc_b200_ksvd_end.argtypes = [vp, ctypes.POINTER(ctypes.c_double)]
    lib.hsc_b200_kmeans_assign.restype = ctypes.c_int
    lib.hsc_b200_kmeans_assign.argtypes = [vp, vp, i64, i64, vp, vp, vp, vp, vp, vp]
    lib.hsc_b200_copy_to_host.restype = ctypes.c_int
    lib.hsc_b200_copy_to_host.argtypes = [vp, vp, vp, sz]
    _lib = lib
    return lib


def check(lib, handle, rc):
    if rc != HSC_OK:
        text = lib.hsc_b200_last_error(handle) if handle else b'engine creation failed (no CUDA device?)'
        raise HscError(rc, (text or b'').decode('utf-8', 'replace'))
