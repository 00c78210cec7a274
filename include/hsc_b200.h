/*
 * hsc_b200.h -- C ABI of the B200-native convolutional matching-pursuit engine.
 *
 * This is the drop-in boundary for the matching-pursuit hot path of
 * sbrodeur/hierarchical-sparse-coding (all citations relative to that tree):
 *
 *   SparseApproximator.computeCoefficients(X, D, ...)              hsc/modeling.py:657-660
 *   ConvolutionalMatchingPursuit.computeCoefficients               hsc/modeling.py:1053-1186
 *   convolve1d (initial correlation)                               hsc/modeling.py:149-188
 *   _selectBestAtoms / _updateResidual / _updateInnerProducts      hsc/modeling.py:899-1051
 *   reconstructSignal (sparse decoder)                             hsc/modeling.py:226-245
 *
 * The reference's in-tree precedent for a native backend behind that interface is the MPTK plug-in
 * (hsc/modeling.py:749-837), which hands the dictionary and the signal to an external library and
 * gets (position, filter, coefficient) atoms back.  The entry points below are what a binding for
 * THIS engine binds instead; INTEGRATION.md shows the ctypes stub.
 *
 * Conventions
 *   - plain C: pointers and sizes only, no torch / C++ types.
 *   - `dtype`: HSC_F32 (float) or HSC_F64 (double) is the arithmetic type of the whole path: signal,
 *     dictionary, correlation map, coefficients.  The reference computes in the NumPy result type of
 *     (signal, dictionary): float32 data -> float32, level >= 1 of the hierarchy -> float64.
 *   - layouts are the reference's, C order: signal x[S][T][F], dictionary D[K][L][F], correlation map
 *     c[S][T][K]; atom position = CENTRE index, centre tap = L/2-1 (even L) or L/2 (odd L)
 *     (hsc/utils.py:76-161, hsc/modeling.py:845-858).
 *   - `*_dev` pointers are device memory of the engine's device, `*_host` pointers are host memory.
 *     `stream` is a cudaStream_t passed as void* (NULL = default stream).  Calls are asynchronous
 *     on that stream unless stated otherwise.
 *   - every function returns HSC_OK (0) or a negative hsc_status; text via hsc_b200_last_error().
 *   - there is no CPU fallback: without a CUDA device hsc_b200_create() fails.
 */
#ifndef HSC_B200_H_
#define HSC_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HSC_B200_ABI_VERSION 2

typedef enum {
    HSC_OK = 0,
    HSC_E_INVALID = -1,      /* bad argument (shape, dtype, null pointer): the reference's AssertionError */
    HSC_E_CUDA = -2,         /* CUDA runtime / driver failure */
    HSC_E_UNSUPPORTED = -3,  /* valid request the engine does not implement */
    HSC_E_STATE = -4,        /* call order (no dictionary set, no encode in flight, ...) */
    HSC_E_NOMEM = -5         /* workspace too small */
} hsc_status;

typedef enum { HSC_F32 = 0, HSC_F64 = 1 } hsc_dtype;

/* Why a signal's pursuit stopped (hsc/modeling.py:1125-1158). */
typedef enum {
    HSC_RUNNING = 0,
    HSC_STOP_ENERGY = 1,     /* residual energy < eps                  (:1125-1130) */
    HSC_STOP_NNZ = 2,        /* nnz >= nbNonzeroCoefs                  (:1135-1138) */
    HSC_STOP_SNR = 3,        /* snr >= toleranceSnr                    (:1139-1142) */
    HSC_STOP_SCALE = 4,      /* max|residual| <= toleranceResidualScale(:1145-1148) */
    HSC_STOP_EMPTY = 5,      /* selection returned no atom             (:1150-1153) */
    HSC_PAUSE_CAPACITY = 6,  /* event buffer full: drain it and call hsc_b200_mp_run again */
    HSC_PAUSE_PASSES = 7,    /* max_passes_per_run reached (host-side stopCondition callbacks) */
    HSC_STOP_MAX_EVENTS = 8, /* max_events_total atoms applied (not a reference rule: bounded samples) */
    HSC_STOP_STALL = 9,      /* LoCOMP: |delta residual energy| < eps          (:1377-1381) */
    HSC_STOP_GROUP = 10      /* LoCOMP: more common-support atoms than the device refit holds (256) */
} hsc_stop;

/* Keyword arguments of computeCoefficients (hsc/modeling.py:1053).  Absent values: negative /
 * NaN as documented per field. */
typedef struct {
    int64_t nb_nonzero_coefs;      /* nbNonzeroCoefs, < 0 = None */
    double tolerance_snr;          /* toleranceSnr in dB, NaN = None */
    double tolerance_residual_scale; /* toleranceResidualScale, NaN = None */
    double min_coefficients;       /* minCoefficients used as the null threshold of the selection
                                      (:1088, :974); < 0 = None.  The final |c| >= minCoefficients
                                      clip of the accumulated code (:1171-1177) is the caller's. */
    int32_t nb_blocks;             /* nbBlocks: 1, > 1, or -1 for 'auto' (block size 4L) */
    int32_t use_weights;           /* 1: bias the selection by the weights given to set_dictionary */
    int32_t coef_mode;             /* 0: coefficient = map entry (the reference's arithmetic path);
                                      1: interior atoms re-evaluate <residual, D[k]> at selection */
    int32_t method;                /* 0: matching pursuit (:1053); 1: LoCOMP, least-squares refit of the
                                      common-support atoms per selection (:1263) */
    int64_t max_passes_per_run;    /* <= 0 = unlimited; 1 lets the host run a stopCondition callback
                                      between selection passes (:1155-1158) */
    int64_t max_events_total;      /* <= 0 = unlimited; bounds applied atoms (bounded timing samples) */
    double rerank_tolerance;       /* float32 maps: before an atom is picked, every map entry whose score lies within
                                      rerank_tolerance * (best score + largest initial score) of the best one is
                                      re-scored from the residual in float64 and the best re-scored entry wins, so that
                                      the pick does not depend on the rounding of the tensor-core correlation or of the
                                      Gram updates (north star: same atoms but for near-ties below 1e-6).  < 0 = the
                                      default (4e-6), 0 = off */
    double energy_eps;             /* threshold of the residual-energy stop (:1125-1130) and of LoCOMP's stall stop
                                      (:1377-1381): the reference uses np.finfo(D.dtype).eps (:1057), the DICTIONARY's
                                      dtype, which differs from the arithmetic type when a float32 dictionary meets
                                      float64 data (levels >= 1 of the hierarchy).  <= 0 = eps of the arithmetic type */
} hsc_mp_options;

/* Per-signal state, readable after hsc_b200_mp_run. */
typedef struct {
    double energy_signal;          /* sum x^2                               (:1070) */
    double energy_residual;        /* incrementally tracked residual energy (:1014) */
    int64_t n_events;              /* atoms applied so far, duplicates included */
    int64_t n_buffered;            /* events currently in the output buffer of this signal */
    int64_t nnz;                   /* distinct (t,k) selected               (:1106-1111) */
    int64_t duplicates;            /* re-selections of an existing (t,k)    (:1108) */
    int64_t passes;                /* selection passes                      (:1160) */
    int32_t status;                /* hsc_stop */
    int32_t offset_flag;           /* block-selection half-block offset toggle (:1163) */
    int32_t initialised;
    int32_t pass_count;            /* atoms selected by the current pass (block selection, :908-963) */
    int32_t pass_cursor;           /* how many of them have been applied (a pause may fall mid-pass) */
    int32_t reserved;              /* float bits of the largest score of the initial map (scale of the re-rank window) */
    int64_t reranked;              /* selections that went through the near-tie re-scoring (rerank_tolerance) */
    uint64_t edge_written[2];      /* rows whose filter support overhangs the signal start / end and that an atom's
                                      window has re-correlated with reflect padding (:1046): bit r / bit T-1-r */
} hsc_signal_state;

typedef struct hsc_engine hsc_engine;

/* Lifetime.  `device` is the CUDA ordinal; the context is created lazily here (per process, so the
 * reference's fork-based fan-out keeps working: scripts/scale_weight_effect_mlcsc.py:165). */
int hsc_b200_create(int device, hsc_engine** out);
int hsc_b200_destroy(hsc_engine* e);
const char* hsc_b200_last_error(const hsc_engine* e);
int hsc_b200_abi_version(void);

/* A second handle on the SAME device dictionary (D, Gram tensor, weights, K1 operand): lets several encodes
 * be in flight at once on different streams (chunked host pipelines).  The view does not own the dictionary:
 * re-create views after hsc_b200_set_dictionary on the parent, destroy them before the parent. */
int hsc_b200_create_view(hsc_engine* parent, hsc_engine** out);

/* Dictionary D[K][L][F] (host memory, `dtype` elements), optional selection weights w[K]
 * (hsc/modeling.py:902-906; NULL = none).  Uploads D, builds the shift Gram tensor
 * G[k][tau+L-1][k'] = sum_{j,f} D[k][j+tau][f] * D[k'][j][f] on the device.  Synchronous. */
int hsc_b200_set_dictionary(hsc_engine* e, const void* D_host, int dtype, int64_t K, int64_t L, int64_t F,
                            const void* weights_host);

/* Device pointers of the uploaded dictionary / Gram tensor (for tests), NULL before set_dictionary. */
const void* hsc_b200_dictionary_dev(const hsc_engine* e);
const void* hsc_b200_gram_dev(const hsc_engine* e);

/* convolve1d(x, D, padding='same') for S signals: map_dev[S][T][K] (hsc/modeling.py:149-188, :1077). */
int hsc_b200_correlate(hsc_engine* e, const void* x_dev, int64_t S, int64_t T, void* map_dev, void* stream);

/* Bytes of device workspace hsc_b200_mp_begin needs for S signals of T samples (0 on error). */
size_t hsc_b200_workspace_bytes(const hsc_engine* e, int64_t S, int64_t T);

/* Starts the pursuit of S independent signals x_dev[S][T][F]: residual_dev (may equal x_dev) becomes
 * the running residual and finally the returned residual (:1071); computes the initial correlation
 * map and the argmax hierarchy inside `workspace_dev`.  The workspace and residual must stay alive
 * until the last hsc_b200_mp_run. */
int hsc_b200_mp_begin(hsc_engine* e, const void* x_dev, void* residual_dev, int64_t S, int64_t T,
                      void* workspace_dev, size_t workspace_bytes, const hsc_mp_options* opt, void* stream);

/* Same, for the signals [s_lo, s_lo + s_count) of the S-signal batch only: lets the caller start the
 * correlation of a chunk as soon as its host-to-device copy has landed while later chunks are still in
 * flight.  x_dev / residual_dev / workspace_dev are the FULL-batch pointers; every chunk must be begun (with
 * the same S, T, options) before hsc_b200_mp_run. */
int hsc_b200_mp_begin_part(hsc_engine* e, const void* x_dev, void* residual_dev, int64_t S, int64_t T,
                           void* workspace_dev, size_t workspace_bytes, const hsc_mp_options* opt,
                           int64_t s_lo, int64_t s_count, void* stream);

/* Runs the select/update loop of every unfinished signal until it stops or has written `capacity`
 * events into its slice of the output buffers: ev_pos_dev/ev_idx_dev/ev_coef_dev are
 * [S][capacity] (int32 centre position, int32 filter, `dtype` coefficient), in selection order.
 * If states_host != NULL the call synchronises the stream and copies the S states out; a signal
 * whose status is HSC_PAUSE_* continues on the next call (its n_buffered restarts at 0). */
int hsc_b200_mp_run(hsc_engine* e, int32_t* ev_pos_dev, int32_t* ev_idx_dev, void* ev_coef_dev, int64_t capacity,
                    hsc_signal_state* states_host, void* stream);

/* Copies the S per-signal states of the encode in flight to the host (synchronises the stream). */
int hsc_b200_mp_states(hsc_engine* e, hsc_signal_state* states_host, void* stream);

/* Same copy, enqueued on the stream WITHOUT synchronising (states_host should be pinned). */
int hsc_b200_mp_states_async(hsc_engine* e, hsc_signal_state* states_host, void* stream);

/* Compacts the event buffers after hsc_b200_mp_run: the n_buffered[s] atoms of every signal of the encode in flight, in
 * signal order, into the flat device arrays pos_out/idx_out/coef_out (`out_capacity` atoms each); offsets_dev[S+1]
 * (int64) receives the start of every signal's atoms, offsets_dev[S] the total.  Atoms past out_capacity are dropped:
 * compare offsets[S] with out_capacity.  This is what leaves the device - the device-to-host read of the codes, or the
 * NCCL gather of the sparse codes over the ranks (the reference returns one scipy.sparse matrix per signal,
 * hsc/modeling.py:1180-1186; 12-16 bytes per atom here instead of the padded [S][capacity] slices).  Asynchronous. */
int hsc_b200_mp_compact_events(hsc_engine* e, const int32_t* ev_pos_dev, const int32_t* ev_idx_dev, const void* ev_coef_dev,
                               int64_t capacity, int64_t* offsets_dev, int32_t* pos_out_dev, int32_t* idx_out_dev, void* coef_out_dev,
                               int64_t out_capacity, void* stream);

/* Level hand-off of the hierarchical encoder (hsc/modeling.py:1489: `input = levelCoefficients.todense()`), on the device:
 * the accumulated code of every signal of the encode in flight (events of one (t,k) summed in float64 in selection order,
 * :992; sums with |c| < min_coefficients dropped, :1171-1177; min_coefficients < 0 = keep all) as the dense float64 map
 * dense_dev[S][T][K], which is the next level's K-channel input signal.  Deterministic (no atomics).  Asynchronous. */
int hsc_b200_mp_events_to_dense(hsc_engine* e, const int32_t* ev_pos_dev, const int32_t* ev_idx_dev, const void* ev_coef_dev,
                                int64_t capacity, double min_coefficients, double* dense_dev, void* stream);

/* Pointer to the correlation map of the encode in flight, [S][T][K] (tests / diagnostics). */
const void* hsc_b200_mp_map_dev(const hsc_engine* e);

/* Sparse decoder, reconstructSignal (hsc/modeling.py:226-245): out_dev[T][F] += sum_n c_n D[k_n]
 * centred at t_n, clipped at the ends.  Deterministic (each sample sums its atoms in list order). */
int hsc_b200_decode(hsc_engine* e, const int32_t* pos_dev, const int32_t* idx_dev, const void* coef_dev, int64_t n,
                    int64_t T, void* out_dev, void* stream);

/* The same decoder for S signals of length T in one launch: out_dev[S][T][F] += the reconstruction of every signal.  The
 * atoms of signal s are entries [offsets_dev[s], offsets_dev[s+1]) of the flat device lists pos_dev / idx_dev / coef_dev,
 * sorted by centre position within the signal; offsets_dev[S+1] (int64, non-decreasing, offsets_dev[0] = 0) is the layout
 * hsc_b200_mp_compact_events writes.  Empty segments are legal.  Each sample sums its own signal's atoms in list order in
 * float64, so signal s gets bit for bit what hsc_b200_decode gives for its atoms alone.  hsc_b200_decode is the S = 1
 * case.  HSC_E_INVALID for a NULL pointer, S <= 0 or T outside [1, 2^31); HSC_E_STATE without a dictionary.  Asynchronous. */
int hsc_b200_decode_batch(hsc_engine* e, const int64_t* offsets_dev, const int32_t* pos_dev, const int32_t* idx_dev,
                          const void* coef_dev, int64_t S, int64_t T, void* out_dev, void* stream);

/* Canonical codes from the flat, selection-ordered events hsc_b200_mp_compact_events writes (offsets_dev[S+1], pos_dev,
 * idx_dev, coef_dev in the engine's dtype; the atoms of signal s are [offsets_dev[s], offsets_dev[s+1]), fewer than 2^31 per
 * signal): for every signal, one entry per distinct (t,k), valued at the float64 sum of its events in selection order
 * (:992); a sum that is exactly 0 or below min_coefficients in absolute value (< 0 = keep all) is dropped (:1171-1181).
 * This is the arithmetic of hsc_b200_mp_events_to_dense.  Within a signal the entries are in ascending (t,k) order, the
 * list order hsc_b200_decode_batch reads.  The entries are split into n_bounds + 1 levels (redistribution, :1556-1594):
 * an entry with filter index k goes to the first level j with k < level_bounds_host[j], else to the last level; the bounds
 * are non-negative and non-decreasing (a bound of 0 leaves its level empty), at most 15 of them.  Level j gets
 * out_offsets_dev[j][S+1] (from 0) and its entries at pos / idx / coef [j][capacity] of out_pos_dev / out_idx_dev /
 * out_coef_dev (float64): the layout hsc_b200_decode_batch reads.  `capacity` is the length of the input event arrays and
 * of every level's output arrays; offsets_dev[S] must not exceed it (events past it are not read).  Positions must lie in
 * [0, T) and filter indices in [0, K).  Empty signals are legal.  Deterministic (no atomics on values).  HSC_E_INVALID
 * for a NULL pointer (the event and output arrays may be NULL when capacity = 0), S outside [1, 65535], T or K outside
 * [1, 2^31), capacity < 0 or bad bounds; HSC_E_STATE without a dictionary.  Asynchronous. */
int hsc_b200_canonicalize_codes(hsc_engine* e, const int64_t* offsets_dev, const int32_t* pos_dev, const int32_t* idx_dev,
                                const void* coef_dev, int64_t capacity, int64_t S, int64_t T, int64_t K,
                                const int64_t* level_bounds_host, int64_t n_bounds, double min_coefficients, int64_t* out_offsets_dev,
                                int32_t* out_pos_dev, int32_t* out_idx_dev, double* out_coef_dev, void* stream);

/* Convenience, host buffers end to end (allocates and frees its own device memory, synchronous):
 * x_host[S][T][F] -> residual_host[S][T][F], events [S][capacity], counts_host[S], states_host[S]
 * (either may be NULL).  Returns HSC_E_NOMEM if a signal needs more than `capacity` events. */
int hsc_b200_mp_encode_host(hsc_engine* e, const void* x_host, int64_t S, int64_t T, const hsc_mp_options* opt,
                            int32_t* ev_pos_host, int32_t* ev_idx_host, void* ev_coef_host, int64_t capacity,
                            int64_t* counts_host, void* residual_host, hsc_signal_state* states_host);

/* Dictionary-update stage of the convolutional K-SVD that consumes the MP codes
 * (ConvolutionalDictionaryLearner._train_ksvd, hsc/modeling.py:593-636), float64 like the reference's learner
 * (its dictionary is float64, :321).  The accumulated code of S independent signals of T samples is given
 * grouped by filter: entries [col_ptr_host[k], col_ptr_host[k+1]) belong to filter k, entry i = (signal
 * sig_dev[i], centre position pos_dev[i], filter idx_dev[i] == k, coefficient coef_dev_io[i]); one entry per
 * distinct (signal, position, filter).  Gauss-Seidel over the filters with at least one entry (:598-599):
 * decode without the filter (:602-607), gather the length-L windows centred at its atoms (zero outside the
 * signal, :610-613), new filter = first left singular vector of the window matrix, new coefficients =
 * s0 * first right singular vector (:627-633).  The sign of a singular pair is arbitrary (LAPACK's in the
 * reference); here <new filter, old filter> >= 0.  D_dev_io[K][L][F] and coef_dev_io are updated in place;
 * *alpha_host = ||D_new - D_old||_F (:636).  Synchronous.
 * Window size q = L*F <= 3072, else HSC_E_UNSUPPORTED.  Accuracy of each new filter u, the dominant eigenvector of the
 * window Gram matrix C = W^T W (c = 32, eps = 2^-52, g = 1 - lambda2/lambda1): ||C u - (u'C u) u|| <= c q eps lambda1
 * and u'C u >= lambda1 (1 - c q eps) for every C, a multiple top eigenvalue included; ||u -+ v1|| <= c q eps / g for
 * gaps down to about 2e-9; all-zero windows give e_0.  W^T W is formed unscaled in float64: window entries below about
 * 1e-160 or above 1e154 underflow or overflow. */
int hsc_b200_ksvd_update(hsc_engine* e, void* D_dev_io, int64_t K, int64_t L, int64_t F, const int64_t* col_ptr_host,
                         const int32_t* sig_dev, const int32_t* pos_dev, const int32_t* idx_dev, void* coef_dev_io, int64_t S,
                         int64_t T, double* alpha_host, void* stream);

/* usePCA=True variant of hsc_b200_ksvd_update (hsc/modeling.py:618-625 with pca(), :48-80): when a filter has two or
 * more windows they are mean-centred, the new filter is the first principal component (eigenvector of the largest
 * eigenvalue of the covariance) and the new coefficients are the projections of the CENTRED windows on it; a single
 * window is normalised as it is.  Sticky per engine; the per-filter sweep API below refuses while it is set (the
 * column means would have to be shared between ranks too). */
int hsc_b200_ksvd_set_pca(hsc_engine* e, int use_pca);

/* The same sweep, one filter at a time, for data-parallel learning: each rank holds the code of its own signals,
 * and the only quantity the ranks must share is the q x q window Gram matrix C = W^T W of the filter being updated
 * (q = L*F; SURVEY 8e).  Between hsc_b200_ksvd_filter_gram (removes filter k's local atoms from the running
 * reconstruction, gathers the local windows, writes their Gram matrix to gram_dev - zeros if the rank has none) and
 * hsc_b200_ksvd_filter_finish (first eigenvector of gram_dev -> D[k], local coefficients = projections, atoms put
 * back) the caller all-reduces gram_dev (sum) over the ranks; every rank then derives the same filter.  `skip` = 1
 * leaves D[k] and the coefficients unchanged (no rank has an atom of this filter, hsc/modeling.py:598-599).
 * gram_dev: caller-owned float64 [q][q] device buffer (NULL: internal, single process).  _end returns
 * alpha = ||D_new - D_old||_F, synchronises and frees the sweep. */
typedef struct hsc_ksvd_sweep hsc_ksvd_sweep;
int hsc_b200_ksvd_begin(hsc_engine* e, void* D_dev_io, int64_t K, int64_t L, int64_t F, const int64_t* col_ptr_host,
                        const int32_t* sig_dev, const int32_t* pos_dev, const int32_t* idx_dev, void* coef_dev_io, int64_t S,
                        int64_t T, void* gram_dev, void* stream, hsc_ksvd_sweep** out);
int hsc_b200_ksvd_filter_gram(hsc_ksvd_sweep* sweep, int64_t k, int64_t* n_local);
int hsc_b200_ksvd_filter_finish(hsc_ksvd_sweep* sweep, int64_t k, int skip);
int hsc_b200_ksvd_end(hsc_ksvd_sweep* sweep, double* alpha_host);

/* Assignment step of the convolutional k-means learner (ConvolutionalDictionaryLearner._train_kmean,
 * hsc/modeling.py:455-480), with the centroids set as the dictionary: for each of B training windows
 * x_dev[B][Tw][F] (Tw >= L; the reference uses Tw = 2L, :426) the 'valid' position and the centroid of maximum
 * |correlation| (np.argmax over the flattened [position][filter] scores, first occurrence, :459-460) ->
 * pos_dev[B] (first sample of the patch), idx_dev[B]; sums_dev[K][L][F] (float64, zeroed here) receives the sum
 * of the L2-normalised patches assigned to each centroid and counts_dev[K] their number, so that the cosine mean
 * of :480 is sums / counts.  map_scratch_dev: [B][Tw][K] elements of the engine dtype.  Asynchronous on `stream`. */
int hsc_b200_kmeans_assign(hsc_engine* e, const void* x_dev, int64_t B, int64_t Tw, void* map_scratch_dev, int32_t* pos_dev,
                           int32_t* idx_dev, double* sums_dev, int32_t* counts_dev, void* stream);

/* Synchronous device -> host copy of `bytes` bytes (tests / diagnostics: Gram tensor, map). */
int hsc_b200_copy_to_host(hsc_engine* e, const void* src_dev, void* dst_host, size_t bytes);

/* Number of kernels this engine has launched since creation (bench.py's gpu_launches). */
int64_t hsc_b200_launch_count(const hsc_engine* e);

#ifdef __cplusplus
}
#endif
#endif /* HSC_B200_H_ */
