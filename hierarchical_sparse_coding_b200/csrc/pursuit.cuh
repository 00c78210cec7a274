// K2: persistent select/update kernel of the convolutional matching pursuit -- one CTA per signal,
// looping over atoms until a stop rule fires (ConvolutionalMatchingPursuit.computeCoefficients,
// hsc/modeling.py:1053-1186, with _selectBestAtoms :899-982, _updateResidual :996-1016,
// _updateInnerProducts :1018-1051).
//
// What stays resident in HBM/L2 per signal: the correlation map c[T][K], the residual r[T][F] and a
// three-level argmax hierarchy over the map,
//     level 1  (val1,idx1)[t]   = max_k |c[t][k]*w[k]| and its lowest k
//     level 2  (val2,idx2)[g]   = best row among the G1 rows of group g
//     level 3  (val3,idx3)[h]   = best row among the G2 level-2 groups of h
// so that selecting an atom reads n3 = T/(G1*G2) entries instead of rescanning T*K (the reference
// allocates |scores| and scans it every pass, :967) and applying it rewrites only the 2L-1 rows the
// reference rewrites (:1049), their level-1 keys (fused with the rewrite, warp shuffles) and the
// <= 2 dirty groups of levels 2 and 3.
//
// Local update.  Interior atoms use the shift Gram tensor: c[p+tau][k'] -= coef*G[k][tau][k'].
// Atoms whose 2L-1 window reaches a row whose filter support overhangs the signal take the EDGE path,
// which restates the reference exactly: re-correlate the window from the residual, REFLECT-padded
// where it overhangs (np.pad mode='reflect', :1046) -- the initial map is zero padded (:161-164), so
// those rows change meaning after their first update and a Gram update would not reproduce that.
#pragma once
#include <limits.h>
#include "common.cuh"

namespace hsc {

template <typename real>
struct MpArgs {
    int T, K, L, F, off;  // T: row stride of every [S][T][...] array, and the length of every signal unless `len` is set
    int G1, n2, G2, n3;
    const real* D;        // [K][L][F]
    const real* G;        // [K][2L-1][K]
    const real* w;        // [K] or nullptr
    real* map;            // [S][T][K]
    real* resid;          // [S][T][F]
    real* val1; int* idx1;    // [S][T]
    real* val2; int* idx2;    // [S][n2]
    real* val3; int* idx3;    // [S][n3]
    unsigned* bitmap;     // [S][bitmap_words]
    long long bitmap_words;
    hsc_signal_state* state;  // [S]
    int* ev_pos; int* ev_idx; real* ev_coef;   // [S][cap]
    long long cap;
    long long max_nnz;        // < 0: none
    real tol_snr; int has_snr;
    real tol_scale; int has_scale;
    real null_thres;          // < 0: none
    real eps;
    int coef_mode;
    long long max_passes;     // <= 0: unlimited
    long long max_events_total;
    int nb_blocks;            // 1 = global argmax per pass; > 1 or -1 ('auto') = block-wise selection (:908-963)
    int ncand_max;            // capacity of the per-signal candidate lists
    int* cand_t; int* cand_k; real* cand_c;       // [S][2][ncand_max] candidate lists (unsorted | sorted)
    double* locomp_scratch;   // LoCOMP: [S][256*257] normal matrices of refit groups too large for shared memory
    real* edge_ext;           // [S][edge_stride] scratch: reflect-padded residual slice of the edge atom being applied
    long long edge_stride;
    int prefetch;             // 1: bulk-prefetch the selected atom's map window + Gram slice into L2 at selection
    int tma_rows, tma_stages; // interior map update through shared memory with bulk copies: rows per stage, stages (0 = off)
    int tma_bytes;            // bytes of the stage rings at the start of dynamic shared memory (the SMH keys follow)
    long long* prof;          // [S][8] phase cycle counters (HSC_PROFILE_PHASES builds), else nullptr
    int scalar_window;        // 1: register window path without the 16-byte vector variants (narrow maps)
    int row32;                // 1: wide rows (32 lanes per row) take the lean window loop gram_update_row32
    int next_prefetch;        // 1: the watch warp pulls the likely next pick's residual / map row / keys towards L2
    int early_issue;          // 1: the first window chunks of an interior atom are issued right after the pick (bulk-copy path)
    float rerank_tol;         // float maps: candidates within rerank_tol * (best score + largest initial score) of the best
                              // approximate score are re-scored from the residual before the pick (0 = off)
    const int* len;           // [S] per-signal lengths in [1, T] (hsc_b200_mp_begin_lengths), or nullptr: all signals have T samples
};

// Length of the signal of this CTA (one CTA per signal).  Every BOUND of the pursuit - edge and overhang tests, window
// and residual clipping, group and block ranges, the energy and residual-scale scans - uses it; a.T stays the stride.
// Samples and map rows at or past it are never read: a ragged batch encodes each signal as if it were alone.
// RAGGED is a compile-time choice of every kernel and helper that bounds with it: a uniform launch compiles to a.T alone.
template <bool RAGGED, typename real>
__device__ __forceinline__ int signal_length(const MpArgs<real>& a) { return RAGGED ? __ldg(a.len + blockIdx.x) : a.T; }

// Packed keys of the shared-memory argmax hierarchy (float scores, pursuit_kernel<..., SMH = true>): the score's
// bit pattern (non-negative floats order like unsigned integers) above ~(row_in_group*K + filter), so that an
// unsigned 64-bit max picks the largest score and, among equal scores, the lowest row, which is np.argmax's
// first-occurrence rule on the row-major map (:967).  A zero score packs to 0 = "no candidate".
__device__ __forceinline__ unsigned long long pack_key(float v, int row_local, int k, int K) {
    const unsigned vb = __float_as_uint(v);
    return vb == 0u ? 0ull : (((unsigned long long)vb << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)(row_local * K + k)));
}
__device__ __forceinline__ unsigned long long pack_key(double, int, int, int) { return 0ull; }    // SMH is float-only

__device__ __forceinline__ unsigned lds_u32(uint32_t saddr) {
    unsigned v;
    asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(saddr));      // not volatile: scans pipeline their loads
    return v;
}

__device__ __forceinline__ unsigned long long warp_max_u64(unsigned long long key) {
    const unsigned hi = (unsigned)(key >> 32);
    const unsigned mx = __reduce_max_sync(0xffffffffu, hi);
    const unsigned lo = hi == mx ? (unsigned)key : 0u;
    const unsigned ml = __reduce_max_sync(0xffffffffu, lo);
    return ((unsigned long long)mx << 32) | ml;
}

// Level-1 keys of rows [row_lo, row_hi] recomputed from the map (g lanes per row).
template <typename real>
__device__ void rekey_rows(const MpArgs<real>& a, const real* map_s, real* v1, int* i1, int row_lo, int row_hi,
                           int g, int nthreads, unsigned long long* dirty = nullptr, int glo = 0, int g1s = 0) {
    const int ngroups = nthreads / g;
    const int grp = threadIdx.x / g, lig = threadIdx.x % g;
    const int nrows = row_hi - row_lo + 1;
    constexpr int R = 4;                        // rows in flight per lane group: independent L2 loads
    for (int base = 0; base < nrows; base += ngroups * R) {
        real bv[R];
        int bi[R];
#pragma unroll
        for (int r = 0; r < R; ++r) { bv[r] = (real)0; bi[r] = INT_MAX; }
        for (int kk = lig; kk < a.K; kk += g) {
            real m[R];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const int rl = base + r * ngroups + grp;
                // L2-coherent: bulk-copy stores of the map do not update L1
                m[r] = rl < nrows ? __ldcg(map_s + (long long)(row_lo + rl) * a.K + kk) : (real)0;
            }
            const real wk = a.w ? a.w[kk] : (real)1;
#pragma unroll
            for (int r = 0; r < R; ++r) take_first_max(bv[r], bi[r], rabs<real>(a.w ? m[r] * wk : m[r]), kk);
        }
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int rl = base + r * ngroups + grp;
            const bool valid = rl < nrows;
            const int row = row_lo + rl;
            group_argmax(bv[r], bi[r], g);
            if (valid && lig == 0) {
                v1[row] = bv[r];
                i1[row] = bi[r];
                if (dirty) {                   // shared-memory hierarchy: fold the row into its level-2 group
                    const unsigned long long key = pack_key(bv[r], row & ((1 << g1s) - 1), bi[r], a.K);
                    if (key) atomicMax(&dirty[(row >> g1s) - glo], key);
                }
            }
        }
    }
}

// One warp per destination group: best (value, row) among `gsize` source entries.
// src_idx == nullptr means the source entry's own position is its row (level 1 -> 2).
template <typename real>
__device__ void rekey_level(const real* src_val, const int* src_idx, int nsrc, real* dst_val, int* dst_idx,
                            int group_lo, int group_hi, int gsize, int nthreads) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = nthreads >> 5;
    for (int gi = group_lo + warp; gi <= group_hi; gi += nwarps) {
        const int e0 = gi * gsize;
        const int e1 = min(e0 + gsize, nsrc);
        real bv = (real)0;
        int bi = INT_MAX;
        for (int e = e0 + lane; e < e1; e += 32) take_first_max(bv, bi, src_val[e], src_idx ? src_idx[e] : e);
        group_argmax(bv, bi, 32);
        if (lane == 0) {
            dst_val[gi] = bv;
            dst_idx[gi] = bi;
        }
    }
}

template <typename real> struct VecOf;
template <> struct VecOf<float> { using type = float4; static constexpr int N = 4; };
template <> struct VecOf<double> { using type = double2; static constexpr int N = 2; };
__device__ __forceinline__ void unpack(const float4& v, float* o) { o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w; }
__device__ __forceinline__ void unpack(const double2& v, double* o) { o[0] = v.x; o[1] = v.y; }
__device__ __forceinline__ float4 pack(const float* o, float4) { return make_float4(o[0], o[1], o[2], o[3]); }
__device__ __forceinline__ double2 pack(const double* o, double2) { return make_double2(o[0], o[1]); }

// Level-1 keys of the whole map after K1, at full-GPU parallelism (the per-signal CTA of the pursuit
// kernel would otherwise walk its 64 MB map alone): g lanes per row, 4 rows in flight per group,
// 16-byte streaming loads.  Grid: (ceil(T / rows_per_cta), S).
template <typename real>
__global__ void __launch_bounds__(256) rowkey_kernel(const real* __restrict__ map, const real* __restrict__ wts,
                                                     real* __restrict__ val1, int* __restrict__ idx1, int T, int K,
                                                     int rows_per_cta) {
    using V = typename VecOf<real>::type;
    constexpr int VN = VecOf<real>::N;
    const long long s = blockIdx.y;
    const real* map_s = map + s * (long long)T * K;
    real* v1 = val1 + s * (long long)T;
    int* i1 = idx1 + s * (long long)T;
    const int row0 = blockIdx.x * rows_per_cta;
    const int row1 = min(row0 + rows_per_cta, T);
    const bool vec = (K % VN) == 0;
    const int nvec = vec ? K / VN : K;
    const int g = min(32, pow2_at_least(nvec));
    const int ngroups = 256 / g;
    const int grp = threadIdx.x / g, lig = threadIdx.x % g;
    constexpr int R = 4;
    for (int base = row0; base < row1; base += ngroups * R) {
        real bv[R];
        int bi[R];
#pragma unroll
        for (int r = 0; r < R; ++r) { bv[r] = (real)0; bi[r] = INT_MAX; }
        for (int v = lig; v < nvec; v += g) {
            if (vec) {
                V m[R];
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const int row = base + r * ngroups + grp;
                    if (row < row1) m[r] = __ldcs(reinterpret_cast<const V*>(map_s + (long long)row * K) + v);
                }
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const int row = base + r * ngroups + grp;
                    if (row < row1) {
                        real pm[VN];
                        unpack(m[r], pm);
#pragma unroll
                        for (int c = 0; c < VN; ++c) {
                            const int kk = v * VN + c;
                            take_first_max(bv[r], bi[r], rabs<real>(wts ? pm[c] * wts[kk] : pm[c]), kk);
                        }
                    }
                }
            } else {
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const int row = base + r * ngroups + grp;
                    if (row < row1) {
                        const real m = map_s[(long long)row * K + v];
                        take_first_max(bv[r], bi[r], rabs<real>(wts ? m * wts[v] : m), v);
                    }
                }
            }
        }
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int row = base + r * ngroups + grp;
            group_argmax(bv[r], bi[r], g);
            if (row < row1 && lig == 0) {
                v1[row] = bv[r];
                i1[row] = bi[r];
            }
        }
    }
}

// The signal length of a CTA inside a kernel: a ragged launch keeps it in a shared-memory slot that is re-read at every
// use (never a live register of the persistent loops); a uniform launch uses its own value.  Only the ragged
// specialization declares the slot - a shared variable in the uniform kernels changes their register allocation.
template <bool RAGGED> struct CtaLength {
    static __device__ __forceinline__ void set(int) {}
    static __device__ __forceinline__ int get(int uniform) { return uniform; }
};
template <> struct CtaLength<true> {
    static __device__ __forceinline__ volatile int* slot() { __shared__ int len; return &len; }
    static __device__ __forceinline__ void set(int v) { *slot() = v; }
    static __device__ __forceinline__ int get(int) { return *slot(); }
};

// Ragged batches (hsc_b200_mp_begin_lengths).  Before K1: samples [len[s], T) of signal s's residual <- 0, so that K1, which
// then reads the residual, sees each signal followed by the 'same' zero padding of a signal of len[s] samples
// (hsc/modeling.py:161-164): map rows below len[s], the per-signal scale of the tensor-core path and the signal energy are
// those of the signal alone, whatever the padding held.  Grid: (x, S).
template <typename real>
__global__ void __launch_bounds__(256) zero_signal_tails_kernel(real* __restrict__ x, const int* __restrict__ len, int T, int F) {
    const long long s = blockIdx.y;
    const long long n = (long long)T * F;
    real* xs = x + s * n;
    for (long long i = (long long)len[s] * F + blockIdx.x * 256ll + threadIdx.x; i < n; i += (long long)gridDim.x * 256)
        xs[i] = (real)0;
}

// ... and after K1: the level-1 keys of rows [len[s], T) <- "no candidate", so that no selection can reach them.
template <typename real>
__global__ void __launch_bounds__(256) clear_tail_keys_kernel(real* __restrict__ val1, int* __restrict__ idx1, const int* __restrict__ len,
                                                              int T) {
    const long long s = blockIdx.y;
    for (long long r = len[s] + blockIdx.x * 256ll + threadIdx.x; r < T; r += (long long)gridDim.x * 256) {
        val1[s * T + r] = (real)0;
        idx1[s * T + r] = 0;
    }
}

// Interior-atom map update, vectorised: c[p+tau][:] -= coef*G[k][tau][:] for the 2L-1 rows of the
// window, 16-byte accesses, g lanes per row, PV vectors per lane per row and R = VIF/PV rows in flight
// per lane, so that every load of a batch is issued before the first store (the map is streamed
// with evict-first loads/stores, the Gram slice goes through the read-only path and stays in L2).
// The level-1 key of each rewritten row is reduced in registers + shuffles and stored with it.
template <typename real, int PV, int NT, int VIF, bool HAS_W>
__device__ __forceinline__ void gram_update_vec(const int K, const int L, const real* __restrict__ wts, real* __restrict__ map_s,
                                                const real* __restrict__ Gk, real* __restrict__ v1, int* __restrict__ i1,
                                                int t, real coef, int g) {
    using V = typename VecOf<real>::type;
    constexpr int VN = VecOf<real>::N;
    constexpr int R = PV >= VIF ? 1 : VIF / PV;
    const int W = 2 * L - 1;
    const int nvec = K / VN;
    const int rows_per_iter = NT / g;
    const int grp = threadIdx.x / g, lig = threadIdx.x % g;
    const real ncoef = -coef;
    // pointers walk down the window by a constant stride: no per-row address arithmetic in the loop
    const long long row_stride = (long long)rows_per_iter * nvec;            // in vectors
    V* mp = reinterpret_cast<V*>(map_s + (long long)(t - (L - 1) + grp) * K) + lig;
    const V* gp = reinterpret_cast<const V*>(Gk + (long long)grp * K) + lig;
    real* v1p = v1 + (t - (L - 1) + grp);
    int* i1p = i1 + (t - (L - 1) + grp);
    bool lane_has[PV];
#pragma unroll
    for (int p = 0; p < PV; ++p) lane_has[p] = (lig + p * g) < nvec;
#pragma unroll 1
    for (int i0 = grp; i0 < W + grp; i0 += rows_per_iter * R) {      // uniform trip count across the CTA
        V m[R][PV], gg[R][PV];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const bool valid = (i0 + r * rows_per_iter) < W;
#pragma unroll
            for (int p = 0; p < PV; ++p) {
                if (valid && lane_has[p]) {
                    m[r][p] = __ldcs(mp + r * row_stride + p * g);
                    gg[r][p] = __ldg(gp + r * row_stride + p * g);
                }
            }
        }
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const bool valid = (i0 + r * rows_per_iter) < W;
            real bv = (real)0;
            int bi = INT_MAX;
#pragma unroll
            for (int p = 0; p < PV; ++p) {
                if (valid && lane_has[p]) {
                    real pm[VN], pg[VN];
                    unpack(m[r][p], pm);
                    unpack(gg[r][p], pg);
                    const int k0 = (lig + p * g) * VN;
#pragma unroll
                    for (int c = 0; c < VN; ++c) {
                        pm[c] = fma(ncoef, pg[c], pm[c]);
                        const real sc = rabs<real>(HAS_W ? pm[c] * wts[k0 + c] : pm[c]);
                        take_first_max(bv, bi, sc, k0 + c);
                    }
                    __stcs(mp + r * row_stride + p * g, pack(pm, V()));
                }
            }
            group_argmax(bv, bi, g);
            if (valid && lig == 0) {
                v1p[r * rows_per_iter] = bv;
                i1p[r * rows_per_iter] = bi;
            }
        }
        mp += R * row_stride;
        gp += R * row_stride;
        v1p += R * rows_per_iter;
        i1p += R * rows_per_iter;
    }
}

// The first NS chunks of every warp's window pipeline (gram_update_tma), issued by lane 0 of each warp as soon as the atom
// is picked: the bulk copies of the map rows and Gram rows then fly while the CTA does its bookkeeping and the residual
// update, instead of starting after them.  Same chunk geometry as gram_update_tma (which is then called with preissued).
template <typename real, int NT, int RPS>
__device__ __noinline__ void gram_window_issue(const int K, const int L, real* map_s, const real* Gk, int t, int g,
                                                  unsigned char* smem, unsigned long long* bars, int NS) {
    constexpr int NW = NT / 32;
    if ((threadIdx.x & 31) != 0) return;
    const int warp = threadIdx.x >> 5;
    const int W = 2 * L - 1;
    const int crows = (32 / g) * RPS;
    const uint32_t row_bytes = (uint32_t)(K * sizeof(real));
    const uint32_t half_bytes = (uint32_t)crows * row_bytes;
    const uint32_t stage_bytes = 2u * half_bytes;
    const uint32_t wsm_u = smem_addr_u32(smem + (size_t)warp * NS * stage_bytes);
    const uint32_t bar_u = smem_addr_u32(bars + warp * NS);
    const int first = warp * crows;
    const int stride_rows = NW * crows;
    const int nsteps = first < W ? (W - first + stride_rows - 1) / stride_rows : 0;
    const long long gstep = (long long)stride_rows * K;
    real* gmap = map_s + (long long)(t - (L - 1) + first) * K;
    const real* ggram = Gk + (long long)first * K;
    for (int j = 0; j < NS && j < nsteps; ++j) {
        const uint32_t bytes = (uint32_t)min(crows, W - first - j * stride_rows) * row_bytes;
        const uint32_t bar = bar_u + 8u * (uint32_t)j;
        const uint32_t dst = wsm_u + (uint32_t)j * stage_bytes;
        mbarrier_expect_tx(bar, 2u * bytes);
        bulk_load_g2s(dst, gmap + j * gstep, bytes, bar);
        bulk_load_g2s(dst + half_bytes, ggram + j * gstep, bytes, bar);
    }
}

// Interior-atom map update staged through shared memory, one independent pipeline per warp.
// The 2L-1 window rows are dealt to the warps in chunks of crows = RPS*32/g consecutive rows (g lanes per row, RPS
// rows per lane group); warp w owns chunks w, w+NW, w+2NW, ...  For each chunk, lane 0 pulls the map rows and the
// matching Gram rows into the warp's stage ring with two bulk asynchronous copies (completion on the stage's
// mbarrier), the warp applies c -= coef*G from shared memory, reduces the level-1 key of each row, and lane 0 sends
// the rewritten rows back with one bulk store.  No CTA-wide barrier inside the window and no registers held by loads
// in flight.  The kernel is ISSUE-bound in this loop (ncu: 87% of its instructions), so everything that does not
// depend on the step is hoisted and RPS = 2 halves the number of steps (and with it the per-step control code).
template <typename real, int NT, bool HAS_W, bool SMH, int RPS>
__device__ __noinline__ unsigned gram_update_tma(const int K, const int L, const real* __restrict__ wts, real* map_s,
                                                 const real* Gk, real* __restrict__ v1, int* __restrict__ i1, int t, real coef,
                                                 int g, unsigned char* smem, unsigned long long* bars, int NS, unsigned phase,
                                                 unsigned long long* dirty, int glo, int g1s, bool preissued = false) {
    using V = typename VecOf<real>::type;
    constexpr int VN = VecOf<real>::N;
    constexpr int NW = NT / 32;
    const int lane = threadIdx.x & 31;
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);     // provably warp-uniform: stays in uniform registers
    const int W = 2 * L - 1;
    const int nvec = K / VN;
    const int rpw = 32 / g;                          // lane groups per warp
    const int crows = rpw * RPS;                     // rows per chunk
    const int rr = lane / g, lig = lane % g;
    const real ncoef = -coef;
    const uint32_t row_bytes = (uint32_t)(K * sizeof(real));
    const uint32_t half_bytes = (uint32_t)crows * row_bytes;        // map part of a stage; the Gram part follows
    const uint32_t stage_bytes = 2u * half_bytes;
    unsigned char* wsm = smem + (size_t)warp * NS * stage_bytes;
    const uint32_t wsm_u = smem_addr_u32(wsm);
    const uint32_t bar_u = smem_addr_u32(bars + warp * NS);
    const int first = warp * crows;
    const int stride_rows = NW * crows;
    const int nsteps = first < W ? (W - first + stride_rows - 1) / stride_rows : 0;
    const long long gstep = (long long)stride_rows * K;             // elements between this warp's consecutive chunks
    real* gmap = map_s + (long long)(t - (L - 1) + first) * K;
    const real* ggram = Gk + (long long)first * K;
    const int trow0 = t - (L - 1) + first;

    auto load_chunk = [&](int j, int s) {
        const uint32_t bytes = (uint32_t)min(crows, W - first - j * stride_rows) * row_bytes;
        const uint32_t bar = bar_u + 8u * (uint32_t)s;
        const uint32_t dst = wsm_u + (uint32_t)s * stage_bytes;
        mbarrier_expect_tx(bar, 2u * bytes);
        bulk_load_g2s(dst, gmap + j * gstep, bytes, bar);
        bulk_load_g2s(dst + half_bytes, ggram + j * gstep, bytes, bar);
    };
    if (lane == 0 && !preissued)           // (issued right after the pick already: gram_window_issue)
        for (int j = 0; j < NS && j < nsteps; ++j) load_chunk(j, j);
    int s = 0;
    int cur_g = -1;                        // SMH, g == 32: running best key of the current level-2 group
    unsigned long long cur_key = 0ull;
#pragma unroll 1
    for (int j = 0; j < nsteps; ++j) {
        mbarrier_wait_parity(bar_u + 8u * (uint32_t)s, (phase >> s) & 1u);
        phase ^= 1u << s;
        const int rows = min(crows, W - first - j * stride_rows);
        unsigned char* stg = wsm + (size_t)s * stage_bytes;
#pragma unroll
        for (int q = 0; q < RPS; ++q) {
            const int r = rr + q * rpw;                             // row of the chunk this lane group works on
            V* mrow = reinterpret_cast<V*>(stg) + (size_t)r * nvec;
            const V* grow = reinterpret_cast<const V*>(stg + half_bytes) + (size_t)r * nvec;
            const bool valid = r < rows;
            real bv = (real)0;
            int bi = INT_MAX;
            if (valid) {
                for (int v = lig; v < nvec; v += g) {
                    real pm[VN], pg[VN];
                    unpack(mrow[v], pm);
                    unpack(grow[v], pg);
#pragma unroll
                    for (int c = 0; c < VN; ++c) {
                        pm[c] = fma(ncoef, pg[c], pm[c]);
                        const real sc = rabs<real>(HAS_W ? pm[c] * wts[v * VN + c] : pm[c]);
                        take_first_max(bv, bi, sc, v * VN + c);
                    }
                    mrow[v] = pack(pm, V());
                }
            }
            group_argmax(bv, bi, g);
            const int trow = trow0 + j * stride_rows + r;
            if (valid && lig == 0) {
                v1[trow] = bv;
                i1[trow] = bi;
            }
            if constexpr (SMH) {
                const unsigned long long key = valid ? pack_key(bv, trow & ((1 << g1s) - 1), bi, K) : 0ull;
                if (g == 32) {             // the warp's rows come in increasing order: flush when the group changes
                    const int gg = trow >> g1s;
                    if (gg != cur_g) {
                        if (lane == 0 && cur_key) atomicMax(&dirty[cur_g - glo], cur_key);
                        cur_g = gg;
                        cur_key = 0ull;
                    }
                    cur_key = key > cur_key ? key : cur_key;
                } else if (lig == 0 && key) {
                    atomicMax(&dirty[(trow >> g1s) - glo], key);
                }
            }
        }
        fence_proxy_async_smem();          // this warp's generic-proxy writes of the stage -> visible to the bulk store
        __syncwarp();
        if (lane == 0) {
            bulk_store_s2g(gmap + j * gstep, wsm_u + (uint32_t)s * stage_bytes, (uint32_t)rows * row_bytes);
            bulk_commit();
            if (j + NS < nsteps) {
                bulk_wait_read_all();      // the store has read the stage: it can be refilled
                load_chunk(j + NS, s);
            }
        }
        s = (s + 1 == NS) ? 0 : s + 1;
    }
    if constexpr (SMH) {
        if (g == 32 && lane == 0 && cur_key) atomicMax(&dirty[cur_g - glo], cur_key);
    }
    return phase;
}

// gram_update_tma for the wide-dictionary shape (g == 32 lanes per row, one row per chunk, no filter weights, first chunks
// already in flight): the same pipeline with everything that is uniform across the warp - the atom, the running global
// addresses, the stage ring - kept provably uniform, the copies issued under elect.sync, and nothing recomputed per row.
// The window loop is where the kernel issues ~80% of its instructions (ncu source page), so its length per row is what the
// step time follows once the rows stream at HBM rate.
template <typename real, int NT, bool SMH>
__device__ __noinline__ unsigned gram_update_row32(const int K, const int L, real* map_s, const real* Gk_in, real* __restrict__ v1,
                                                   int* __restrict__ i1, int t_in, real coef, unsigned char* smem,
                                                   unsigned long long* bars, int NS, unsigned phase, unsigned long long* dirty,
                                                   int glo, int g1s) {
    using V = typename VecOf<real>::type;
    constexpr int VN = VecOf<real>::N;
    constexpr int NW = NT / 32;
    const int lane = threadIdx.x & 31;
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
    const int t = __shfl_sync(0xffffffffu, t_in, 0);
    const real* Gk = reinterpret_cast<const real*>(__shfl_sync(0xffffffffu, reinterpret_cast<unsigned long long>(Gk_in), 0));
    const int W = 2 * L - 1;
    const int nvec = K / VN;
    const real ncoef = -coef;
    const uint32_t row_bytes = (uint32_t)(K * sizeof(real));
    const uint32_t stage_bytes = 2u * row_bytes;                    // map row, then the Gram row
    unsigned char* wsm = smem + (size_t)warp * NS * stage_bytes;
    const uint32_t wsm_u = smem_addr_u32(wsm);
    const uint32_t bar_u = smem_addr_u32(bars + warp * NS);
    const int nsteps = warp < W ? (W - warp + NW - 1) / NW : 0;
    const long long gstep = (long long)NW * K;                      // elements between this warp's consecutive rows
    const long long ahead = (long long)NS * gstep;                  // ... and to the row that refills the stage
    real* gmap = map_s + (long long)(t - (L - 1) + warp) * K;       // the row in hand
    const real* ggram = Gk + (long long)warp * K;
    int trow = t - (L - 1) + warp;
    int s = 0;
    int cur_g = -1;
    unsigned long long cur_key = 0ull;
#pragma unroll 1
    for (int j = 0; j < nsteps; ++j) {
        const uint32_t bar = bar_u + 8u * (uint32_t)s;
        mbarrier_wait_parity(bar, (phase >> s) & 1u);
        phase ^= 1u << s;
        unsigned char* stg = wsm + (size_t)s * stage_bytes;
        V* mrow = reinterpret_cast<V*>(stg);
        const V* grow = reinterpret_cast<const V*>(stg + row_bytes);
        real bv = (real)0;
        int bi = INT_MAX;
#pragma unroll 2
        for (int v = lane; v < nvec; v += 32) {
            real pm[VN], pg[VN];
            unpack(mrow[v], pm);
            unpack(grow[v], pg);
#pragma unroll
            for (int c = 0; c < VN; ++c) {
                pm[c] = fma(ncoef, pg[c], pm[c]);
                take_first_max(bv, bi, rabs<real>(pm[c]), v * VN + c);
            }
            mrow[v] = pack(pm, V());
        }
        fence_proxy_async_smem();          // this warp's generic-proxy writes of the stage -> visible to the bulk store
        __syncwarp();
        if (elect_one_sync()) {
            bulk_store_s2g(gmap, wsm_u + (uint32_t)s * stage_bytes, row_bytes);
            bulk_commit();
            if (j + NS < nsteps) {
                bulk_wait_read_all();      // the store has read the stage: it can be refilled
                mbarrier_expect_tx(bar, stage_bytes);
                bulk_load_g2s(wsm_u + (uint32_t)s * stage_bytes, gmap + ahead, row_bytes, bar);
                bulk_load_g2s(wsm_u + (uint32_t)s * stage_bytes + row_bytes, ggram + ahead, row_bytes, bar);
            }
        }
        group_argmax(bv, bi, 32);
        if (lane == 0) {
            v1[trow] = bv;
            i1[trow] = bi;
        }
        if constexpr (SMH) {               // the warp's rows come in increasing order: flush when the level-2 group changes
            const unsigned long long key = pack_key(bv, trow & ((1 << g1s) - 1), bi, K);
            const int gg = trow >> g1s;
            if (gg != cur_g) {
                if (lane == 0 && cur_key) atomicMax(&dirty[cur_g - glo], cur_key);
                cur_g = gg;
                cur_key = 0ull;
            }
            cur_key = key > cur_key ? key : cur_key;
        }
        gmap += gstep;
        ggram += gstep;
        trow += NW;
        s = (s + 1 == NS) ? 0 : s + 1;
    }
    if constexpr (SMH) {
        if (lane == 0 && cur_key) atomicMax(&dirty[cur_g - glo], cur_key);
    }
    return phase;
}

// Edge path: rows [ra, rb] of the map <- correlation of every filter with the residual slice, reflect-padded where a
// filter's support leaves it (np.pad(mode='reflect') + convolve1d 'valid', hsc/modeling.py:1046-1047).  `ext` holds the
// padded slice materialised once per edge atom (ext[0] = first tap of row ext_row0), so that a row's L*F taps are
// contiguous and the correlation is a plain dot product.  One filter per thread, R rows at a time; the filter is
// read in batches of 8 independent loads (it streams from L2: dependent scalar loads made an edge atom cost ~1 ms),
// the slice values are warp-wide broadcasts out of L1.  Accumulation: taps ascending in float64, independent of the
// work split.
template <typename real, int NT>
__device__ __noinline__ void edge_recorrelate(const MpArgs<real>& a, real* map_s, const real* ext, int ext_row0, int ra, int rb) {
    const int K = a.K, F = a.F, LF = a.L * a.F;
    constexpr int R = 8, U = 8;
    constexpr int KPT = NT <= 128 ? 2 : 1;       // filters per thread in flight (the 4-warp launch shape has the registers)
    const int kt = K < NT ? K : NT;              // threads per row chunk
    const int ngroups = NT / kt;
    const int grp = threadIdx.x / kt;
    if (grp >= ngroups) return;
    const int nchunks = (rb - ra + 1 + R - 1) / R;
    for (int kk = threadIdx.x - grp * kt; kk < K; kk += KPT * kt) {
        const real* dd[KPT];
#pragma unroll
        for (int p = 0; p < KPT; ++p) dd[p] = a.D + (long long)min(kk + p * kt, K - 1) * LF;   // a filter past K repeats the last one (not stored)
        for (int c = grp; c < nchunks; c += ngroups) {
            const int r0 = ra + c * R;
            const real* e0 = ext + (long long)(r0 - ext_row0) * F;
            int roff[R];                                               // rows past rb repeat the last one (not stored)
#pragma unroll
            for (int r = 0; r < R; ++r) roff[r] = (min(r0 + r, rb) - r0) * F;
            double acc[KPT][R];
#pragma unroll
            for (int p = 0; p < KPT; ++p)
#pragma unroll
                for (int r = 0; r < R; ++r) acc[p][r] = 0.0;
            for (int q0 = 0; q0 < LF; q0 += U) {
                real dv[KPT][U];
#pragma unroll
                for (int p = 0; p < KPT; ++p)
#pragma unroll
                    for (int u = 0; u < U; ++u) dv[p][u] = (q0 + u < LF) ? dd[p][q0 + u] : (real)0;
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    if (q0 + u < LF) {
#pragma unroll
                        for (int r = 0; r < R; ++r) {
                            const double ev = (double)e0[roff[r] + q0 + u];
#pragma unroll
                            for (int p = 0; p < KPT; ++p) acc[p][r] = fma(ev, (double)dv[p][u], acc[p][r]);
                        }
                    }
                }
            }
#pragma unroll
            for (int p = 0; p < KPT; ++p)
#pragma unroll
                for (int r = 0; r < R; ++r)
                    if (r0 + r <= rb && kk + p * kt < K) map_s[(long long)(r0 + r) * K + kk + p * kt] = (real)acc[p][r];
        }
    }
}

// The same re-correlation for float maps whose channel count is a compile-time 1, 2, 4 or 8 and whose filters are a
// multiple of 8 taps long, with the padded slice in SHARED memory: a step covers R = 8 rows x U = 8 taps, whose
// (R-1)*F + U distinct slice values are loaded once (128-bit shared loads) instead of once per (row, tap), and the filter
// taps come as 128-bit loads.  Same accumulation order (taps ascending, float64) - bit-identical to edge_recorrelate,
// 2.3x faster on the config-4 shape (tools/edge_probe.cu variant F, profiles/r1e_edge_probe.txt).  `ext` must be readable
// (finite values) for R*F + U floats past the last row's slice.
template <int NT, int F>
__device__ __noinline__ void edge_recorrelate_win(const MpArgs<float>& a, float* map_s, const float* ext, int ext_row0, int ra, int rb) {
    const int K = a.K, LF = a.L * F;
    constexpr int R = 8, U = 8;
    constexpr int WN = (R - 1) * F + U;            // multiple of 4 for F in {1,2,4,8}... F=1: 15 -> padded to 16 below
    constexpr int WN4 = (WN + 3) / 4;
    const int kt = K < NT ? K : NT;
    const int ngroups = NT / kt;
    const int grp = threadIdx.x / kt;
    if (grp >= ngroups) return;
    const int nchunks = (rb - ra + 1 + R - 1) / R;
    for (int kk = threadIdx.x - grp * kt; kk < K; kk += kt) {
        const float4* dd = reinterpret_cast<const float4*>(a.D + (long long)kk * LF);
        for (int c = grp; c < nchunks; c += ngroups) {
            const int r0 = ra + c * R;
            const float* e0 = ext + (long long)(r0 - ext_row0) * F;
            double acc[R];
#pragma unroll
            for (int r = 0; r < R; ++r) acc[r] = 0.0;
            for (int q0 = 0; q0 < LF; q0 += U) {
                float dv[U], ew[WN4 * 4];
#pragma unroll
                for (int u = 0; u < U / 4; ++u) {
                    const float4 v = __ldg(dd + q0 / 4 + u);
                    dv[4 * u] = v.x; dv[4 * u + 1] = v.y; dv[4 * u + 2] = v.z; dv[4 * u + 3] = v.w;
                }
#pragma unroll
                for (int i = 0; i < WN4; ++i) {
                    ew[4 * i] = e0[q0 + 4 * i]; ew[4 * i + 1] = e0[q0 + 4 * i + 1]; ew[4 * i + 2] = e0[q0 + 4 * i + 2]; ew[4 * i + 3] = e0[q0 + 4 * i + 3];
                }
#pragma unroll
                for (int u = 0; u < U; ++u)
#pragma unroll
                    for (int r = 0; r < R; ++r) acc[r] = fma((double)ew[r * F + u], (double)dv[u], acc[r]);
            }
#pragma unroll
            for (int r = 0; r < R; ++r)
                if (r0 + r <= rb) map_s[(long long)(r0 + r) * K + kk] = (float)acc[r];
        }
    }
}

// Dispatch: the window variant where it applies (float, F in {1,2,4,8}, L*F a multiple of 8, slice in shared memory).
template <typename real, int NT>
__device__ __noinline__ void edge_recorrelate_any(const MpArgs<real>& a, real* map_s, const real* ext, bool ext_in_smem, int ext_row0, int ra, int rb) {
    if constexpr (sizeof(real) == 4) {
        if (ext_in_smem && (a.L * a.F) % 8 == 0) {
            const MpArgs<float>& af = reinterpret_cast<const MpArgs<float>&>(a);
            float* mf = reinterpret_cast<float*>(map_s);
            const float* ef = reinterpret_cast<const float*>(ext);
            switch (a.F) {
                case 1: edge_recorrelate_win<NT, 1>(af, mf, ef, ext_row0, ra, rb); return;
                case 2: edge_recorrelate_win<NT, 2>(af, mf, ef, ext_row0, ra, rb); return;
                case 4: edge_recorrelate_win<NT, 4>(af, mf, ef, ext_row0, ra, rb); return;
                case 8: edge_recorrelate_win<NT, 8>(af, mf, ef, ext_row0, ra, rb); return;
                default: break;
            }
        }
    }
    edge_recorrelate<real, NT>(a, map_s, ext, ext_row0, ra, rb);
}

// ---------------------------------------------------------------------------------------------------------------
// Near-tie re-ranking (float maps).  The map the engine ranks on is not the reference's bit for bit: its initial
// values come from the tensor-core K1 (3xFP16 split, fp32 accumulation in TMEM: up to ~1.2e-6 of max|c| away from
// the exact product, where NumPy's sgemm is at ~1e-7) and interior windows are kept current by Gram updates, which
// accumulate rounding, while the reference re-correlates every window from the residual (:1018-1051).  The north
// star allows a different pick only at near-ties below 1e-6 relative correlation gap, so the pick must not depend
// on that noise: whenever another entry of the map comes within `tol` of the best approximate score, ALL entries
// within `tol` are re-scored from the residual itself - <r[t-off : t-off+L], D[k]> accumulated in float64, which is
// what the reference's map holds up to its own rounding - and the best re-scored entry wins (lowest (t,k) among
// equals, np.argmax's rule, :967).  Rows whose filter support overhangs the signal keep their stored value: the
// edge path writes them with the reference's reflect-padded arithmetic in float64.
// The test for "another entry within tol" rides on loads the atom needs anyway (its map row, the level-1 keys of its
// 128-row group) and on the scan of the group keys; the re-scoring itself runs for a fraction of a percent of the atoms.

// Rows whose filter support overhangs the signal (r < off or r > T-L+off) hold, in the reference, the ZERO-padded
// initial correlation (:161-164) until an atom's window reaches them, and REFLECT-padded re-correlations afterwards
// (:1046).  The edge path writes the latter exactly (float64 accumulation); the former come from K1.  One bit per
// overhanging row (hsc_signal_state::edge_written, head rows / tail rows, up to 64 each) records which kind a row
// holds, so that a never-rewritten row can be re-scored from the residual with zero padding - the residual under
// its support is still the input signal there.
__device__ __forceinline__ bool overhang_row_written(const hsc_signal_state& st, int r, int off, int T, int L) {
    if (r < off) return r < 64 ? ((st.edge_written[0] >> r) & 1ull) != 0ull : true;
    const int d = T - 1 - r;                       // tail rows counted from the end
    return d < 64 ? ((st.edge_written[1] >> d) & 1ull) != 0ull : true;
}

__device__ __forceinline__ void mark_overhang_rows(hsc_signal_state& st, int lo, int hi, int off, int T, int L) {
    // rows [lo, hi] were re-correlated by the edge path: set the bits of the overhanging ones
    for (int r = lo; r <= hi && r < off && r < 64; ++r) st.edge_written[0] |= 1ull << r;
    for (int r = max(lo, T - L + off + 1); r <= hi; ++r) {
        const int d = T - 1 - r;
        if (d >= 0 && d < 64) st.edge_written[1] |= 1ull << d;
    }
}

// Score of map entry (r, k) from the residual by one warp: <r[r-off : r-off+L], D[k]> in float64, clipped (= zero
// padded) at the signal ends.  Returns the signed value; only meaningful for rows that are NOT reflect-rewritten.
template <typename real>
__device__ __forceinline__ double residual_dot_warp(const MpArgs<real>& a, const real* res_s, int r, int k, int T) {
    const int lane = threadIdx.x & 31;
    const int sstart = r - a.off;
    const int jlo = sstart < 0 ? -sstart : 0;
    const int jhi = (sstart + a.L > T) ? (T - sstart) : a.L;
    const real* rr = res_s + (long long)sstart * a.F;
    const real* dd = a.D + (long long)k * a.L * a.F;
    double acc = 0.0;
    for (int q = jlo * a.F + lane; q < jhi * a.F; q += 32) acc = fma((double)rr[q], (double)dd[q], acc);
    return warp_sum(acc);
}

// Exact score of map entry (r, k): |<residual window, D[k]>| * w[k], or the stored value for a reflect-rewritten row.
template <typename real>
__device__ __forceinline__ double exact_score_warp(const MpArgs<real>& a, const hsc_signal_state& st, const real* map_s, const real* res_s,
                                                   int r, int k) {
    double sc;
    const int T = a.T;
    const bool overhang = (r < a.off) || (r > T - a.L + a.off);
    if (!overhang || !overhang_row_written(st, r, a.off, T, a.L)) sc = fabs(residual_dot_warp<real>(a, res_s, r, k, T));
    else sc = fabs((double)__ldcg(map_s + (long long)r * a.K + k));
    return a.w ? sc * fabs((double)a.w[k]) : sc;
}

// Slow path, one warp, a fraction of a percent of the atoms (a few percent on dense single sequences): enumerate every
// map entry whose approximate score is >= thr - level 2 -> rows -> entries, each stage one batch of independent loads -
// re-score the candidates from the residual (four at a time, eight lanes each), keep the best.
// `lvl2(g)` gives the approximate best score of 128-row group g.
constexpr int kRerankMax = 32;          // candidates per stage; beyond that the surplus is dropped (the window holds a handful)

template <bool RAGGED, typename real, typename Lvl2>
__device__ __forceinline__ void rerank_candidates(const MpArgs<real>& a, const hsc_signal_state& st, const real* map_s, const real* res_s,
                                                  const real* v1, Lvl2 lvl2, uint32_t slot3_saddr, int g1s, real thr, int& t_out, int& k_out) {
    __shared__ int cand_g[kRerankMax], cand_r[kRerankMax], cand_k[kRerankMax];
    const int lane = threadIdx.x & 31;
    const int T = signal_length<RAGGED>(a), K = a.K, L = a.L, F = a.F, LF = a.L * a.F;
    const int n2 = RAGGED ? (T + (1 << g1s) - 1) >> g1s : a.n2;    // the signal's groups (a.n2: those of the stride)
    // stage 1: groups - through the block scores where the hierarchy has them (a block below thr holds no candidate group)
    int ng = 0;
    if (slot3_saddr) {
        const int n3 = (n2 + 31) >> 5;
        for (int b0 = 0; b0 < n3; b0 += 32) {
            const int b = b0 + lane;
            unsigned mb = __ballot_sync(0xffffffffu, b < n3 && (real)__uint_as_float(lds_u32(slot3_saddr + 4u * (unsigned)b)) >= thr);
            while (mb) {                                           // (warp-uniform) candidate blocks, ascending
                const int g = ((b0 + __ffs(mb) - 1) << 5) + lane;
                mb &= mb - 1;
                const bool h = g < n2 && lvl2(g) >= thr;
                const unsigned m = __ballot_sync(0xffffffffu, h);
                if (h) { const int slot = ng + __popc(m & ((1u << lane) - 1u)); if (slot < kRerankMax) cand_g[slot] = g; }
                ng += __popc(m);
            }
        }
    } else
    for (int g0 = 0; g0 < n2; g0 += 128) {                         // four independent key loads per lane and step
        bool h[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) { const int g = g0 + u * 32 + lane; h[u] = g < n2 && lvl2(g) >= thr; }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const unsigned m = __ballot_sync(0xffffffffu, h[u]);
            if (h[u]) { const int slot = ng + __popc(m & ((1u << lane) - 1u)); if (slot < kRerankMax) cand_g[slot] = g0 + u * 32 + lane; }
            ng += __popc(m);
        }
    }
    ng = min(ng, kRerankMax);
    __syncwarp();
    // stage 2: rows of the candidate groups (G1 = 128 rows = 4 per lane)
    int nr = 0;
    for (int i = 0; i < ng; ++i) {
        const int r0 = cand_g[i] << g1s, r_end = min(r0 + (1 << g1s), T);
        for (int rb = r0; rb < r_end; rb += 128) {
            bool h[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) { const int r = rb + u * 32 + lane; h[u] = r < r_end && v1[r] >= thr; }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const unsigned m = __ballot_sync(0xffffffffu, h[u]);
                if (h[u]) { const int slot = nr + __popc(m & ((1u << lane) - 1u)); if (slot < kRerankMax) cand_r[slot] = rb + u * 32 + lane; }
                nr += __popc(m);
            }
        }
    }
    nr = min(nr, kRerankMax);
    __syncwarp();
    // stage 3: entries of the candidate rows
    int nc = 0;
    for (int i = 0; i < nr; ++i) {
        const int rr = cand_r[i];
        const real* mrow = map_s + (long long)rr * K;
        for (int kb = 0; kb < K; kb += 128) {
            bool h[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int kk = kb + u * 32 + lane;
                h[u] = false;
                if (kk < K) { const real m = __ldcg(mrow + kk); h[u] = rabs<real>(a.w ? m * a.w[kk] : m) >= thr; }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const unsigned m = __ballot_sync(0xffffffffu, h[u]);
                if (h[u]) {
                    const int slot = nc + __popc(m & ((1u << lane) - 1u));
                    if (slot < kRerankMax) { cand_g[slot] = rr; cand_k[slot] = kb + u * 32 + lane; }      // cand_g now holds the candidate's row
                }
                nc += __popc(m);
            }
        }
    }
    nc = min(nc, kRerankMax);
    __syncwarp();
    // stage 4: exact scores, four candidates at a time (eight lanes each)
    const int sub = lane >> 3, sl = lane & 7;
    double best = -1.0;
    long long best_flat = LLONG_MAX;
    for (int c0 = 0; c0 < nc; c0 += 4) {
        const int c = c0 + sub;
        double sc = -1.0;
        long long flat = LLONG_MAX;
        if (c < nc) {
            const int r = cand_g[c], k = cand_k[c];
            flat = (long long)r * K + k;
            const bool overhang = (r < a.off) || (r > T - L + a.off);
            if (!overhang || !overhang_row_written(st, r, a.off, T, L)) {
                const int sstart = r - a.off;
                const int jlo = sstart < 0 ? -sstart : 0;
                const int jhi = (sstart + L > T) ? (T - sstart) : L;
                const real* rr = res_s + (long long)sstart * F;
                const real* dd = a.D + (long long)k * LF;
                double acc = 0.0;
                for (int q = jlo * F + sl; q < jhi * F; q += 8) acc = fma((double)rr[q], (double)dd[q], acc);
                sc = acc;
            } else {
                sc = sl == 0 ? (double)__ldcg(map_s + flat) : 0.0;
            }
        }
        for (int m = 4; m > 0; m >>= 1) sc += __shfl_xor_sync(0xffffffffu, sc, m);          // sum over the eight lanes
        if (c < nc) {
            sc = fabs(sc);
            if (a.w) sc *= fabs((double)a.w[cand_k[c]]);
        } else {
            sc = -1.0;
        }
        // best over the four sub-groups: larger score, then lower flat index
        for (int m = 16; m >= 8; m >>= 1) {
            const double os = __shfl_xor_sync(0xffffffffu, sc, m);
            const long long of = __shfl_xor_sync(0xffffffffu, flat, m);
            if (os > sc || (os == sc && of < flat)) { sc = os; flat = of; }
        }
        if (sc > best || (sc == best && flat < best_flat)) { best = sc; best_flat = flat; }
    }
    if (best_flat != LLONG_MAX && best >= 0.0) {
        t_out = (int)(best_flat / K);
        k_out = (int)(best_flat - (long long)t_out * K);
    }
}

// Fast test by one warp, after the approximate pick (t, k): is any OTHER entry of the atom's own row or of the other rows
// of its 128-row group within tol?  (Other groups are tested by the caller on the group keys.)
template <typename real, bool RAGGED>
__device__ __forceinline__ bool near_tie_in_group(const MpArgs<real>& a, const real* map_s, const real* v1, int g1s, int t, int k, real thr) {
    const int lane = threadIdx.x & 31;
    bool amb = false;
    const int r0 = (t >> g1s) << g1s, r1 = min(r0 + (1 << g1s), signal_length<RAGGED>(a));
    const real* mrow = map_s + (long long)t * a.K;
    // every load of the test is issued before the first compare: the level-1 keys of the group's rows and the first 256
    // entries of the atom's map row fly together (one dependent round trip under load instead of two)
    constexpr int RU = 4, MU = 8;
    real vv[RU], mm[MU];
#pragma unroll
    for (int u = 0; u < RU; ++u) { const int r = r0 + lane + 32 * u; vv[u] = r < r1 ? v1[r] : (real)-1; }
#pragma unroll
    for (int u = 0; u < MU; ++u) { const int kk = lane + 32 * u; mm[u] = kk < a.K ? __ldcg(mrow + kk) : (real)0; }
#pragma unroll
    for (int u = 0; u < RU; ++u) { const int r = r0 + lane + 32 * u; amb |= r < r1 && r != t && vv[u] >= thr; }
    for (int r = r0 + lane + 32 * RU; r < r1; r += 32) amb |= (r != t) && (v1[r] >= thr);
#pragma unroll
    for (int u = 0; u < MU; ++u) {
        const int kk = lane + 32 * u;
        amb |= kk < a.K && (kk != k) && (rabs<real>(a.w ? mm[u] * a.w[kk] : mm[u]) >= thr);
    }
    for (int kk = lane + 32 * MU; kk < a.K; kk += 32) {
        const real m = __ldcg(mrow + kk);
        amb |= (kk != k) && (rabs<real>(a.w ? m * a.w[kk] : m) >= thr);
    }
    return __any_sync(0xffffffffu, amb);
}

// The near-tie TEST of one selection, by warp 1 while warp 0 evaluates the coefficient of the same approximate pick (t, k)
// of score vbest (out of line, so that the persistent loop's register allocation is not disturbed): does any OTHER map
// entry score within the re-rank window of it - the other 128-row groups on their keys (SMH: `second`, a by-product of
// warp 0's scan of the group keys), the other rows of the atom's group on their level-1 keys, the other filters of its row
// on the map?  Returns the score threshold of the candidate set, or a negative value when the pick is unambiguous.
template <typename real, bool SMH, bool RAGGED>
__device__ __noinline__ real near_tie_watch(const MpArgs<real>& a, hsc_signal_state& st, const real* map_s, const real* res_s,
                                            const real* v1, const int* i1, const real* v2g, const real* v3g, const int* i3g, int g1s,
                                            int t, int k, real vbest, real second, uint32_t slot2_saddr, int next_g) {
    const int lane = threadIdx.x & 31;
    if constexpr (!SMH) {                          // global hierarchy: repeat warp 0's (deterministic) pick
        real bv = (real)0;
        int bt = INT_MAX;
        for (int e = lane; e < a.n3; e += 32) take_first_max(bv, bt, v3g[e], i3g[e]);
        group_argmax(bv, bt, 32);
        if (bt == INT_MAX) return (real)-1;
        t = bt;
        k = i1[t];
        vbest = bv;
    }
    if (st.reserved == 0) {                        // largest score of the initial map: the scale of K1's rounding
        __syncwarp();
        if (lane == 0) st.reserved = (int)__float_as_uint((float)vbest);
        __syncwarp();
    }
    const real thr = vbest - (real)a.rerank_tol * (vbest + (real)__uint_as_float((unsigned)st.reserved));
    bool amb;
    if constexpr (SMH) {
        amb = second >= thr;
    } else {
        const int gsel = t >> g1s;
        const int n2 = RAGGED ? (signal_length<RAGGED>(a) + (1 << g1s) - 1) >> g1s : a.n2;
        amb = false;
        for (int e = lane; e < n2; e += 32) amb |= (e != gsel) && (v2g[e] >= thr);
        amb = __any_sync(0xffffffffu, amb);
    }
    if (!amb) amb = near_tie_in_group<real, RAGGED>(a, map_s, v1, g1s, t, k, thr);
    if constexpr (SMH) {
        // The best entry of the OTHER groups is, most of the time, the next pick (an update only changes the 2L-1 rows
        // around its atom): pull what its selection will read - the residual under its support, its map row, the level-1
        // keys of its group - towards L2 now, off the critical path, so that the next atom's dependent loads do not pay a
        // DRAM round trip under load.
        if (a.next_prefetch && next_g < 0 && second > (real)0) {
            // the best of the other groups lies in another block (select_smh only knows its score): find the block, then the group
            const unsigned sbits = __float_as_uint((float)second);
            const uint32_t slot3_saddr = slot2_saddr + 8u * (unsigned)a.n2;
            const int n3 = (a.n2 + 31) >> 5;
            int bb = INT_MAX;
            for (int e = lane; e < n3; e += 32)
                if (lds_u32(slot3_saddr + 4u * (unsigned)e) == sbits && e != ((t >> g1s) >> 5)) bb = min(bb, e);
            bb = __reduce_min_sync(0xffffffffu, bb);
            if (bb != INT_MAX) {
                const int g = (bb << 5) + lane;
                const unsigned ghi = g < a.n2 ? lds_u32(slot2_saddr + 8u * (unsigned)g + 4u) : 0u;
                const int gg = __reduce_min_sync(0xffffffffu, ghi == sbits ? g : INT_MAX);
                if (gg != INT_MAX) next_g = gg;
            }
        }
        if (a.next_prefetch && next_g >= 0 && lane < 3) {
            const unsigned low = 0xFFFFFFFFu - lds_u32(slot2_saddr + 8u * (unsigned)next_g);
            const int rl = (int)(low / (unsigned)a.K);
            const int t2 = (next_g << g1s) + rl;
            const void* p;
            unsigned bytes;
            if (lane == 0) {
                const int s0 = max(t2 - a.off, 0);
                p = res_s + (long long)s0 * a.F;
                bytes = (unsigned)(min(t2 - a.off + a.L, signal_length<RAGGED>(a)) - s0) * a.F * sizeof(real);
            } else if (lane == 1) {
                p = map_s + (long long)t2 * a.K;
                bytes = (unsigned)a.K * sizeof(real);
            } else {
                const int r0 = next_g << g1s;
                p = v1 + r0;
                bytes = (unsigned)(min(r0 + (1 << g1s), signal_length<RAGGED>(a)) - r0) * sizeof(real);
            }
            if ((((unsigned long long)p) & 15ull) == 0 && (bytes & 15u) == 0 && bytes > 0)
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" :: "l"(p), "r"(bytes) : "memory");
        }
    }
    return amb ? thr : (real)-1;
}

// ... and its resolution, by warp 0, in the rare case the test fires: every entry with an approximate score >= thr is
// re-scored from the residual and (t, k) becomes the best of them; returns its coefficient.
template <typename real, bool SMH, bool RAGGED>
__device__ __noinline__ real near_tie_resolve(const MpArgs<real>& a, hsc_signal_state& st, const real* map_s, const real* res_s,
                                              const real* v1, uint32_t slot2_saddr, const real* v2g, int g1s, real thr,
                                              int& t, int& k) {
    if constexpr (SMH) {
        auto lvl2 = [&](int g) { return (real)__uint_as_float(lds_u32(slot2_saddr + 8u * (unsigned)g + 4u)); };
        rerank_candidates<RAGGED, real>(a, st, map_s, res_s, v1, lvl2, slot2_saddr + 8u * (unsigned)a.n2, g1s, thr, t, k);   // (slot3 follows slot2)
    } else {
        auto lvl2 = [&](int g) { return v2g[g]; };
        rerank_candidates<RAGGED, real>(a, st, map_s, res_s, v1, lvl2, 0u, g1s, thr, t, k);
    }
    const int T = signal_length<RAGGED>(a);
    const bool row_overhangs = (t < a.off) || (t > T - a.L + a.off);
    const bool from_residual = a.coef_mode == 1 && (!row_overhangs || !overhang_row_written(st, t, a.off, T, a.L));
    return from_residual ? (real)residual_dot_warp<real>(a, res_s, t, k, T) : __ldcg(map_s + (long long)t * a.K + k);
}

// Block-wise selection of one pass (_selectBestAtoms with nbBlocks > 1 or 'auto', hsc/modeling.py:908-963,
// plus the weak-atom filter of computeCoefficients, :1090-1099): one argmax per time block (blocks shifted
// by half a block on 'offset' passes), range / null / interference filters, sort by |c| descending.  The
// coefficient of every atom is captured HERE, before any atom of the pass is applied (:946, :1101-1120).
// Returns the number of atoms, left in selection order in list 1 (cand_*[ncand_max ...]).
template <typename real, int NT, bool RAGGED>
__device__ __noinline__ int build_pass_list(const MpArgs<real>& a, const real* map_s, const real* res_s, const real* v1,
                                            const int* i1, int* ct, int* ck, real* cc, int offset_flag, double energy_signal) {
    const int T = signal_length<RAGGED>(a), K = a.K, L = a.L, F = a.F, off = a.off, LF = L * F;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = NT >> 5;
    __shared__ int s_count;
    int bs = a.nb_blocks < 0 ? 4 * L : (int)floor((double)T / (double)a.nb_blocks);
    if (bs & 1) bs += 1;
    int nblk = (T + bs - 1) / bs;
    const int front = offset_flag ? bs / 2 : 0;
    if (offset_flag) nblk += 1;
    int* ct2 = ct + a.ncand_max; int* ck2 = ck + a.ncand_max; real* cc2 = cc + a.ncand_max;

    // 1. argmax of every block over the level-1 keys (lowest row wins a tie, like the flattened argmax)
    for (int b = warp; b < nblk; b += nwarps) {
        const int r0 = max(b * bs - front, 0), r1 = min((b + 1) * bs - front, T);
        real bv = (real)0;
        int bt = INT_MAX;
        for (int r = r0 + lane; r < r1; r += 32) take_first_max(bv, bt, v1[r], r);
        group_argmax(bv, bt, 32);
        const bool all_zero = bt == INT_MAX;              // every row's key is 0: np.argmax gives the block's first entry,
        if (r0 < r1 && all_zero) bt = r0;                 // (first row, filter 0), of coefficient 0 - an all-zero row's key
        int k = 0;                                        // index is INT_MAX, not a filter
        real c = (real)0;
        if (r0 < r1) {
            k = all_zero ? 0 : i1[bt];
            c = __ldcg(map_s + (long long)bt * K + k);
            const bool edge = (bt - (L - 1) < off) || (bt + (L - 1) > T - L + off);
            if (a.coef_mode == 1 && !edge) {
                const real* rr = res_s + (long long)(bt - off) * F;
                const real* dd = a.D + (long long)k * LF;
                double acc = 0.0;
                for (int q = lane; q < LF; q += 32) acc = fma((double)rr[q], (double)dd[q], acc);
                acc = warp_sum(acc);
                c = (real)acc;
            }
        }
        if (lane == 0) {
            ct[b] = r0 < r1 ? bt : -1;
            ck[b] = k;
            cc[b] = c;
        }
    }
    __syncthreads();
    // 2. range + null + interference filters, in time order (single thread: the lists are short)
    if (tid == 0) {
        int n = 0;
        for (int b = 0; b < nblk; ++b) {
            const int t = ct[b];
            if (t < 0) continue;
            const real c = cc[b];
            const bool keep = a.null_thres >= (real)0 ? (rabs<real>(c) > a.null_thres) : true;
            if (!keep) continue;
            ct[n] = t; ck[n] = ck[b]; cc[n] = c;
            ++n;
        }
        bool any_far = false;
        for (int i = 0; i + 1 < n; ++i) any_far |= (ct[i + 1] - ct[i]) >= L;
        if (any_far) {
            int m = 1;                                     // element 0 is always kept (:954)
            int prev = ct[0];
            for (int i = 1; i < n; ++i) {
                const int cur = ct[i];
                if (cur - prev >= L) { ct[m] = cur; ck[m] = ck[i]; cc[m] = cc[i]; ++m; }
                prev = cur;                                // gap to the PREDECESSOR IN TIME, kept or not (:951)
            }
            n = m;
        }
        s_count = n;
    }
    __syncthreads();
    int n = s_count;
    // 3. weak-atom filter (:1090-1099): only when an SNR target is set and the pass holds more than one atom
    if (a.has_snr && n > 1) {
        const double thr = (double)(real)((real)energy_signal / (real)pow(10.0, (double)a.tol_snr / 10.0)) / ((double)T * F);
        for (int i = warp; i < n; i += nwarps) {
            const int sstart = ct[i] - off;
            const int jlo = sstart < 0 ? -sstart : 0;
            const int jhi = (sstart + L > T) ? (T - sstart) : L;
            const real* rr = res_s + (long long)sstart * F;
            double acc = 0.0;
            for (int q = jlo * F + lane; q < jhi * F; q += 32) acc = fma((double)rr[q], (double)rr[q], acc);
            acc = warp_sum(acc);
            const double mean_e = (double)(real)(acc / (double)((jhi - jlo) * F));
            if (lane == 0) ck2[i] = mean_e >= thr ? 1 : 0;  // ck2 doubles as the keep flag here
        }
        __syncthreads();
        if (tid == 0) {
            int m = 0;
            for (int i = 0; i < n; ++i)
                if (ck2[i]) { ct[m] = ct[i]; ck[m] = ck[i]; cc[m] = cc[i]; ++m; }
            s_count = m;
        }
        __syncthreads();
        n = s_count;
    }
    // 4. order by |c| descending; equal magnitudes in reverse list order (np.argsort(...)[::-1], :960-962)
    for (int i = tid; i < n; i += NT) {
        const real ai = rabs<real>(cc[i]);
        int rank = 0;
        for (int j = 0; j < n; ++j) {
            const real aj = rabs<real>(cc[j]);
            rank += (aj > ai) || (aj == ai && j > i);
        }
        ct2[rank] = ct[i]; ck2[rank] = ck[i]; cc2[rank] = cc[i];
    }
    __syncthreads();
    return n;
}

// SMH (float scores, TMA window path, T <= kSlotMax * G1, or longer sequences when the launch has at most one CTA per SM): levels 2 and 3 of the argmax hierarchy are replaced by one
// packed key per 128-row group held in SHARED memory for the kernel's lifetime.  Selecting reads shared memory
// only, and an update folds the rewritten rows into their <= kDirtyMax groups with a handful of shared atomics, so the
// serial chain of an atom keeps a single dependent global round trip (the residual/dictionary dot product) instead
// of five (level 3 -> row -> map entry, then level-1 -> level-2 -> level-3 re-keying).
// Selection on the shared-memory hierarchy by one warp: the best packed key of all 128-row groups -> out[0] = row t (or -1
// if every key is zero), out[1] = filter k, out[2] = score bits, out[3] = best score bits among the OTHER groups (equal
// scores included; the near-tie watch compares it with the re-rank threshold), out[4] = that group (-1: none).
__device__ __noinline__ void select_smh(uint32_t slot2_saddr, uint32_t slot3_saddr, int n2, int K, int g1s, int* out) {
    // Two steps: the best score of every block of 32 consecutive groups (slot3, one word per block), then the 32 groups of
    // the winning block - a few shared-memory loads per lane whatever the length of the sequence (a flat scan of the
    // group keys of a 1e6-sample sequence, 7813 of them, was half of the time per selection at the config-2 shape).
    // Ties go to the lowest block, then the lowest group, then the key's own (row, filter) order: np.argmax's rule.
    const int lane = threadIdx.x & 31;
    const int n3 = (n2 + 31) >> 5;
    unsigned bhi = 0u, bhi2 = 0u;                  // best block score, and best score of the other blocks, of this lane's blocks
    int bb = INT_MAX;
    for (int e = lane; e < n3; e += 32) {
        const unsigned hi = lds_u32(slot3_saddr + 4u * (unsigned)e);
        if (hi > bhi) { bhi2 = bhi; bhi = hi; bb = e; }
        else if (hi > bhi2) bhi2 = hi;
    }
    const unsigned mx = __reduce_max_sync(0xffffffffu, bhi);
    const int lane_bb = bb;
    bb = __reduce_min_sync(0xffffffffu, (bhi == mx && mx != 0u) ? bb : INT_MAX);
    unsigned second = __reduce_max_sync(0xffffffffu, lane_bb == bb ? bhi2 : bhi);     // best score of the other blocks
    int bg = INT_MAX, g2 = INT_MAX;
    if (bb != INT_MAX) {
        const int g = (bb << 5) + lane;
        const unsigned ghi = g < n2 ? lds_u32(slot2_saddr + 8u * (unsigned)g + 4u) : 0u;
        bg = __reduce_min_sync(0xffffffffu, ghi == mx ? g : INT_MAX);
        const unsigned in2 = __reduce_max_sync(0xffffffffu, g == bg ? 0u : ghi);         // ... and of the block's other groups
        if (in2 >= second) {
            second = in2;
            g2 = __reduce_min_sync(0xffffffffu, (g != bg && ghi == in2 && in2 != 0u) ? g : INT_MAX);
        }
    }
    if (lane == 0) {
        if (bg == INT_MAX) {
            out[0] = -1; out[1] = 0;
        } else {
            const unsigned low = 0xFFFFFFFFu - lds_u32(slot2_saddr + 8u * (unsigned)bg);
            const unsigned rl = low / (unsigned)K;
            out[0] = (bg << g1s) + (int)rl;
            out[1] = (int)(low - rl * (unsigned)K);
        }
        out[2] = (int)mx;
        out[3] = (int)second;
        out[4] = g2 == INT_MAX ? -1 : g2;          // group of the best score among the other groups when it lies in the same block (else unknown)
    }
    __threadfence_block();
}

// Best score of block b of 32 consecutive groups, recomputed from the group keys by one warp.
__device__ __forceinline__ void refold_block(const unsigned long long* slot2, unsigned* slot3, int b, int n2) {
    const int g = (b << 5) + (int)(threadIdx.x & 31);
    const unsigned hi = g < n2 ? (unsigned)(slot2[g] >> 32) : 0u;
    const unsigned mx = __reduce_max_sync(0xffffffffu, hi);
    if ((threadIdx.x & 31) == 0) slot3[b] = mx;
}

constexpr int kSlotMax = 1024;
constexpr int kDirtyMax = 8;

// The body of K2 (pursuit_kernel / pursuit_kernel_ragged).  RAGGED: the signals have their own lengths (a.len,
// hsc_b200_mp_begin_lengths); a separate kernel, so that the uniform launches bound everything by the parameter a.T
// exactly as before and pay nothing for it.
template <typename real, int NT, int VIF, bool TMA, bool SMH, int RPS, bool RAGGED>
__device__ __forceinline__ void pursuit_body(MpArgs<real> a) {
    const int s = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = NT / 32;
    const int Tst = a.T, K = a.K, L = a.L, F = a.F, off = a.off;       // Tst: the row stride (and a uniform batch's length)
    const int W = 2 * L - 1;
    const int LF = L * F;
#ifdef HSC_PROFILE_PHASES
    long long prof_kernel_t0;
    { unsigned long long ns_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns_)); prof_kernel_t0 = (long long)ns_; }
#endif

    // per-signal base pointers live in shared memory (loaded at the use sites) to keep the persistent
    // loop's register footprint small; so does a ragged signal's length T, which bounds everything below (the arrays
    // keep the row stride a.T)
    struct Ctx {
        real* map_s; real* res_s; real* v1; int* i1; real* v2; int* i2; real* v3; int* i3;
        unsigned* bits; int* evp; int* evi; real* evc;
        int* ct; int* ck; real* cc;
    };
    __shared__ Ctx cx;
    if (threadIdx.x == 0) {
        cx.map_s = a.map + (long long)s * Tst * K;
        cx.res_s = a.resid + (long long)s * Tst * F;
        cx.v1 = a.val1 + (long long)s * Tst;
        cx.i1 = a.idx1 + (long long)s * Tst;
        cx.v2 = a.val2 + (long long)s * a.n2;
        cx.i2 = a.idx2 + (long long)s * a.n2;
        cx.v3 = a.val3 + (long long)s * a.n3;
        cx.i3 = a.idx3 + (long long)s * a.n3;
        cx.bits = a.bitmap + (long long)s * a.bitmap_words;
        cx.evp = a.ev_pos + (long long)s * a.cap;
        cx.evi = a.ev_idx + (long long)s * a.cap;
        cx.evc = a.ev_coef + (long long)s * a.cap;
        cx.ct = a.cand_t ? a.cand_t + (long long)s * 2 * a.ncand_max : nullptr;
        cx.ck = a.cand_k ? a.cand_k + (long long)s * 2 * a.ncand_max : nullptr;
        cx.cc = a.cand_c ? a.cand_c + (long long)s * 2 * a.ncand_max : nullptr;
        if constexpr (RAGGED) CtaLength<true>::set(a.len[s]);
    }
#define T (CtaLength<RAGGED>::get(Tst))
#define map_s (cx.map_s)
#define res_s (cx.res_s)
#define v1 (cx.v1)
#define i1 (cx.i1)
#define v2 (cx.v2)
#define i2 (cx.i2)
#define v3 (cx.v3)
#define i3 (cx.i3)
#define bits (cx.bits)
#define evp (cx.evp)
#define evi (cx.evi)
#define evc (cx.evc)

    __shared__ hsc_signal_state st;
    __shared__ struct {
        int t, k, edge, stop, last;
        real coef;
        real thr;           // near-tie re-ranking: score threshold of the candidate set, < 0 = the pick is unambiguous
    } sel;
    __shared__ double red_a[NW], red_b[NW];
    __shared__ real red_m[NW];
    __shared__ struct { int t, k; unsigned vbest, second; int g2; } watch;     // warp 0's approximate pick (select_smh), also read by warp 1's near-tie watch

    // interior window update through shared memory (gram_update_tma): stage ring + one mbarrier per stage
    extern __shared__ __align__(128) unsigned char win_smem[];
    __shared__ __align__(8) unsigned long long win_bar[(NT / 32) * 4];
    constexpr bool tma_on = TMA;
    unsigned win_phase = 0;                      // mbarrier parity per stage, tracked by every thread
    unsigned long long* slot2 = reinterpret_cast<unsigned long long*>(win_smem + a.tma_bytes);   // [n2] packed best key of every level-2 group (SMH)
    unsigned* slot3 = reinterpret_cast<unsigned*>(slot2 + a.n2);                                // [ceil(n2/32)] best score of every block of 32 groups
    __shared__ unsigned long long dirty_slot[kDirtyMax];        // the groups an update touches, rebuilt per atom
    const int g1s = 31 - __clz(a.G1);                           // G1 is a power of two (128)
    if (tid == 0) {
        st = a.state[s];
        if (tma_on) {
            for (int i = 0; i < (NT / 32) * a.tma_stages; ++i) mbarrier_init(smem_addr_u32(&win_bar[i]), 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            fence_proxy_async_all();
        }
    }
    __syncthreads();
    if (st.status != HSC_RUNNING && st.status != HSC_PAUSE_CAPACITY && st.status != HSC_PAUSE_PASSES) return;

    const int g = min(32, pow2_at_least(K));     // lanes per map row
    const int ngroups = NT / g;
    const int grp = tid / g, lig = tid % g;
    // vector path of the interior update: K a multiple of the 16-byte vector, <= 8 vectors per lane per row
    constexpr int VN = VecOf<real>::N;
    const int nvec = (K % VN == 0) ? K / VN : 0;
    const int gv = min(32, pow2_at_least(nvec > 0 ? nvec : 1));
    int vec_pv = 0;
    if (nvec > 0) {
        const int per_lane = (nvec + gv - 1) / gv;
        vec_pv = per_lane <= 1 ? 1 : per_lane <= 2 ? 2 : per_lane <= 4 ? 4 : 0;
    }

    if (!st.initialised) {
        // energySignal = sum x^2 (:1070); the residual buffer holds x at this point (:1071)
        double acc = 0.0;
        {
            const real* rr = res_s;
            const long long n = (long long)T * F;
            double p0 = 0.0, p1 = 0.0, p2 = 0.0, p3 = 0.0;
            long long e = tid;
            for (; e + 3ll * NT < n; e += 4ll * NT) {
                const double a0 = (double)rr[e], a1 = (double)rr[e + NT], a2 = (double)rr[e + 2ll * NT], a3 = (double)rr[e + 3ll * NT];
                p0 = fma(a0, a0, p0); p1 = fma(a1, a1, p1); p2 = fma(a2, a2, p2); p3 = fma(a3, a3, p3);
            }
            for (; e < n; e += NT) {
                const double a0 = (double)rr[e];
                p0 = fma(a0, a0, p0);
            }
            acc = (p0 + p1) + (p2 + p3);
        }
        acc = warp_sum(acc);
        if (lane == 0) red_a[warp] = acc;
        __syncthreads();
        if (tid == 0) {
            double tot = 0.0;
            for (int i = 0; i < NW; ++i) tot += red_a[i];
            real es = (real)tot;
            st.energy_signal = (double)es;
            st.energy_residual = (double)es;
            st.n_events = st.nnz = st.duplicates = st.passes = 0;
            st.offset_flag = 0;
            st.pass_count = 0;
            st.pass_cursor = 0;
            st.initialised = 1;
        }
        // level-1 keys were written by rowkey_kernel (hsc_b200_mp_begin)
        if constexpr (!SMH) {
            rekey_level<real>(v1, nullptr, T, v2, i2, 0, a.n2 - 1, a.G1, NT);
            __syncthreads();
            rekey_level<real>(v2, i2, a.n2, v3, i3, 0, a.n3 - 1, a.G2, NT);
            __syncthreads();
        }
    }
    if constexpr (SMH) {
        // (re)build the shared-memory level from the level-1 keys in global memory: first launch and resumes alike
        if (tid < kDirtyMax) dirty_slot[tid] = 0ull;
        for (int gi = warp; gi < a.n2; gi += NW) {
            unsigned long long best = 0ull;
            const int e1 = min((gi + 1) << g1s, T);
            for (int r = (gi << g1s) + lane; r < e1; r += 32) {
                const unsigned long long key = pack_key(v1[r], r & (a.G1 - 1), i1[r], K);
                best = key > best ? key : best;
            }
            best = warp_max_u64(best);
            if (lane == 0) slot2[gi] = best;
        }
        __syncthreads();
        for (int b = warp; b < (a.n2 + 31) >> 5; b += NW) refold_block(slot2, slot3, b, a.n2);
    }
    if (tid == 0) {
        st.status = HSC_RUNNING;
        st.n_buffered = 0;
    }
    __syncthreads();

    long long passes_this_run = 0;
    const bool rerank_on = sizeof(real) == 4 && a.rerank_tol > 0.f && a.nb_blocks == 1;
#ifdef HSC_PROFILE_PHASES
    long long prof_t = clock64(), prof_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    long long prof_edge[4] = {0, 0, 0, 0};
    long long prof_loop_t0;
    { unsigned long long ns_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns_)); prof_loop_t0 = (long long)ns_; }
#define HSC_STAMP(i) do { if (tid == 0) { long long now_ = clock64(); prof_acc[i] += now_ - prof_t; prof_t = now_; } } while (0)
#else
#define HSC_STAMP(i) do { } while (0)
#endif
    while (true) {
        HSC_STAMP(0);
        // ------------------------------------------------------------------ pause rules
        if (st.n_buffered >= a.cap) {
            if (tid == 0) st.status = HSC_PAUSE_CAPACITY;
            break;
        }
        const bool block_mode = a.nb_blocks != 1;
        const bool new_pass = !block_mode || st.pass_cursor >= st.pass_count;
        if (new_pass && a.max_passes > 0 && passes_this_run >= a.max_passes) {
            if (tid == 0) st.status = HSC_PAUSE_PASSES;
            break;
        }
        if (block_mode && new_pass) {
            // ---------------------------------------------------------------- block-wise selection of a pass
            const int n = build_pass_list<real, NT, RAGGED>(a, map_s, res_s, v1, i1, cx.ct, cx.ck, cx.cc, st.offset_flag, st.energy_signal);
            if (tid == 0) {
                st.pass_count = n;
                st.pass_cursor = 0;
            }
            __syncthreads();
            if (n == 0) {                                      // empty selection -> converged (:1150-1153)
                if (tid == 0) {
                    st.passes += 1;
                    st.status = HSC_STOP_EMPTY;
                }
                break;
            }
        }
        // ------------------------------------------------------------------ select (:965-975)
        if (block_mode) {
            if (warp == 0) {
                const int cur = st.pass_cursor;
                const int t = cx.ct[a.ncand_max + cur], k = cx.ck[a.ncand_max + cur];
                const real coef = cx.cc[a.ncand_max + cur];
                const int edge = (t - (L - 1) < off) || (t + (L - 1) > T - L + off);
                if (lane == 0) {
                    sel.t = t;
                    sel.k = k;
                    sel.edge = edge;
                    sel.coef = coef;
                    sel.stop = 0;
                    sel.last = (cur + 1 >= st.pass_count);
                }
                if (a.prefetch && !edge && lane < 2) {
                    const real* p = lane == 0 ? (const real*)(map_s + (long long)(t - (L - 1)) * K) : (a.G + (long long)k * W * K);
                    const unsigned bytes = (unsigned)((long long)W * K * sizeof(real));
                    if ((((unsigned long long)p) & 15ull) == 0 && (bytes & 15u) == 0)
                        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" :: "l"(p), "r"(bytes) : "memory");
                }
            }
        } else if (warp == 0) {
            int t, k;
            if constexpr (SMH) {
                // scan of the group keys (out of line: its registers do not weigh on the persistent loop); the result
                // comes back through `watch`, which also hands the pick to warp 1's near-tie watch
                select_smh(smem_addr_u32(slot2), smem_addr_u32(slot3), a.n2, K, g1s, &watch.t);
                __syncwarp();
                t = watch.t < 0 ? 0 : watch.t;                 // < 0: all-zero map, np.argmax gives (0, 0), a null coefficient
                k = watch.k;
                if (rerank_on) asm volatile("bar.arrive 1, 64;" ::: "memory");      // named barrier 1: warps 0 and 1
            } else {
                real bv = (real)0;
                int bt = INT_MAX;
                for (int e = lane; e < a.n3; e += 32) take_first_max(bv, bt, v3[e], i3[e]);
                group_argmax(bv, bt, 32);
                if (bt == INT_MAX) {                           // all-zero map: np.argmax gives (0, 0), a null coefficient
                    t = 0; k = 0;
                } else {
                    t = bt;
                    k = i1[t];
                }
            }
            const int edge = (t - (L - 1) < off) || (t + (L - 1) > T - L + off);
            // coefficient = UNWEIGHTED map entry (:970).  coef_mode 1: re-evaluated from the residual instead wherever
            // the row is not a reflect-rewritten one (interior rows: drift-free; never-rewritten overhanging rows of a
            // float map: the zero-padded product in float64 instead of K1's tensor-core value)
            const bool row_overhangs = (t < off) || (t > T - L + off);
            const bool from_residual = a.coef_mode == 1 && (!row_overhangs || (sizeof(real) == 4 && !overhang_row_written(st, t, off, T, L)));
            real coef = from_residual ? (real)residual_dot_warp<real>(a, res_s, t, k, T) : __ldcg(map_s + (long long)t * K + k);
            if (lane == 0) {
                sel.t = t;
                sel.k = k;
                sel.edge = edge;
                sel.coef = coef;
                sel.stop = 0;
                sel.last = 1;
            }
            // one instruction pulls the whole 2L-1 row window (and the Gram slice) towards L2 while the
            // bookkeeping / residual phases run: DRAM-level parallelism without registers or shared memory
            if (a.prefetch && !edge && lane < 2) {
                const real* p = lane == 0 ? (const real*)(map_s + (long long)(t - (L - 1)) * K) : (a.G + (long long)k * W * K);
                const unsigned bytes = (unsigned)((long long)W * K * sizeof(real));
                if ((((unsigned long long)p) & 15ull) == 0 && (bytes & 15u) == 0)
                    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" :: "l"(p), "r"(bytes) : "memory");
            }
        } else if (warp == 1 && rerank_on) {
            // near-tie watch (float maps): while warp 0 evaluates the coefficient, warp 1 tests whether any other entry
            // comes within the re-rank window of the pick - the atom's serial chain keeps its single dependent global
            // round trip
            real thr = (real)-1;
            if constexpr (SMH) {
                asm volatile("bar.sync 1, 64;" ::: "memory");           // warp 0's pick is in `watch`
                if (watch.t >= 0)
                    thr = near_tie_watch<real, true, RAGGED>(a, st, map_s, res_s, v1, i1, v2, v3, i3, g1s, watch.t, watch.k,
                                                     (real)__uint_as_float(watch.vbest), (real)__uint_as_float(watch.second),
                                                     smem_addr_u32(slot2), watch.g2);
            } else {
                thr = near_tie_watch<real, false, RAGGED>(a, st, map_s, res_s, v1, i1, v2, v3, i3, g1s, 0, 0, (real)0, (real)-1, 0u, -1);
            }
            if (lane == 0) sel.thr = thr;
        }
        __syncthreads();
        if (rerank_on && sel.thr >= (real)0) {
            // near-tie (a fraction of a percent of the atoms): warp 0 re-scores the candidate set from the residual
            if (warp == 0) {
                int t = sel.t, k = sel.k;
                const real coef = near_tie_resolve<real, SMH, RAGGED>(a, st, map_s, res_s, v1, smem_addr_u32(slot2), v2, g1s, sel.thr, t, k);
                __syncwarp();
                if (lane == 0) {
                    sel.t = t;
                    sel.k = k;
                    sel.edge = (t - (L - 1) < off) || (t + (L - 1) > T - L + off);
                    sel.coef = coef;
                    st.reranked += 1;
                }
            }
            __syncthreads();
        }
        HSC_STAMP(1);   // select
        const int t = sel.t, k = sel.k, edge = sel.edge;
        const real coef = sel.coef;
        const bool pass_ends = sel.last != 0;                 // last atom of its selection pass

        // null coefficient -> empty selection -> converged (:974-975, :1150-1153)
        const bool is_null = (a.null_thres >= (real)0) ? !(rabs<real>(coef) > a.null_thres) : (coef == (real)0);
        if (!block_mode && is_null) {
            if (tid == 0) {
                st.passes += 1;
                st.status = HSC_STOP_EMPTY;
            }
            break;
        }

        // interior atom on the bulk-copy window path: its first window chunks start flying now
        if constexpr (TMA) {
            if (!edge && a.early_issue) gram_window_issue<real, NT, RPS>(K, L, map_s, a.G + (long long)k * W * K, t, gv, win_smem, win_bar, a.tma_stages);
        }

        // ------------------------------------------------------------------ bookkeeping (:1106-1114)
        // The selection bitmap's test-and-set is ONE atomic whose result (first selection of (t,k) or a duplicate) is
        // only needed by the stop rules after the window update: no dependent round trip here.
        unsigned bk_old = 0u, bk_m = 0u;
        if (tid == 0) {
            const unsigned long long bit = (unsigned long long)t * K + k;
            bk_m = 1u << (bit & 31);
            bk_old = atomicOr(bits + (bit >> 5), bk_m);
            evp[st.n_buffered] = t;
            evi[st.n_buffered] = k;
            evc[st.n_buffered] = coef;
            st.n_buffered += 1;
            st.n_events += 1;
        }
        HSC_STAMP(5);   // bookkeeping (thread 0's own timeline)

        // ------------------------------------------------------------------ residual (:996-1016), loads first
        const int row_lo = max(t - (L - 1), 0), row_hi = min(t + (L - 1), T - 1);
        const int g2_lo = row_lo >> g1s, g2_hi = row_hi >> g1s;
        const int sstart = t - off;
        const int jlo = sstart < 0 ? -sstart : 0;
        const int jhi = (sstart + L > T) ? (T - sstart) : L;
        const real* dd = a.D + (long long)k * LF;
        real* rr = res_s + (long long)sstart * F;
        const int q_first = jlo * F + tid;
        real ro_first = (real)0, dq_first = (real)0;
        if (q_first < jhi * F) {                                  // in flight while the level-1 keys below are fetched
            ro_first = rr[q_first];
            dq_first = dd[q_first];
        }

        // ------------------------------------------------------------------ SMH: rows of the dirty groups outside the window
        if constexpr (SMH) {
            // their level-1 keys are unchanged: fold them into the groups' fresh keys straight from global memory
            // (32 consecutive rows per warp step lie in one group: G1 is a multiple of 32)
            const int span0 = g2_lo << g1s, span1 = min((g2_hi + 1) << g1s, T);
            for (int r0 = span0 + warp * 32; r0 < span1; r0 += NT) {
                const int r = r0 + lane;
                unsigned long long key = 0ull;
                if (r < span1 && (r < row_lo || r > row_hi)) key = pack_key(v1[r], r & (a.G1 - 1), i1[r], K);
                key = warp_max_u64(key);
                if (lane == 0 && key) atomicMax(&dirty_slot[(r0 >> g1s) - g2_lo], key);
            }
        }

        {
            double eb = 0.0, ea = 0.0;
            if (q_first < jhi * F) {
                const real rn = sub_scaled(ro_first, coef, dq_first);
                rr[q_first] = rn;
                eb = fma((double)ro_first, (double)ro_first, eb);
                ea = fma((double)rn, (double)rn, ea);
            }
            for (int q = q_first + NT; q < jhi * F; q += NT) {
                real ro = rr[q];
                real rn = sub_scaled(ro, coef, dd[q]);
                rr[q] = rn;
                eb = fma((double)ro, (double)ro, eb);
                ea = fma((double)rn, (double)rn, ea);
            }
            eb = warp_sum(eb);
            ea = warp_sum(ea);
            if (lane == 0) {
                red_b[warp] = eb;
                red_a[warp] = ea;
            }
        }
        HSC_STAMP(6);   // residual

        // ------------------------------------------------------------------ map window (:1018-1051)
        if (!edge) {
            const real* Gk = a.G + (long long)k * W * K;
            if constexpr (TMA) {
                if (!a.early_issue) gram_window_issue<real, NT, RPS>(K, L, map_s, Gk, t, gv, win_smem, win_bar, a.tma_stages);
                if (a.w) win_phase = gram_update_tma<real, NT, true, SMH, RPS>(K, L, a.w, map_s, Gk, v1, i1, t, coef, gv, win_smem, win_bar, a.tma_stages, win_phase, dirty_slot, g2_lo, g1s, true);
                else if (RPS == 1 && gv == 32 && a.row32) win_phase = gram_update_row32<real, NT, SMH>(K, L, map_s, Gk, v1, i1, t, coef, win_smem, win_bar, a.tma_stages, win_phase, dirty_slot, g2_lo, g1s);
                else win_phase = gram_update_tma<real, NT, false, SMH, RPS>(K, L, a.w, map_s, Gk, v1, i1, t, coef, gv, win_smem, win_bar, a.tma_stages, win_phase, dirty_slot, g2_lo, g1s, true);
            }
            // (the register path under the shared-memory hierarchy only ever runs narrow maps, which take the plain loop below:
            //  the vector variants are not instantiated there - they cost that variant 500 bytes of spills for dead code)
            else if (!(SMH && !TMA) && vec_pv == 1 && !a.w && !a.scalar_window) gram_update_vec<real, 1, NT, VIF, false>(K, L, a.w, map_s, Gk, v1, i1, t, coef, gv);
            else if (!(SMH && !TMA) && vec_pv == 2 && !a.w && !a.scalar_window) gram_update_vec<real, 2, NT, VIF, false>(K, L, a.w, map_s, Gk, v1, i1, t, coef, gv);
            else if (!(SMH && !TMA) && vec_pv == 4 && VIF >= 4 && !a.w && !a.scalar_window) gram_update_vec<real, 4, NT, VIF, false>(K, L, a.w, map_s, Gk, v1, i1, t, coef, gv);
            else {
                for (int base = 0; base < W; base += ngroups) {
                    const int i = base + grp;
                    const bool valid = i < W;
                    real bv = (real)0;
                    int bi = INT_MAX;
                    const int tr = t - (L - 1) + i;
                    if (valid) {
                        real* mrow = map_s + (long long)tr * K;
                        const real* grow = Gk + (long long)i * K;
                        for (int kk = lig; kk < K; kk += g) {
                            real m = fma(-coef, grow[kk], mrow[kk]);
                            mrow[kk] = m;
                            real sc = rabs<real>(a.w ? m * a.w[kk] : m);
                            take_first_max(bv, bi, sc, kk);
                        }
                    }
                    group_argmax(bv, bi, g);
                    if (valid && lig == 0) {
                        v1[tr] = bv;
                        i1[tr] = bi;
                        if constexpr (SMH) {           // (register path under the shared-memory hierarchy: fold the row right here)
                            const unsigned long long key = pack_key(bv, tr & (a.G1 - 1), bi, K);
                            if (key) atomicMax(&dirty_slot[(tr >> g1s) - g2_lo], key);
                        }
                    }
                }
            }
        } else {
            __syncthreads();   // the recompute reads the updated residual
#ifdef HSC_PROFILE_PHASES
            const long long edge_t0 = clock64();
#endif
            const long long first = (long long)t - off - (L - 1);
            const long long last = (long long)t + L / 2 + (L - 1);
            const long long lo = first < 0 ? 0 : first;
            const long long hi = last > T - 1 ? T - 1 : last;
            // Rows whose filter support overhangs the signal are re-correlated from the residual with the
            // reference's reflect padding; so is the whole window if the atom itself was clipped (the Gram
            // tensor describes an unclipped atom).  The other rows of the window take the Gram update.
            const bool clipped = (t - off < 0) || (t - off + L > T);
            const real* Gk = a.G + (long long)k * W * K;
            // rows to re-correlate: everything if clipped, else the head rows (tr < off) and the tail rows (tr > T-L+off)
            const int head_hi = clipped ? row_hi : min(row_hi, off - 1);             // [row_lo, head_hi]
            const int tail_lo = clipped ? row_hi + 1 : max(max(row_lo, T - L + off + 1), head_hi + 1); // [tail_lo, row_hi]
            {   // the reflect-padded slice those rows read: samples row_lo-off .. row_hi-off+L-1.  It is staged in the (idle)
                // stage rings of the window pipeline when they are large enough (+ one step of zero padding: the window
                // variant of the re-correlation reads a little past the last row), else in global scratch
                const int nx = (row_hi - row_lo + L) * F;
                const int nx_pad = nx + 8 * F + 8;
                const bool ext_in_smem = tma_on && (size_t)nx_pad * sizeof(real) <= (size_t)a.tma_bytes;
                real* ext = ext_in_smem ? reinterpret_cast<real*>(win_smem) : a.edge_ext + (long long)s * a.edge_stride;
                for (int e = tid; e < (ext_in_smem ? nx_pad : nx); e += NT) {
                    const int xs = e / F;
                    ext[e] = e < nx ? res_s[reflect_index((long long)row_lo - off + xs, lo, hi) * F + (e - xs * F)] : (real)0;
                }
                __syncthreads();
                if (head_hi >= row_lo) edge_recorrelate_any<real, NT>(a, map_s, ext, ext_in_smem, row_lo, row_lo, head_hi);
                if (tail_lo <= row_hi) edge_recorrelate_any<real, NT>(a, map_s, ext, ext_in_smem, row_lo, tail_lo, row_hi);
                if (tid == 0) {                                // those rows now hold reflect-padded values
                    if (head_hi >= row_lo) mark_overhang_rows(st, row_lo, head_hi, off, T, L);
                    if (tail_lo <= row_hi) mark_overhang_rows(st, tail_lo, row_hi, off, T, L);
                }
            }
            const int g_lo = max(row_lo, head_hi + 1), g_hi = min(row_hi, tail_lo - 1);  // rows that take the Gram update
            for (int e = tid; e < (g_hi - g_lo + 1) * K; e += NT) {
                const int rr_ = e / K, kk = e - rr_ * K;
                const int tr = g_lo + rr_;
                const long long o = (long long)tr * K + kk;
                map_s[o] = fma(-coef, Gk[(long long)(tr - t + (L - 1)) * K + kk], __ldcg(map_s + o));
            }
            if (tma_on) fence_proxy_async_all();               // generic-proxy map writes -> later bulk loads of these rows
            __syncthreads();
#ifdef HSC_PROFILE_PHASES
            const long long edge_t1 = clock64();
#endif
            rekey_rows(a, map_s, v1, i1, row_lo, row_hi, g, NT, SMH ? dirty_slot : nullptr, g2_lo, g1s);
#ifdef HSC_PROFILE_PHASES
            prof_edge[0] += edge_t1 - edge_t0; prof_edge[1] += clock64() - edge_t1; prof_edge[2] += 1; prof_edge[3] += clipped ? 1 : 0;
#endif
        }
        HSC_STAMP(7);   // map window, warp 0's share
        __syncthreads();
        // (register window path under the shared-memory hierarchy - narrow maps -: the plain window loop above has folded its
        //  rows' fresh level-1 keys into the dirty groups itself, the edge path's re-key likewise)
        HSC_STAMP(2);   // bookkeeping + residual + map window

        // ------------------------------------------------------------------ hierarchy levels 2, 3
        if constexpr (SMH) {
            if (warp == 1) {                                  // publish the rebuilt groups, re-arm the scratch keys, refresh their blocks
                if (lane <= g2_hi - g2_lo) {
                    slot2[g2_lo + lane] = dirty_slot[lane];
                    dirty_slot[lane] = 0ull;
                }
                __syncwarp();
                for (int b = g2_lo >> 5; b <= g2_hi >> 5; ++b) refold_block(slot2, slot3, b, a.n2);
            }
        } else {
            rekey_level<real>(v1, nullptr, T, v2, i2, g2_lo, g2_hi, a.G1, NT);
        }
        // energy + stop rules ride on the same barrier (:1014, :1125-1142)
        if (tid == 0) {
            double eb = 0.0, ea = 0.0;
            for (int i = 0; i < NW; ++i) {
                eb += red_b[i];
                ea += red_a[i];
            }
            if (bk_old & bk_m) st.duplicates += 1;              // (t,k) had been selected before (:1106-1111)
            else st.nnz += 1;
            const real loss = (real)eb - (real)ea;
            const real e_now = (real)st.energy_residual - loss;
            st.energy_residual = (double)e_now;
            if (block_mode) st.pass_cursor += 1;
            int stop = 0;
            if (e_now < a.eps) {
                stop = HSC_STOP_ENERGY;
            } else {
                const real snr = (real)10 * rlog10<real>((real)st.energy_signal / e_now);
                if (a.max_nnz >= 0 && st.nnz >= a.max_nnz) stop = HSC_STOP_NNZ;
                else if (a.has_snr && snr >= a.tol_snr) stop = HSC_STOP_SNR;
                else if (a.max_events_total > 0 && st.n_events >= a.max_events_total) stop = HSC_STOP_MAX_EVENTS;
            }
            if (pass_ends || stop) {                          // end of the selection pass (:1160-1163)
                st.passes += 1;
                st.offset_flag ^= 1;
                if (stop) st.pass_cursor = st.pass_count;      // converged mid-pass: the rest of the list is dropped
            }
            sel.stop = stop;
        }
        if (pass_ends) ++passes_this_run;
        if (!SMH || a.has_scale) __syncthreads();             // SMH: sel.stop is published by the barrier that ends the body
        HSC_STAMP(3);   // level 2 + energy/stop rules
        if constexpr (!SMH) rekey_level<real>(v2, i2, a.n2, v3, i3, g2_lo / a.G2, g2_hi / a.G2, a.G2, NT);

        // ------------------------------------------------------------------ residual scale (:1145-1148)
        if (a.has_scale && (pass_ends || sel.stop)) {     // once per selection pass (:1144-1148)
            real m = (real)0;
            for (long long e = tid; e < (long long)T * F; e += NT) {
                real v = rabs<real>(res_s[e]);
                m = v > m ? v : m;
            }
            m = warp_max<real>(m);
            if (lane == 0) red_m[warp] = m;
            __syncthreads();
            if (tid == 0) {
                real mm = (real)0;
                for (int i = 0; i < NW; ++i) mm = red_m[i] > mm ? red_m[i] : mm;
                if (mm <= a.tol_scale && sel.stop == 0) sel.stop = HSC_STOP_SCALE;
            }
        }
        // every warp's bulk stores of this atom's window: complete, and ordered before the generic-proxy reads of the
        // map and the next atom's bulk loads that follow the barrier (they were issued two phases ago: no stall)
        {   // (the lanes that issued them: gram_update_row32 stores from the elect.sync lane - the same one every time for the
            //  full mask -, the general window loop and the edge path from lane 0)
            const bool elected = elect_one_sync();
            if (tma_on && (elected || lane == 0)) {
                bulk_wait_all();
                fence_proxy_async_all();
            }
        }
        __syncthreads();
        HSC_STAMP(4);   // level 3 (+ residual scale)
        if (sel.stop) {
            if (tid == 0) st.status = sel.stop;
            break;
        }
    }
    __syncthreads();
#ifdef HSC_PROFILE_PHASES
    if (tid == 0 && a.prof) {
        for (int i = 0; i < 8; ++i) a.prof[(long long)s * 16 + i] = prof_acc[i];
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        a.prof[(long long)s * 16 + 8] = (long long)smid;
        a.prof[(long long)s * 16 + 9] = prof_kernel_t0;                    // globaltimer at kernel entry (ns)
        a.prof[(long long)s * 16 + 10] = prof_loop_t0;                     // ... at the first atom
        unsigned long long now_ns;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now_ns));
        a.prof[(long long)s * 16 + 11] = (long long)now_ns;                // ... at exit
        for (int i = 0; i < 4; ++i) a.prof[(long long)s * 16 + 12 + i] = prof_edge[i];   // edge path: recompute cycles, rekey cycles, atoms, clipped
    }
#endif
    if (tid == 0) a.state[s] = st;
#undef HSC_STAMP
#undef T
#undef map_s
#undef res_s
#undef v1
#undef i1
#undef v2
#undef i2
#undef v3
#undef i3
#undef bits
#undef evp
#undef evi
#undef evc
}

template <typename real, int NT, int MINB, int VIF, bool TMA, bool SMH, int RPS = 1>
__global__ void __launch_bounds__(NT, MINB) pursuit_kernel(MpArgs<real> a) { pursuit_body<real, NT, VIF, TMA, SMH, RPS, false>(a); }

template <typename real, int NT, int MINB, int VIF, bool TMA, bool SMH, int RPS = 1>
__global__ void __launch_bounds__(NT, MINB) pursuit_kernel_ragged(MpArgs<real> a) { pursuit_body<real, NT, VIF, TMA, SMH, RPS, true>(a); }

}  // namespace hsc
