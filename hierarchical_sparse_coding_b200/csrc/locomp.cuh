// LoCOMP on the device (LoCOMP.computeCoefficients, hsc/modeling.py:1263-1425): matching pursuit plus, per
// selected atom, a least-squares refit of the atom and the already-selected atoms that share its support
// (_findCommonSupportAtoms :1221-1239, _getDictionaryFromSupportAtoms :1241-1261, pinv solve :1330-1333).
//
// One CTA per signal like the MP kernel, same workspace (map, argmax hierarchy, selection bitmap).
//  * neighbours: the selection bitmap IS the support of the code, so the common-support search is a scan of the
//    bits of rows [lo, hi] around the atom; the reference's predicate is replicated as written (:1238: an entry
//    is kept iff (row - lo) != t AND filter != k - it compares a slice-relative row with an absolute position).
//  * refit: coef = pinv(Dsup)^T r  ==  (Dsup Dsup^T)^+ (Dsup r).  The n x n normal matrix comes straight from the
//    shift Gram tensor (A_ij = G[k_i][t_j - t_i][k_j], zero beyond L-1 shifts; direct sums for clipped atoms) and
//    the right-hand side is <r, atom_i> from the residual; solved in float64 by Cholesky in shared memory.
//  * the fitted values are INCREMENTS (they are fitted to the residual, :1336-1338): every group atom emits an
//    event (t, k, delta); all residual subtractions come first (:1341), then the map windows (:1353).
#pragma once
#include "pursuit.cuh"

namespace hsc {

constexpr int kLocompMaxGroup = 256;      // selected atom + at most 255 common-support atoms
constexpr int kLocompSmemGroup = 64;      // groups up to this size keep their normal equations in shared memory
// engine scratch per signal (doubles): the normal matrix of a large group, then the group list of the fast kernel's apply phase
constexpr long long kLocompScratchStride = (long long)kLocompMaxGroup * (kLocompMaxGroup + 1) + 2 * kLocompMaxGroup;
// the fast kernel's refit scratch, overlaid on the (idle) stage rings of the window pipeline
constexpr int kLocompOverlayBytes = kLocompSmemGroup * (kLocompSmemGroup + 1) * 8 + kLocompMaxGroup * (8 + 8 + 8 + 4 + 4);

// An atom at t whose window (rows t-L+1 .. t+L-1) reaches a row with overhanging support: its window takes the two-phase
// element-wise path of locomp_window, and a coef_mode == 1 pick keeps the map's coefficient.
__device__ __forceinline__ bool locomp_edge(int t, int L, int T, int off) {
    return (t - (L - 1) < off) || (t + (L - 1) > T - L + off);
}

// <atom (ti,ki), atom (tj,kj)> with both atoms clipped to [0,T) (T: the signal's length).
template <typename real, bool RAGGED>
__device__ double atom_inner(const MpArgs<real>& a, int ti, int ki, int tj, int kj) {
    const int L = a.L, F = a.F, T = signal_length<RAGGED>(a), off = a.off;
    const int d = tj - ti;
    if (d >= L || d <= -L) return 0.0;
    const int si = ti - off, sj = tj - off;
    const bool clipped = si < 0 || sj < 0 || si + L > T || sj + L > T;
    if (!clipped) return (double)a.G[((long long)ki * (2 * L - 1) + (d + L - 1)) * a.K + kj];
    const int x0 = max(max(si, sj), 0), x1 = min(min(si, sj) + L, T);
    const real* di = a.D + (long long)ki * L * F;
    const real* dj = a.D + (long long)kj * L * F;
    double acc = 0.0;
    for (int x = x0; x < x1; ++x)
        for (int f = 0; f < F; ++f) acc = fma((double)di[(x - si) * F + f], (double)dj[(x - sj) * F + f], acc);
    return acc;
}

// Map window of one applied atom, in two phases so that a whole refit group stays consistent:
//   phase 0 (incremental): rows whose support lies inside the signal take c -= coef * G (skipped for a clipped
//            atom, whose whole window is absolute);
//   phase 1 (absolute):    overhang rows - or the whole window of a clipped atom - are re-correlated from the
//            residual with reflect padding (hsc/modeling.py:1046).
// All incremental updates of a group must precede all absolute ones: a re-correlated row already reflects
// every residual change of the group, so a later increment on it would count an atom twice.
template <typename real, int NT, bool RAGGED>
__device__ void locomp_window(const MpArgs<real>& a, real* map_s, const real* res_s, int t, int k, real coef, int phase) {
    const int T = signal_length<RAGGED>(a), K = a.K, L = a.L, F = a.F, off = a.off, W = 2 * L - 1, LF = L * F;
    const int tid = threadIdx.x;
    const int row_lo = max(t - (L - 1), 0), row_hi = min(t + (L - 1), T - 1);
    const long long first = (long long)t - off - (L - 1);
    const long long last = (long long)t + L / 2 + (L - 1);
    const long long lo = first < 0 ? 0 : first;
    const long long hi = last > T - 1 ? T - 1 : last;
    const int nrows = row_hi - row_lo + 1;
    const bool clipped = (t - off < 0) || (t - off + L > T);
    const real* Gk = a.G + (long long)k * W * K;
    for (int e = tid; e < nrows * K; e += NT) {
        const int rr_ = e / K, kk = e - rr_ * K;
        const int tr = row_lo + rr_;
        const bool absolute = clipped || (tr < off) || (tr > T - L + off);
        if (phase == 1 && absolute) {
            const real* dd = a.D + (long long)kk * LF;
            double acc = 0.0;
            for (int j = 0; j < L; ++j) {
                const long long src = reflect_index((long long)tr - off + j, lo, hi);
                const real* rp = res_s + src * F;
                for (int f = 0; f < F; ++f) acc = fma((double)rp[f], (double)dd[j * F + f], acc);
            }
            map_s[(long long)tr * K + kk] = (real)acc;
        } else if (phase == 0 && !absolute) {
            const long long o = (long long)tr * K + kk;
            map_s[o] = fma(-coef, Gk[(long long)(tr - t + (L - 1)) * K + kk], __ldcg(map_s + o));   // (L2-coherent: bulk stores do not update L1)
        }
    }
    __syncthreads();
}

// ---------------------------------------------------------------------------------------------------------------------
// The steps both kernels below share.  They differ only in the argmax hierarchy, where the fitted group lives and how the
// map windows are applied; everything else is one copy here.  A ragged kernel passes its signal's length T (and the fast
// kernel its per-signal pointers) as read at the call site.  Barriers that differ between the kernels stay at the call
// sites or are template parameters.

// One atom of a fitted group, as a kernel's group storage hands it to locomp_record and locomp_subtract.
template <typename real> struct LocompAtom { int t, k; real x; };

// First launch of a signal: its energy over the n = T * F samples, rounded to the data's precision, and a fresh state.
template <typename real, int NT>
__device__ __forceinline__ void locomp_init_state(hsc_signal_state& st, const real* res_s, long long n, double* red_a) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double acc = 0.0;
    for (long long e = tid; e < n; e += NT) {
        const double v = (double)res_s[e];
        acc = fma(v, v, acc);
    }
    acc = warp_sum(acc);
    if (lane == 0) red_a[warp] = acc;
    __syncthreads();
    if (tid == 0) {
        double tot = 0.0;
        for (int i = 0; i < NT / 32; ++i) tot += red_a[i];
        const real es = (real)tot;
        st.energy_signal = (double)es;
        st.energy_residual = (double)es;
        st.n_events = st.nnz = st.duplicates = st.passes = 0;
        st.offset_flag = 0;
        st.pass_count = 0;
        st.pass_cursor = 0;
        st.initialised = 1;
    }
}

// Head of each selection: pause when the event buffers could not take a whole group or the launch's pass budget is spent;
// in block mode, build the next pass list, and stop when it is empty.  Returns true to leave the loop (st.status says why).
template <typename real, int NT, bool RAGGED>
__device__ __forceinline__ bool locomp_loop_head(const MpArgs<real>& a, hsc_signal_state& st, bool block_mode, long long passes_this_run,
                                                 const real* map_s, const real* res_s, const real* v1, const int* i1,
                                                 int* ct, int* ck, real* cc) {
    const int tid = threadIdx.x;
    if (st.n_buffered + kLocompMaxGroup > a.cap) {         // a selection may emit up to kLocompMaxGroup events
        if (tid == 0) st.status = HSC_PAUSE_CAPACITY;
        return true;
    }
    const bool new_pass = !block_mode || st.pass_cursor >= st.pass_count;
    if (new_pass && a.max_passes > 0 && passes_this_run >= a.max_passes) {
        if (tid == 0) st.status = HSC_PAUSE_PASSES;
        return true;
    }
    if (block_mode && new_pass) {
        const int n = build_pass_list<real, NT, RAGGED>(a, map_s, res_s, v1, i1, ct, ck, cc, st.offset_flag, st.energy_signal);
        if (tid == 0) {
            st.pass_count = n;
            st.pass_cursor = 0;
        }
        __syncthreads();
        if (n == 0) {
            if (tid == 0) {
                st.passes += 1;
                st.status = HSC_STOP_EMPTY;
            }
            return true;
        }
    }
    return false;
}

// Block mode: the next atom of the pass list, with the coefficient captured when the list was built.
template <typename real>
__device__ __forceinline__ void locomp_pass_pick(const MpArgs<real>& a, const hsc_signal_state& st, const int* ct, const int* ck,
                                                 const real* cc, int& t, int& k, real& coef, int& last) {
    const int cur = st.pass_cursor;
    t = ct[a.ncand_max + cur];
    k = ck[a.ncand_max + cur];
    coef = cc[a.ncand_max + cur];
    last = (cur + 1 >= st.pass_count);
}

// Coefficient of an argmax pick (one warp): the map's value, or with coef_mode == 1 and an interior atom <r, atom> from the
// residual.
template <typename real>
__device__ __forceinline__ real locomp_pick_coef(const MpArgs<real>& a, const real* res_s, int T, int L, int F, int off, int t, int k,
                                                  real map_value) {
    const int LF = L * F;
    if (a.coef_mode != 1 || locomp_edge(t, L, T, off)) return map_value;
    const real* rr = res_s + (long long)(t - off) * F;
    const real* dd = a.D + (long long)k * LF;
    double acc = 0.0;
    for (int q = threadIdx.x & 31; q < LF; q += 32) acc = fma((double)rr[q], (double)dd[q], acc);
    acc = warp_sum(acc);
    return (real)acc;
}

// Argmax mode: a null coefficient ends the pursuit.  Returns true to leave the loop.
template <typename real>
__device__ __forceinline__ bool locomp_null_stop(const MpArgs<real>& a, hsc_signal_state& st, bool block_mode, real coef) {
    const bool is_null = (a.null_thres >= (real)0) ? !(rabs<real>(coef) > a.null_thres) : (coef == (real)0);
    if (block_mode || !is_null) return false;
    if (threadIdx.x == 0) {
        st.passes += 1;
        st.status = HSC_STOP_EMPTY;
    }
    return true;
}

// Common-support atoms of the pick (t, k) (:1221-1239): the selected bits of rows [lo, hi] that pass the reference's
// predicate go to g_key[1 ..] (s_n counts the group, from 1); more than kLocompMaxGroup stops the signal with
// HSC_STOP_GROUP.  Returns true to leave the loop.
template <int NT>
__device__ __forceinline__ bool locomp_common_support(hsc_signal_state& st, const unsigned* bits, int t, int k, int T, int K, int L, int off,
                                                      long long* g_key, int& s_n, int& s_bad) {
    const int tid = threadIdx.x;
    const int sp0 = max(t - off, 0), ep0 = min(t + L / 2, T - 1);               // Atom.getPositionSpanIndices (:845-858)
    const int lo = max(sp0 - L / 2, 0);
    const int hi = min(min(ep0 + ((L % 2 == 0) ? L / 2 - 1 : L / 2), T), T - 1);
    const long long b0 = (long long)lo * K, b1 = (long long)(hi + 1) * K;       // bit range [b0, b1)
    for (long long wI = (b0 >> 5) + tid; wI <= ((b1 - 1) >> 5); wI += NT) {
        unsigned wv = bits[wI];
        while (wv) {
            const int bpos = __ffs(wv) - 1;
            wv &= wv - 1;
            const long long bit = (wI << 5) + bpos;
            if (bit < b0 || bit >= b1) continue;
            const int tt = (int)(bit / K), kk = (int)(bit - (long long)tt * K);
            if ((tt - lo) != t && kk != k) {                                     // the reference's predicate, as written (:1238)
                const int slot = atomicAdd(&s_n, 1);
                if (slot < kLocompMaxGroup) g_key[slot] = bit;
                else s_bad = 1;
            }
        }
    }
    __syncthreads();
    if (s_bad) {
        if (tid == 0) st.status = HSC_STOP_GROUP;
        return true;
    }
    return false;
}

// Least-squares refit of a group of n atoms (:1322-1338): (g_t[0], g_k[0]) is the pick, g_key[1 .. n-1] its common-support
// atoms.  Sorts the neighbours into row-major order (the COO order of the reference's LIL slice), builds the right-hand side
// <r, atom_i> and the normal matrix, and solves by Cholesky in float64: increments in g_x.  The normal matrix lives at
// A_smem (pitch kLocompSmemGroup + 1) for n <= kLocompSmemGroup, else in this signal's slice of the engine's scratch.  A
// numerically dependent support falls back to a plain MP step: s_n = 1, g_x[0] = coef.  No barrier after the last write.
template <typename real, int NT, bool RAGGED>
__device__ __forceinline__ void locomp_refit(const MpArgs<real>& a, const real* res_s, int T, int K, int L, int F, int off, int n, real coef,
                                             double* A_smem, const long long* g_key, int* g_t, int* g_k, double* g_b, double* g_x, int& s_n) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = NT / 32;
    const int LF = L * F;
    if (n <= 1) {
        if (tid == 0) g_x[0] = (double)coef;
        return;
    }
    const bool big = n > kLocompSmemGroup;
    double* const A = big ? a.locomp_scratch + (long long)blockIdx.x * kLocompScratchStride : A_smem;
    const int pitch = big ? kLocompMaxGroup + 1 : kLocompSmemGroup + 1;
    auto Aij = [&](int i, int j) -> double& { return A[(long long)i * pitch + j]; };
    for (int i = 1 + tid; i < n; i += NT) {
        const long long key = g_key[i];
        int rank = 1;
        for (int j = 1; j < n; ++j) rank += g_key[j] < key;
        g_t[rank] = (int)(key / K);
        g_k[rank] = (int)(key - (long long)(key / K) * K);
    }
    __syncthreads();
    // right-hand side <r, atom_i> (clipped) and normal matrix
    for (int i = warp; i < n; i += NW) {
        const int si = g_t[i] - off;
        const int jlo = si < 0 ? -si : 0, jhi = (si + L > T) ? (T - si) : L;
        const real* rr = res_s + (long long)si * F;
        const real* dd = a.D + (long long)g_k[i] * LF;
        double acc = 0.0;
        for (int q = jlo * F + lane; q < jhi * F; q += 32) acc = fma((double)rr[q], (double)dd[q], acc);
        acc = warp_sum(acc);
        if (lane == 0) g_b[i] = acc;
    }
    for (int e = tid; e < n * n; e += NT) {
        const int i = e / n, j = e - i * n;
        if (j >= i) {
            const double v = atom_inner<real, RAGGED>(a, g_t[i], g_k[i], g_t[j], g_k[j]);
            Aij(i, j) = v;
            Aij(j, i) = v;
        }
    }
    __syncthreads();
    // Cholesky A = L L^T, then two triangular solves (float64, warp 0)
    if (warp != 0) return;
    bool ok = true;
    double dmax = 0.0;
    for (int i = lane; i < n; i += 32) dmax = fmax(dmax, Aij(i, i));
    for (int m = 16; m > 0; m >>= 1) dmax = fmax(dmax, __shfl_xor_sync(0xffffffffu, dmax, m));
    for (int j = 0; j < n; ++j) {
        double d = Aij(j, j);
        for (int p = 0; p < j; ++p) d -= Aij(j, p) * Aij(j, p);              // all lanes compute the same scalar
        if (!(d > 1e-13 * dmax)) { ok = false; break; }
        const double ljj = sqrt(d);
        __syncwarp();
        for (int i = j + 1 + lane; i < n; i += 32) {
            double v = Aij(i, j);
            for (int p = 0; p < j; ++p) v -= Aij(i, p) * Aij(j, p);
            Aij(i, j) = v / ljj;
        }
        if (lane == 0) Aij(j, j) = ljj;
        __syncwarp();
    }
    if (ok && lane == 0) {
        for (int i = 0; i < n; ++i) {                                            // L y = b
            double v = g_b[i];
            for (int p = 0; p < i; ++p) v -= Aij(i, p) * g_x[p];
            g_x[i] = v / Aij(i, i);
        }
        for (int i = n - 1; i >= 0; --i) {                                       // L^T x = y
            double v = g_x[i];
            for (int p = i + 1; p < n; ++p) v -= Aij(p, i) * g_x[p];
            g_x[i] = v / Aij(i, i);
        }
    }
    if (lane == 0 && !ok) {                  // numerically dependent support: plain MP step for this atom
        s_n = 1;
        g_x[0] = (double)coef;
    }
}

// Thread 0: the pick's bit in the code (a repeat counts as a duplicate, 'Redundant atom selected', :1314-1315) and one event
// (t, k, increment) per group atom.
template <typename real, typename Group>
__device__ __forceinline__ void locomp_record(hsc_signal_state& st, unsigned* bits, int* evp, int* evi, real* evc, int t, int k, int K,
                                              int ng, Group atom) {
    if (threadIdx.x != 0) return;
    const unsigned long long bit = (unsigned long long)t * K + k;
    const unsigned wv = bits[bit >> 5], m = 1u << (bit & 31);
    if (wv & m) {
        st.duplicates += 1;
    } else {
        st.nnz += 1;
        bits[bit >> 5] = wv | m;
    }
    for (int i = 0; i < ng; ++i) {
        const LocompAtom<real> g = atom(i);
        evp[st.n_buffered] = g.t;
        evi[st.n_buffered] = g.k;
        evc[st.n_buffered] = g.x;
        st.n_buffered += 1;
    }
    st.n_events += 1;
}

// The group's residual subtractions, atom by atom (:1341, :996-1016).  Returns the energy loss, summed in the data's
// precision like the reference's energyLoss (meaningful in thread 0).  SYNC_LAST: a barrier after the last atom too.
template <typename real, int NT, bool SYNC_LAST, typename Group>
__device__ __forceinline__ double locomp_subtract(const MpArgs<real>& a, real* res_s, int T, int L, int F, int off, int ng, Group atom,
                                                  double* red_a, double* red_b) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int LF = L * F;
    double loss_sum = 0.0;
    for (int i = 0; i < ng; ++i) {
        const LocompAtom<real> g = atom(i);
        const int si = g.t - off;
        const int jlo = si < 0 ? -si : 0, jhi = (si + L > T) ? (T - si) : L;
        const real* dd = a.D + (long long)g.k * LF;
        real* rr = res_s + (long long)si * F;
        double eb = 0.0, ea = 0.0;
        for (int q = jlo * F + tid; q < jhi * F; q += NT) {
            const real ro = rr[q];
            const real rn = sub_scaled(ro, g.x, dd[q]);
            rr[q] = rn;
            eb = fma((double)ro, (double)ro, eb);
            ea = fma((double)rn, (double)rn, ea);
        }
        eb = warp_sum(eb);
        ea = warp_sum(ea);
        if (lane == 0) { red_b[warp] = eb; red_a[warp] = ea; }
        __syncthreads();
        if (tid == 0) {
            double sb = 0.0, sa = 0.0;
            for (int w = 0; w < NT / 32; ++w) { sb += red_b[w]; sa += red_a[w]; }
            loss_sum = (double)((real)loss_sum + ((real)sb - (real)sa));
        }
        if (SYNC_LAST || i + 1 < ng) __syncthreads();
    }
    return loss_sum;
}

// Stop rules after a selection (:1358-1382), then, where a pass ends or a rule fired, the residual-scale test over the
// n = T * F samples.  Returns true to leave the loop (st.status says why).
template <typename real, int NT>
__device__ __forceinline__ bool locomp_stop_rules(const MpArgs<real>& a, hsc_signal_state& st, int& sel_stop, bool block_mode, bool pass_ends,
                                                  double loss_sum, long long& passes_this_run, const real* res_s, long long n, real* red_m) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        const real e_prev = (real)st.energy_residual;
        const real e_now = e_prev - (real)loss_sum;
        st.energy_residual = (double)e_now;
        if (block_mode) st.pass_cursor += 1;
        int stop = 0;
        if (e_now < a.eps) {
            stop = HSC_STOP_ENERGY;
        } else {
            const real snr = (real)10 * rlog10<real>((real)st.energy_signal / e_now);
            if (a.max_nnz >= 0 && st.nnz >= a.max_nnz) stop = HSC_STOP_NNZ;
            else if (a.has_snr && snr >= a.tol_snr) stop = HSC_STOP_SNR;
            else if (rabs<real>(e_prev - e_now) < a.eps) stop = HSC_STOP_STALL;
            else if (a.max_events_total > 0 && st.n_events >= a.max_events_total) stop = HSC_STOP_MAX_EVENTS;
        }
        if (pass_ends || stop) {
            st.passes += 1;
            st.offset_flag ^= 1;
            if (stop) st.pass_cursor = st.pass_count;
        }
        sel_stop = stop;
    }
    if (pass_ends) ++passes_this_run;
    __syncthreads();
    if (a.has_scale && (pass_ends || sel_stop)) {
        real m = (real)0;
        for (long long e = tid; e < n; e += NT) {
            const real v = rabs<real>(res_s[e]);
            m = v > m ? v : m;
        }
        m = warp_max<real>(m);
        if (lane == 0) red_m[warp] = m;
        __syncthreads();
        if (tid == 0) {
            real mm = (real)0;
            for (int i = 0; i < NT / 32; ++i) mm = red_m[i] > mm ? red_m[i] : mm;
            if (mm <= a.tol_scale && sel_stop == 0) sel_stop = HSC_STOP_SCALE;
        }
        __syncthreads();
    }
    if (sel_stop) {
        if (tid == 0) st.status = sel_stop;
        return true;
    }
    return false;
}

template <typename real, int NT, bool RAGGED = false>       // RAGGED: per-signal lengths (see pursuit_kernel)
__global__ void __launch_bounds__(NT, 512 / NT) locomp_kernel(MpArgs<real> a) {       // 512 threads per SM: 128 registers each
    const int s = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = NT / 32;
    constexpr int NG = kLocompMaxGroup;
    const int T = RAGGED ? a.len[s] : a.T, K = a.K, L = a.L, F = a.F, off = a.off;     // (a.T: the row stride)

    real* map_s = a.map + (long long)s * a.T * K;
    real* res_s = a.resid + (long long)s * a.T * F;
    real* v1 = a.val1 + (long long)s * a.T;
    int* i1 = a.idx1 + (long long)s * a.T;
    real* v2 = a.val2 + (long long)s * a.n2;
    int* i2 = a.idx2 + (long long)s * a.n2;
    real* v3 = a.val3 + (long long)s * a.n3;
    int* i3 = a.idx3 + (long long)s * a.n3;
    unsigned* bits = a.bitmap + (long long)s * a.bitmap_words;
    int* evp = a.ev_pos + (long long)s * a.cap;
    int* evi = a.ev_idx + (long long)s * a.cap;
    real* evc = a.ev_coef + (long long)s * a.cap;
    int* ct = a.cand_t + (long long)s * 2 * a.ncand_max;
    int* ck = a.cand_k + (long long)s * 2 * a.ncand_max;
    real* cc = a.cand_c + (long long)s * 2 * a.ncand_max;

    __shared__ hsc_signal_state st;
    __shared__ struct { int t, k, stop, last, n; real coef; } sel;
    __shared__ int g_t[NG], g_k[NG];
    __shared__ long long g_key[NG];
    __shared__ double g_b[NG], g_x[NG];
    __shared__ double g_As[kLocompSmemGroup][kLocompSmemGroup + 1];
    __shared__ double red_a[NW], red_b[NW];
    __shared__ real red_m[NW];
    __shared__ int s_n, s_bad;
    auto atom = [&](int i) { return LocompAtom<real>{g_t[i], g_k[i], (real)g_x[i]}; };

    if (tid == 0) st = a.state[s];
    __syncthreads();
    if (st.status != HSC_RUNNING && st.status != HSC_PAUSE_CAPACITY && st.status != HSC_PAUSE_PASSES) return;

    if (!st.initialised) {
        locomp_init_state<real, NT>(st, res_s, (long long)T * F, red_a);
        rekey_level<real>(v1, nullptr, T, v2, i2, 0, a.n2 - 1, a.G1, NT);
        __syncthreads();
        rekey_level<real>(v2, i2, a.n2, v3, i3, 0, a.n3 - 1, a.G2, NT);
        __syncthreads();
    }
    if (tid == 0) {
        st.status = HSC_RUNNING;
        st.n_buffered = 0;
    }
    __syncthreads();

    const bool block_mode = a.nb_blocks != 1;
    long long passes_this_run = 0;
    while (true) {
        if (locomp_loop_head<real, NT, RAGGED>(a, st, block_mode, passes_this_run, map_s, res_s, v1, i1, ct, ck, cc)) break;
        // ------------------------------------------------------------------ select
        if (warp == 0) {
            int t, k;
            real coef;
            int last = 1;
            if (block_mode) {
                locomp_pass_pick<real>(a, st, ct, ck, cc, t, k, coef, last);
            } else {
                real bv = (real)0;
                int bt = INT_MAX;
                for (int e = lane; e < a.n3; e += 32) take_first_max(bv, bt, v3[e], i3[e]);
                group_argmax(bv, bt, 32);
                t = bt == INT_MAX ? 0 : bt;                    // all-zero map: np.argmax gives (0, 0), a null coefficient
                k = bt == INT_MAX ? 0 : i1[t];
                coef = locomp_pick_coef<real>(a, res_s, T, L, F, off, t, k, map_s[(long long)t * K + k]);
            }
            if (lane == 0) {
                sel.t = t; sel.k = k; sel.coef = coef; sel.stop = 0; sel.last = last;
                s_n = 1; s_bad = 0;
                g_t[0] = t; g_k[0] = k;
            }
        }
        __syncthreads();
        const int t = sel.t, k = sel.k;
        const real coef = sel.coef;
        const bool pass_ends = sel.last != 0;
        if (locomp_null_stop<real>(a, st, block_mode, coef)) break;
        if (locomp_common_support<NT>(st, bits, t, k, T, K, L, off, g_key, s_n, s_bad)) break;
        const int n = s_n;
        locomp_refit<real, NT, RAGGED>(a, res_s, T, K, L, F, off, n, coef, &g_As[0][0], g_key, g_t, g_k, g_b, g_x, s_n);
        __syncthreads();
        const int ng = s_n;
        locomp_record<real>(st, bits, evp, evi, evc, t, k, K, ng, atom);
        const double loss_sum = locomp_subtract<real, NT, true>(a, res_s, T, L, F, off, ng, atom, red_a, red_b);
        // ------------------------------------------------------------------ map windows of the group (:1353)
        // Interior atoms (no row of the window is "absolute") take the vectorised Gram update of the MP kernel, which
        // also rewrites the level-1 keys of its rows; edge atoms keep the two-phase element-wise path + a re-key.
        // All incremental updates precede all absolute ones (see locomp_window).
        {
            constexpr int VN = VecOf<real>::N;
            const int W = 2 * L - 1;
            const int nvec = (K % VN == 0) ? K / VN : 0;
            const int gv = min(32, pow2_at_least(nvec > 0 ? nvec : 1));
            int vec_pv = 0;
            if (nvec > 0 && !a.w) {
                const int per_lane = (nvec + gv - 1) / gv;
                vec_pv = per_lane <= 1 ? 1 : per_lane <= 2 ? 2 : per_lane <= 4 ? 4 : 0;
            }
            for (int i = 0; i < ng; ++i) {
                const int ti = g_t[i];
                if (!locomp_edge(ti, L, T, off) && vec_pv) {
                    const real* Gk = a.G + (long long)g_k[i] * W * K;
                    if (vec_pv == 1) gram_update_vec<real, 1, NT, 4, false>(K, L, a.w, map_s, Gk, v1, i1, ti, (real)g_x[i], gv);
                    else if (vec_pv == 2) gram_update_vec<real, 2, NT, 4, false>(K, L, a.w, map_s, Gk, v1, i1, ti, (real)g_x[i], gv);
                    else gram_update_vec<real, 4, NT, 4, false>(K, L, a.w, map_s, Gk, v1, i1, ti, (real)g_x[i], gv);
                    __syncthreads();
                } else {
                    locomp_window<real, NT, RAGGED>(a, map_s, res_s, ti, g_k[i], (real)g_x[i], 0);
                }
            }
            for (int i = 0; i < ng; ++i) {
                const int ti = g_t[i];
                if (locomp_edge(ti, L, T, off)) locomp_window<real, NT, RAGGED>(a, map_s, res_s, ti, g_k[i], (real)g_x[i], 1);
            }
            for (int i = 0; i < ng; ++i) {
                const int ti = g_t[i];
                const int row_lo = max(ti - (L - 1), 0), row_hi = min(ti + (L - 1), T - 1);
                if (locomp_edge(ti, L, T, off) || !vec_pv) {
                    rekey_rows(a, map_s, v1, i1, row_lo, row_hi, min(32, pow2_at_least(K)), NT);
                    __syncthreads();
                }
                const int g2_lo = row_lo / a.G1, g2_hi = row_hi / a.G1;
                rekey_level<real>(v1, nullptr, T, v2, i2, g2_lo, g2_hi, a.G1, NT);
                __syncthreads();
                rekey_level<real>(v2, i2, a.n2, v3, i3, g2_lo / a.G2, g2_hi / a.G2, a.G2, NT);
                __syncthreads();
            }
        }
        if (locomp_stop_rules<real, NT>(a, st, sel.stop, block_mode, pass_ends, loss_sum, passes_this_run, res_s, (long long)T * F, red_m)) break;
    }
    __syncthreads();
    if (tid == 0) a.state[s] = st;
}

// ---------------------------------------------------------------------------------------------------------------------
// LoCOMP on the MP kernel's fast path (float maps with wide rows: the config-4 / config-5 shapes).  Same algorithm, same
// arithmetic and the same events as locomp_kernel above, with
//  * the upper levels of the argmax hierarchy in shared memory (select_smh / slot2 / slot3 of pursuit.cuh) instead of three
//    levels in global memory re-keyed with two barriers per group atom,
//  * interior windows through the per-warp bulk-copy pipelines (gram_update_row32), 8 warps per signal, 4 CTAs per SM,
//  * the refit scratch (normal matrix, right-hand side, rank-sort keys) overlaid on the stage rings, which are idle while a
//    group is fitted; the fitted group (t, k, delta) goes to a small per-signal list in global memory for the apply phase.
// Groups that contain an edge atom keep the two-phase element-wise windows (all increments before all re-correlations).
template <typename real, int NT, bool RAGGED = false>       // RAGGED: per-signal lengths (see pursuit_kernel)
__global__ void __launch_bounds__(NT, 4) locomp_fast_kernel(MpArgs<real> a) {
    const int s = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = NT / 32;
    constexpr int NG = kLocompMaxGroup;
    const int Tst = a.T, K = a.K, L = a.L, F = a.F, off = a.off, W = 2 * L - 1;     // Tst: the row stride

    // per-signal base pointers and a ragged signal's length T (which bounds everything below; the arrays keep the row stride
    // Tst) live in shared memory, loaded at the use sites (CtaLength)
    struct Ctx { real* map_s; real* res_s; real* v1; int* i1; unsigned* bits; int* evp; int* evi; real* evc; int* ct; int* ck; real* cc;
                 double* gl_x; int* gl_t; int* gl_k; };
    __shared__ Ctx cx;
    if (tid == 0) {
        cx.map_s = a.map + (long long)s * Tst * K;
        cx.res_s = a.resid + (long long)s * Tst * F;
        cx.v1 = a.val1 + (long long)s * Tst;
        cx.i1 = a.idx1 + (long long)s * Tst;
        cx.bits = a.bitmap + (long long)s * a.bitmap_words;
        cx.evp = a.ev_pos + (long long)s * a.cap;
        cx.evi = a.ev_idx + (long long)s * a.cap;
        cx.evc = a.ev_coef + (long long)s * a.cap;
        cx.ct = a.cand_t ? a.cand_t + (long long)s * 2 * a.ncand_max : nullptr;
        cx.ck = a.cand_k ? a.cand_k + (long long)s * 2 * a.ncand_max : nullptr;
        cx.cc = a.cand_c ? a.cand_c + (long long)s * 2 * a.ncand_max : nullptr;
        cx.gl_x = a.locomp_scratch + (long long)s * kLocompScratchStride + (long long)NG * (NG + 1);
        cx.gl_t = reinterpret_cast<int*>(cx.gl_x + NG);
        cx.gl_k = cx.gl_t + NG;
        if constexpr (RAGGED) CtaLength<true>::set(a.len[s]);
    }
#define T (CtaLength<RAGGED>::get(Tst))
#define map_s (cx.map_s)
#define res_s (cx.res_s)
#define v1 (cx.v1)
#define i1 (cx.i1)
#define bits (cx.bits)

    __shared__ hsc_signal_state st;
    __shared__ struct { int t, k, stop, last; real coef; } sel;
    __shared__ int sel_out[5];                                   // select_smh's result
    __shared__ double red_a[NW], red_b[NW];
    __shared__ real red_m[NW];
    __shared__ int s_n, s_bad, s_edge;
    constexpr int NSL = 8;                                       // the first atoms of a group: list in shared memory (most groups fit)
    __shared__ int sl_t[NSL], sl_k[NSL];
    __shared__ real sl_x[NSL];
    extern __shared__ __align__(128) unsigned char win_smem[];
    __shared__ __align__(8) unsigned long long win_bar[NW * 4];
    __shared__ unsigned long long dirty_slot[kDirtyMax];
    unsigned win_phase = 0;
    unsigned long long* slot2 = reinterpret_cast<unsigned long long*>(win_smem + a.tma_bytes);
    unsigned* slot3 = reinterpret_cast<unsigned*>(slot2 + a.n2);
    const int g1s = 31 - __clz(a.G1);
    // refit scratch on the stage rings
    double* g_As = reinterpret_cast<double*>(win_smem);
    long long* g_key = reinterpret_cast<long long*>(win_smem + kLocompSmemGroup * (kLocompSmemGroup + 1) * 8);
    double* g_b = reinterpret_cast<double*>(g_key + NG);
    double* g_x = g_b + NG;
    int* g_t = reinterpret_cast<int*>(g_x + NG);
    int* g_k = g_t + NG;
    // the fitted group once it has left the rings
    auto atom = [&](int i) {
        return i < NSL ? LocompAtom<real>{sl_t[i], sl_k[i], sl_x[i]} : LocompAtom<real>{cx.gl_t[i], cx.gl_k[i], (real)cx.gl_x[i]};
    };

    if (tid == 0) {
        st = a.state[s];
        for (int i = 0; i < NW * a.tma_stages; ++i) mbarrier_init(smem_addr_u32(&win_bar[i]), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        fence_proxy_async_all();
    }
    __syncthreads();
    if (st.status != HSC_RUNNING && st.status != HSC_PAUSE_CAPACITY && st.status != HSC_PAUSE_PASSES) return;

    if (!st.initialised) locomp_init_state<real, NT>(st, res_s, (long long)T * F, red_a);
    // (re)build the shared-memory levels from the level-1 keys in global memory: first launch and resumes alike
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
    if (tid == 0) {
        st.status = HSC_RUNNING;
        st.n_buffered = 0;
    }
    __syncthreads();

    const bool block_mode = a.nb_blocks != 1;
    long long passes_this_run = 0;
    while (true) {
        if (locomp_loop_head<real, NT, RAGGED>(a, st, block_mode, passes_this_run, map_s, res_s, v1, i1, cx.ct, cx.ck, cx.cc)) break;
        // ------------------------------------------------------------------ select
        if (warp == 0) {
            int t, k;
            real coef;
            int last = 1;
            if (block_mode) {
                locomp_pass_pick<real>(a, st, cx.ct, cx.ck, cx.cc, t, k, coef, last);
            } else {
                select_smh(smem_addr_u32(slot2), smem_addr_u32(slot3), a.n2, K, g1s, sel_out);
                __syncwarp();
                t = sel_out[0] < 0 ? 0 : sel_out[0];           // all-zero map: np.argmax gives (0, 0), a null coefficient
                k = sel_out[0] < 0 ? 0 : sel_out[1];
                coef = locomp_pick_coef<real>(a, res_s, T, L, F, off, t, k, __ldcg(map_s + (long long)t * K + k));
            }
            if (lane == 0) {
                sel.t = t; sel.k = k; sel.coef = coef; sel.stop = 0; sel.last = last;
                s_n = 1; s_bad = 0; s_edge = 0;
                g_t[0] = t; g_k[0] = k;
            }
        }
        __syncthreads();
        const int t = sel.t, k = sel.k;
        const real coef = sel.coef;
        const bool pass_ends = sel.last != 0;
        if (locomp_null_stop<real>(a, st, block_mode, coef)) break;
        if (locomp_common_support<NT>(st, bits, t, k, T, K, L, off, g_key, s_n, s_bad)) break;
        const int n = s_n;
        locomp_refit<real, NT, RAGGED>(a, res_s, T, K, L, F, off, n, coef, g_As, g_key, g_t, g_k, g_b, g_x, s_n);
        if (n > 1) __syncthreads();             // (a lone atom: thread 0 wrote g_x[0] and writes the list entry itself below)
        const int ng = n > 1 ? s_n : 1;
        // the fitted group leaves the stage rings: list in global memory, edge flag
        for (int i = tid; i < ng; i += NT) {
            const int ti = g_t[i];
            if (i < NSL) {
                sl_t[i] = ti; sl_k[i] = g_k[i]; sl_x[i] = (real)g_x[i];
            } else {
                cx.gl_t[i] = ti; cx.gl_k[i] = g_k[i]; cx.gl_x[i] = g_x[i];
            }
            if (locomp_edge(ti, L, T, off)) s_edge = 1;
        }
        fence_proxy_async_smem();               // generic writes to the rings, then bulk copies into them
        __syncthreads();
        const bool any_edge = s_edge != 0;
        locomp_record<real>(st, bits, cx.evp, cx.evi, cx.evc, t, k, K, ng, atom);
        const double loss_sum = locomp_subtract<real, NT, false>(a, res_s, T, L, F, off, ng, atom, red_a, red_b);
        // ------------------------------------------------------------------ map windows of the group (:1353)
        for (int i = 0; i < ng; ++i) {
            const LocompAtom<real> g = atom(i);
            const int ti = g.t;
            if (locomp_edge(ti, L, T, off)) {
                locomp_window<real, NT, RAGGED>(a, map_s, res_s, ti, g.k, g.x, 0);       // increments on the rows that are not re-correlated
                fence_proxy_async_all();            // generic map writes -> later bulk loads of these rows
                __syncthreads();
                continue;
            }
            const int row_lo = ti - (L - 1), row_hi = ti + (L - 1);
            const int g2_lo = row_lo >> g1s, g2_hi = row_hi >> g1s;
            {   // rows of the touched groups outside the window: their level-1 keys are unchanged
                const int span0 = g2_lo << g1s, span1 = min((g2_hi + 1) << g1s, T);
                for (int r0 = span0 + warp * 32; r0 < span1; r0 += NT) {
                    const int r = r0 + lane;
                    unsigned long long key = 0ull;
                    if (r < span1 && (r < row_lo || r > row_hi)) key = pack_key(v1[r], r & (a.G1 - 1), i1[r], K);
                    key = warp_max_u64(key);
                    if (lane == 0 && key) atomicMax(&dirty_slot[(r0 >> g1s) - g2_lo], key);
                }
            }
            const real* Gk = a.G + (long long)g.k * W * K;
            gram_window_issue<real, NT, 1>(K, L, map_s, Gk, ti, 32, win_smem, win_bar, a.tma_stages);
            win_phase = gram_update_row32<real, NT, true>(K, L, map_s, Gk, v1, i1, ti, g.x, win_smem, win_bar, a.tma_stages, win_phase, dirty_slot, g2_lo, g1s);
            __syncthreads();
            if (warp == 1) {                        // publish the rebuilt groups, re-arm the scratch keys, refresh their blocks
                if (lane <= g2_hi - g2_lo) {
                    slot2[g2_lo + lane] = dirty_slot[lane];
                    dirty_slot[lane] = 0ull;
                }
                __syncwarp();
                for (int b = g2_lo >> 5; b <= g2_hi >> 5; ++b) refold_block(slot2, slot3, b, a.n2);
            }
            if (elect_one_sync()) {                 // this warp's bulk stores: complete, and ordered before later generic reads / bulk loads
                bulk_wait_all();
                fence_proxy_async_all();
            }
            __syncthreads();
        }
        if (any_edge) {
            for (int i = 0; i < ng; ++i) {
                const LocompAtom<real> g = atom(i);
                if (locomp_edge(g.t, L, T, off)) locomp_window<real, NT, RAGGED>(a, map_s, res_s, g.t, g.k, g.x, 1);
            }
            fence_proxy_async_all();
            __syncthreads();
            for (int i = 0; i < ng; ++i) {
                const int ti = atom(i).t;
                if (!locomp_edge(ti, L, T, off)) continue;
                const int row_lo = max(ti - (L - 1), 0), row_hi = min(ti + (L - 1), T - 1);
                const int g2_lo = row_lo >> g1s, g2_hi = row_hi >> g1s;
                const int span0 = g2_lo << g1s, span1 = min((g2_hi + 1) << g1s, T);
                for (int r0 = span0 + warp * 32; r0 < span1; r0 += NT) {
                    const int r = r0 + lane;
                    unsigned long long key = 0ull;
                    if (r < span1 && (r < row_lo || r > row_hi)) key = pack_key(v1[r], r & (a.G1 - 1), i1[r], K);
                    key = warp_max_u64(key);
                    if (lane == 0 && key) atomicMax(&dirty_slot[(r0 >> g1s) - g2_lo], key);
                }
                rekey_rows(a, map_s, v1, i1, row_lo, row_hi, 32, NT, dirty_slot, g2_lo, g1s);
                __syncthreads();
                if (warp == 1) {
                    if (lane <= g2_hi - g2_lo) {
                        slot2[g2_lo + lane] = dirty_slot[lane];
                        dirty_slot[lane] = 0ull;
                    }
                    __syncwarp();
                    for (int b = g2_lo >> 5; b <= g2_hi >> 5; ++b) refold_block(slot2, slot3, b, a.n2);
                }
                __syncthreads();
            }
        }
        if (locomp_stop_rules<real, NT>(a, st, sel.stop, block_mode, pass_ends, loss_sum, passes_this_run, res_s, (long long)T * F, red_m)) break;
    }
    __syncthreads();
    if (tid == 0) a.state[s] = st;
#undef T
#undef map_s
#undef res_s
#undef v1
#undef i1
#undef bits
}

}  // namespace hsc
