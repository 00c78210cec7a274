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
constexpr int HSC_STOP_STALL_ = 9;        // |delta E| < eps (:1377-1381)
constexpr int HSC_STOP_GROUP_ = 10;       // common-support group larger than kLocompMaxGroup

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

template <typename real, int NT, bool RAGGED = false>       // RAGGED: per-signal lengths (see pursuit_kernel)
__global__ void __launch_bounds__(NT, 512 / NT) locomp_kernel(MpArgs<real> a) {       // 512 threads per SM: 128 registers each
    const int s = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = NT / 32;
    constexpr int NG = kLocompMaxGroup;
    const int T = RAGGED ? a.len[s] : a.T, K = a.K, L = a.L, F = a.F, off = a.off, LF = L * F;     // (a.T: the row stride)

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
    // normal matrix of the current group: shared memory for n <= 64, else this signal's slice of the engine's scratch
    double* g_Ap = &g_As[0][0];
    int g_pitch = kLocompSmemGroup + 1;
#define g_A(i, j) g_Ap[(long long)(i) * g_pitch + (j)]
    __shared__ double red_a[NW], red_b[NW];
    __shared__ real red_m[NW];
    __shared__ int s_n, s_bad;

    if (tid == 0) st = a.state[s];
    __syncthreads();
    if (st.status != HSC_RUNNING && st.status != HSC_PAUSE_CAPACITY && st.status != HSC_PAUSE_PASSES) return;

    if (!st.initialised) {
        double acc = 0.0;
        for (long long e = tid; e < (long long)T * F; e += NT) {
            const double v = (double)res_s[e];
            acc = fma(v, v, acc);
        }
        acc = warp_sum(acc);
        if (lane == 0) red_a[warp] = acc;
        __syncthreads();
        if (tid == 0) {
            double tot = 0.0;
            for (int i = 0; i < NW; ++i) tot += red_a[i];
            const real es = (real)tot;
            st.energy_signal = (double)es;
            st.energy_residual = (double)es;
            st.n_events = st.nnz = st.duplicates = st.passes = 0;
            st.offset_flag = 0;
            st.pass_count = 0;
            st.pass_cursor = 0;
            st.initialised = 1;
        }
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
        if (st.n_buffered + NG > a.cap) {                     // a selection may emit up to NG events
            if (tid == 0) st.status = HSC_PAUSE_CAPACITY;
            break;
        }
        const bool new_pass = !block_mode || st.pass_cursor >= st.pass_count;
        if (new_pass && a.max_passes > 0 && passes_this_run >= a.max_passes) {
            if (tid == 0) st.status = HSC_PAUSE_PASSES;
            break;
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
                break;
            }
        }
        // ------------------------------------------------------------------ select
        if (warp == 0) {
            int t, k;
            real coef;
            int last = 1;
            if (block_mode) {
                const int cur = st.pass_cursor;
                t = ct[a.ncand_max + cur];
                k = ck[a.ncand_max + cur];
                coef = cc[a.ncand_max + cur];
                last = (cur + 1 >= st.pass_count);
            } else {
                real bv = (real)0;
                int bt = INT_MAX;
                for (int e = lane; e < a.n3; e += 32) take_first_max(bv, bt, v3[e], i3[e]);
                group_argmax(bv, bt, 32);
                t = bt == INT_MAX ? 0 : bt;                    // all-zero map: np.argmax gives (0, 0), a null coefficient
                k = bt == INT_MAX ? 0 : i1[t];
                coef = map_s[(long long)t * K + k];
                const int edge = (t - (L - 1) < off) || (t + (L - 1) > T - L + off);
                if (a.coef_mode == 1 && !edge) {
                    const real* rr = res_s + (long long)(t - off) * F;
                    const real* dd = a.D + (long long)k * LF;
                    double acc = 0.0;
                    for (int q = lane; q < LF; q += 32) acc = fma((double)rr[q], (double)dd[q], acc);
                    acc = warp_sum(acc);
                    coef = (real)acc;
                }
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
        const bool is_null = (a.null_thres >= (real)0) ? !(rabs<real>(coef) > a.null_thres) : (coef == (real)0);
        if (!block_mode && is_null) {
            if (tid == 0) {
                st.passes += 1;
                st.status = HSC_STOP_EMPTY;
            }
            break;
        }

        // ------------------------------------------------------------------ common-support atoms (:1221-1239)
        {
            const int sp0 = max(t - off, 0), ep0 = min(t + L / 2, T - 1);           // Atom.getPositionSpanIndices (:845-858)
            const int lo = max(sp0 - L / 2, 0);
            const int hi = min(min(ep0 + ((L % 2 == 0) ? L / 2 - 1 : L / 2), T), T - 1);
            const long long b0 = (long long)lo * K, b1 = (long long)(hi + 1) * K;   // bit range [b0, b1)
            for (long long wI = (b0 >> 5) + tid; wI <= ((b1 - 1) >> 5); wI += NT) {
                unsigned wv = bits[wI];
                while (wv) {
                    const int bpos = __ffs(wv) - 1;
                    wv &= wv - 1;
                    const long long bit = (wI << 5) + bpos;
                    if (bit < b0 || bit >= b1) continue;
                    const int tt = (int)(bit / K), kk = (int)(bit - (long long)tt * K);
                    if ((tt - lo) != t && kk != k) {                                 // the reference's predicate, as written (:1238)
                        const int slot = atomicAdd(&s_n, 1);
                        if (slot < NG) {
                            g_key[slot] = bit;
                        } else {
                            s_bad = 1;
                        }
                    }
                }
            }
        }
        __syncthreads();
        if (s_bad) {
            if (tid == 0) st.status = HSC_STOP_GROUP_;
            break;
        }
        const int n = s_n;
        if (n > kLocompSmemGroup) {
            g_Ap = a.locomp_scratch + (long long)s * kLocompScratchStride;
            g_pitch = kLocompMaxGroup + 1;
        } else {
            g_Ap = &g_As[0][0];
            g_pitch = kLocompSmemGroup + 1;
        }
        if (n > 1) {
            // row-major order of the neighbours (COO of the LIL slice): rank sort of the keys
            for (int i = tid; i < n; i += NT) {
                if (i < 1) continue;
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
                    g_A(i, j) = v;
                    g_A(j, i) = v;
                }
            }
            __syncthreads();
            // Cholesky A = L L^T, then two triangular solves (float64, warp 0)
            if (warp == 0) {
                bool ok = true;
                double dmax = 0.0;
                for (int i = lane; i < n; i += 32) dmax = fmax(dmax, g_A(i, i));
                for (int m = 16; m > 0; m >>= 1) dmax = fmax(dmax, __shfl_xor_sync(0xffffffffu, dmax, m));
                for (int j = 0; j < n; ++j) {
                    double d = g_A(j, j);
                    for (int p = 0; p < j; ++p) d -= g_A(j, p) * g_A(j, p);      // all lanes compute the same scalar
                    if (!(d > 1e-13 * dmax)) { ok = false; break; }
                    const double ljj = sqrt(d);
                    __syncwarp();
                    for (int i = j + 1 + lane; i < n; i += 32) {
                        double v = g_A(i, j);
                        for (int p = 0; p < j; ++p) v -= g_A(i, p) * g_A(j, p);
                        g_A(i, j) = v / ljj;
                    }
                    if (lane == 0) g_A(j, j) = ljj;
                    __syncwarp();
                }
                if (ok && lane == 0) {
                    for (int i = 0; i < n; ++i) {                                    // L y = b
                        double v = g_b[i];
                        for (int p = 0; p < i; ++p) v -= g_A(i, p) * g_x[p];
                        g_x[i] = v / g_A(i, i);
                    }
                    for (int i = n - 1; i >= 0; --i) {                               // L^T x = y
                        double v = g_x[i];
                        for (int p = i + 1; p < n; ++p) v -= g_A(p, i) * g_x[p];
                        g_x[i] = v / g_A(i, i);
                    }
                }
                if (lane == 0 && !ok) {          // numerically dependent support: plain MP step for this atom
                    s_n = 1;
                    g_x[0] = (double)coef;
                }
            }
        } else if (tid == 0) {
            g_x[0] = (double)coef;
        }
        __syncthreads();
        const int ng = s_n;

        // ------------------------------------------------------------------ code bookkeeping + events
        if (tid == 0) {
            const unsigned long long bit = (unsigned long long)t * K + k;
            const unsigned wv = bits[bit >> 5], m = 1u << (bit & 31);
            if (wv & m) {
                st.duplicates += 1;                 // 'Redundant atom selected' (:1314-1315)
            } else {
                st.nnz += 1;
                bits[bit >> 5] = wv | m;
            }
            for (int i = 0; i < ng; ++i) {
                evp[st.n_buffered] = g_t[i];
                evi[st.n_buffered] = g_k[i];
                evc[st.n_buffered] = (real)g_x[i];
                st.n_buffered += 1;
            }
            st.n_events += 1;
        }
        // ------------------------------------------------------------------ residual, atom by atom (:1341, :996-1016)
        double loss_sum = 0.0;                      // meaningful in thread 0
        for (int i = 0; i < ng; ++i) {
            const int si = g_t[i] - off;
            const int jlo = si < 0 ? -si : 0, jhi = (si + L > T) ? (T - si) : L;
            const real ci = (real)g_x[i];
            const real* dd = a.D + (long long)g_k[i] * LF;
            real* rr = res_s + (long long)si * F;
            double eb = 0.0, ea = 0.0;
            for (int q = jlo * F + tid; q < jhi * F; q += NT) {
                const real ro = rr[q];
                const real rn = sub_scaled(ro, ci, dd[q]);
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
                for (int w = 0; w < NW; ++w) { sb += red_b[w]; sa += red_a[w]; }
                loss_sum = (double)((real)loss_sum + ((real)sb - (real)sa));       // energyLoss += before - after, in the data's precision
            }
            __syncthreads();
        }
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
                const bool edge_i = (ti - (L - 1) < off) || (ti + (L - 1) > T - L + off);
                if (!edge_i && vec_pv) {
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
                const bool edge_i = (ti - (L - 1) < off) || (ti + (L - 1) > T - L + off);
                if (edge_i) locomp_window<real, NT, RAGGED>(a, map_s, res_s, ti, g_k[i], (real)g_x[i], 1);
            }
            for (int i = 0; i < ng; ++i) {
                const int ti = g_t[i];
                const bool edge_i = (ti - (L - 1) < off) || (ti + (L - 1) > T - L + off);
                const int row_lo = max(ti - (L - 1), 0), row_hi = min(ti + (L - 1), T - 1);
                if (edge_i || !vec_pv) {
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
        // ------------------------------------------------------------------ stop rules (:1358-1382)
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
                else if (rabs<real>(e_prev - e_now) < a.eps) stop = HSC_STOP_STALL_;
                else if (a.max_events_total > 0 && st.n_events >= a.max_events_total) stop = HSC_STOP_MAX_EVENTS;
            }
            if (pass_ends || stop) {
                st.passes += 1;
                st.offset_flag ^= 1;
                if (stop) st.pass_cursor = st.pass_count;
            }
            sel.stop = stop;
        }
        if (pass_ends) ++passes_this_run;
        __syncthreads();
        if (a.has_scale && (pass_ends || sel.stop)) {
            real m = (real)0;
            for (long long e = tid; e < (long long)T * F; e += NT) {
                const real v = rabs<real>(res_s[e]);
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
            __syncthreads();
        }
        if (sel.stop) {
            if (tid == 0) st.status = sel.stop;
            break;
        }
    }
    __syncthreads();
    if (tid == 0) a.state[s] = st;
#undef g_A
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
    const int Tst = a.T, K = a.K, L = a.L, F = a.F, off = a.off, LF = L * F, W = 2 * L - 1;     // Tst: the row stride

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
    double* g_Ap = g_As;
    int g_pitch = kLocompSmemGroup + 1;
#define g_A(i, j) g_Ap[(long long)(i) * g_pitch + (j)]
#define GL_T(i) ((i) < NSL ? sl_t[i] : cx.gl_t[i])
#define GL_K(i) ((i) < NSL ? sl_k[i] : cx.gl_k[i])
#define GL_X(i) ((i) < NSL ? sl_x[i] : (real)cx.gl_x[i])

    if (tid == 0) {
        st = a.state[s];
        for (int i = 0; i < NW * a.tma_stages; ++i) mbarrier_init(smem_addr_u32(&win_bar[i]), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        fence_proxy_async_all();
    }
    __syncthreads();
    if (st.status != HSC_RUNNING && st.status != HSC_PAUSE_CAPACITY && st.status != HSC_PAUSE_PASSES) return;

    if (!st.initialised) {
        double acc = 0.0;
        for (long long e = tid; e < (long long)T * F; e += NT) {
            const double v = (double)res_s[e];
            acc = fma(v, v, acc);
        }
        acc = warp_sum(acc);
        if (lane == 0) red_a[warp] = acc;
        __syncthreads();
        if (tid == 0) {
            double tot = 0.0;
            for (int i = 0; i < NW; ++i) tot += red_a[i];
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
        if (st.n_buffered + NG > a.cap) {                     // a selection may emit up to NG events
            if (tid == 0) st.status = HSC_PAUSE_CAPACITY;
            break;
        }
        const bool new_pass = !block_mode || st.pass_cursor >= st.pass_count;
        if (new_pass && a.max_passes > 0 && passes_this_run >= a.max_passes) {
            if (tid == 0) st.status = HSC_PAUSE_PASSES;
            break;
        }
        if (block_mode && new_pass) {
            const int n = build_pass_list<real, NT, RAGGED>(a, map_s, res_s, v1, i1, cx.ct, cx.ck, cx.cc, st.offset_flag, st.energy_signal);
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
                break;
            }
        }
        // ------------------------------------------------------------------ select
        if (warp == 0) {
            int t, k;
            real coef;
            int last = 1;
            if (block_mode) {
                const int cur = st.pass_cursor;
                t = cx.ct[a.ncand_max + cur];
                k = cx.ck[a.ncand_max + cur];
                coef = cx.cc[a.ncand_max + cur];
                last = (cur + 1 >= st.pass_count);
            } else {
                select_smh(smem_addr_u32(slot2), smem_addr_u32(slot3), a.n2, K, g1s, sel_out);
                __syncwarp();
                t = sel_out[0] < 0 ? 0 : sel_out[0];           // all-zero map: np.argmax gives (0, 0), a null coefficient
                k = sel_out[0] < 0 ? 0 : sel_out[1];
                coef = __ldcg(map_s + (long long)t * K + k);
                const int edge = (t - (L - 1) < off) || (t + (L - 1) > T - L + off);
                if (a.coef_mode == 1 && !edge) {
                    const real* rr = res_s + (long long)(t - off) * F;
                    const real* dd = a.D + (long long)k * LF;
                    double acc = 0.0;
                    for (int q = lane; q < LF; q += 32) acc = fma((double)rr[q], (double)dd[q], acc);
                    acc = warp_sum(acc);
                    coef = (real)acc;
                }
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
        const bool is_null = (a.null_thres >= (real)0) ? !(rabs<real>(coef) > a.null_thres) : (coef == (real)0);
        if (!block_mode && is_null) {
            if (tid == 0) {
                st.passes += 1;
                st.status = HSC_STOP_EMPTY;
            }
            break;
        }

        // ------------------------------------------------------------------ common-support atoms (:1221-1239)
        {
            const int sp0 = max(t - off, 0), ep0 = min(t + L / 2, T - 1);           // Atom.getPositionSpanIndices (:845-858)
            const int lo = max(sp0 - L / 2, 0);
            const int hi = min(min(ep0 + ((L % 2 == 0) ? L / 2 - 1 : L / 2), T), T - 1);
            const long long b0 = (long long)lo * K, b1 = (long long)(hi + 1) * K;   // bit range [b0, b1)
            for (long long wI = (b0 >> 5) + tid; wI <= ((b1 - 1) >> 5); wI += NT) {
                unsigned wv = bits[wI];
                while (wv) {
                    const int bpos = __ffs(wv) - 1;
                    wv &= wv - 1;
                    const long long bit = (wI << 5) + bpos;
                    if (bit < b0 || bit >= b1) continue;
                    const int tt = (int)(bit / K), kk = (int)(bit - (long long)tt * K);
                    if ((tt - lo) != t && kk != k) {                                 // the reference's predicate, as written (:1238)
                        const int slot = atomicAdd(&s_n, 1);
                        if (slot < NG) g_key[slot] = bit;
                        else s_bad = 1;
                    }
                }
            }
        }
        __syncthreads();
        if (s_bad) {
            if (tid == 0) st.status = HSC_STOP_GROUP_;
            break;
        }
        const int n = s_n;
        if (n > kLocompSmemGroup) {
            g_Ap = a.locomp_scratch + (long long)s * kLocompScratchStride;
            g_pitch = kLocompMaxGroup + 1;
        } else {
            g_Ap = g_As;
            g_pitch = kLocompSmemGroup + 1;
        }
        if (n > 1) {
            // row-major order of the neighbours (COO of the LIL slice): rank sort of the keys
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
                    g_A(i, j) = v;
                    g_A(j, i) = v;
                }
            }
            __syncthreads();
            // Cholesky A = L L^T, then two triangular solves (float64, warp 0)
            if (warp == 0) {
                bool ok = true;
                double dmax = 0.0;
                for (int i = lane; i < n; i += 32) dmax = fmax(dmax, g_A(i, i));
                for (int m = 16; m > 0; m >>= 1) dmax = fmax(dmax, __shfl_xor_sync(0xffffffffu, dmax, m));
                for (int j = 0; j < n; ++j) {
                    double d = g_A(j, j);
                    for (int p = 0; p < j; ++p) d -= g_A(j, p) * g_A(j, p);      // all lanes compute the same scalar
                    if (!(d > 1e-13 * dmax)) { ok = false; break; }
                    const double ljj = sqrt(d);
                    __syncwarp();
                    for (int i = j + 1 + lane; i < n; i += 32) {
                        double v = g_A(i, j);
                        for (int p = 0; p < j; ++p) v -= g_A(i, p) * g_A(j, p);
                        g_A(i, j) = v / ljj;
                    }
                    if (lane == 0) g_A(j, j) = ljj;
                    __syncwarp();
                }
                if (ok && lane == 0) {
                    for (int i = 0; i < n; ++i) {                                    // L y = b
                        double v = g_b[i];
                        for (int p = 0; p < i; ++p) v -= g_A(i, p) * g_x[p];
                        g_x[i] = v / g_A(i, i);
                    }
                    for (int i = n - 1; i >= 0; --i) {                               // L^T x = y
                        double v = g_x[i];
                        for (int p = i + 1; p < n; ++p) v -= g_A(p, i) * g_x[p];
                        g_x[i] = v / g_A(i, i);
                    }
                }
                if (lane == 0 && !ok) {          // numerically dependent support: plain MP step for this atom
                    s_n = 1;
                    g_x[0] = (double)coef;
                }
            }
        } else if (tid == 0) {
            g_x[0] = (double)coef;
        }
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
            if ((ti - (L - 1) < off) || (ti + (L - 1) > T - L + off)) s_edge = 1;
        }
        fence_proxy_async_smem();               // generic writes to the rings, then bulk copies into them
        __syncthreads();
        const bool any_edge = s_edge != 0;

        // ------------------------------------------------------------------ code bookkeeping + events
        if (tid == 0) {
            const unsigned long long bit = (unsigned long long)t * K + k;
            const unsigned wv = bits[bit >> 5], m = 1u << (bit & 31);
            if (wv & m) {
                st.duplicates += 1;                 // 'Redundant atom selected' (:1314-1315)
            } else {
                st.nnz += 1;
                bits[bit >> 5] = wv | m;
            }
            for (int i = 0; i < ng; ++i) {
                cx.evp[st.n_buffered] = GL_T(i);
                cx.evi[st.n_buffered] = GL_K(i);
                cx.evc[st.n_buffered] = GL_X(i);
                st.n_buffered += 1;
            }
            st.n_events += 1;
        }
        // ------------------------------------------------------------------ residual, atom by atom (:1341, :996-1016)
        double loss_sum = 0.0;                      // meaningful in thread 0
        for (int i = 0; i < ng; ++i) {
            const int si = GL_T(i) - off;
            const int jlo = si < 0 ? -si : 0, jhi = (si + L > T) ? (T - si) : L;
            const real ci = GL_X(i);
            const real* dd = a.D + (long long)GL_K(i) * LF;
            real* rr = res_s + (long long)si * F;
            double eb = 0.0, ea = 0.0;
            for (int q = jlo * F + tid; q < jhi * F; q += NT) {
                const real ro = rr[q];
                const real rn = sub_scaled(ro, ci, dd[q]);
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
                for (int w = 0; w < NW; ++w) { sb += red_b[w]; sa += red_a[w]; }
                loss_sum = (double)((real)loss_sum + ((real)sb - (real)sa));       // energyLoss += before - after, in the data's precision
            }
            if (i + 1 < ng) __syncthreads();
        }
        // ------------------------------------------------------------------ map windows of the group (:1353)
        for (int i = 0; i < ng; ++i) {
            const int ti = GL_T(i), ki = GL_K(i);
            const real ci = GL_X(i);
            const bool edge_i = (ti - (L - 1) < off) || (ti + (L - 1) > T - L + off);
            if (edge_i) {
                locomp_window<real, NT, RAGGED>(a, map_s, res_s, ti, ki, ci, 0);         // increments on the rows that are not re-correlated
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
            const real* Gk = a.G + (long long)ki * W * K;
            gram_window_issue<real, NT, 1>(K, L, map_s, Gk, ti, 32, win_smem, win_bar, a.tma_stages);
            win_phase = gram_update_row32<real, NT, true>(K, L, map_s, Gk, v1, i1, ti, ci, win_smem, win_bar, a.tma_stages, win_phase, dirty_slot, g2_lo, g1s);
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
                const int ti = GL_T(i);
                if ((ti - (L - 1) < off) || (ti + (L - 1) > T - L + off)) locomp_window<real, NT, RAGGED>(a, map_s, res_s, ti, GL_K(i), GL_X(i), 1);
            }
            fence_proxy_async_all();
            __syncthreads();
            for (int i = 0; i < ng; ++i) {
                const int ti = GL_T(i);
                if (!((ti - (L - 1) < off) || (ti + (L - 1) > T - L + off))) continue;
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
        // ------------------------------------------------------------------ stop rules (:1358-1382)
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
                else if (rabs<real>(e_prev - e_now) < a.eps) stop = HSC_STOP_STALL_;
                else if (a.max_events_total > 0 && st.n_events >= a.max_events_total) stop = HSC_STOP_MAX_EVENTS;
            }
            if (pass_ends || stop) {
                st.passes += 1;
                st.offset_flag ^= 1;
                if (stop) st.pass_cursor = st.pass_count;
            }
            sel.stop = stop;
        }
        if (pass_ends) ++passes_this_run;
        __syncthreads();
        if (a.has_scale && (pass_ends || sel.stop)) {
            real m = (real)0;
            for (long long e = tid; e < (long long)T * F; e += NT) {
                const real v = rabs<real>(res_s[e]);
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
            __syncthreads();
        }
        if (sel.stop) {
            if (tid == 0) st.status = sel.stop;
            break;
        }
    }
    __syncthreads();
    if (tid == 0) a.state[s] = st;
#undef g_A
#undef GL_T
#undef GL_K
#undef GL_X
#undef T
#undef map_s
#undef res_s
#undef v1
#undef i1
#undef bits
}

}  // namespace hsc
