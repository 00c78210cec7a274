// Event-buffer compaction: the pursuit kernels write each signal's atoms into its own slice [s][capacity] of the event
// buffers; what leaves the device (device-to-host read of the codes, NCCL gather of the sparse codes, SURVEY 8e) is the
// flat list of the n_buffered[s] atoms of every signal in signal order, 12-16 bytes per atom instead of the padded slices.
#pragma once
#include "common.cuh"

namespace hsc {
namespace events {

// offsets[s] = sum_{s' < s} count(s'), offsets[S] = total.  One block of 1024 threads; S <= 65535 signals.
template <typename Count>
__device__ __forceinline__ void exclusive_offsets(const Count& count, int S, long long* __restrict__ offsets) {
    __shared__ long long warp_tot[32];
    __shared__ long long carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < S; base += 1024) {
        const int s = base + tid;
        const long long n = s < S ? count(s) : 0;
        long long incl = n;                                       // inclusive scan inside the warp
        for (int d = 1; d < 32; d <<= 1) {
            const long long o = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += o;
        }
        if (lane == 31) warp_tot[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            long long w = warp_tot[lane];
            for (int d = 1; d < 32; d <<= 1) {
                const long long o = __shfl_up_sync(0xffffffffu, w, d);
                if (lane >= d) w += o;
            }
            warp_tot[lane] = w;                                   // inclusive totals of the warps
        }
        __syncthreads();
        const long long before = carry + (warp > 0 ? warp_tot[warp - 1] : 0) + (incl - n);
        if (s < S) offsets[s] = before;
        __syncthreads();
        if (tid == 1023) carry = before + n;
        __syncthreads();
    }
    if (tid == 0) offsets[S] = carry;
}

struct BufferedCount {
    const hsc_signal_state* states;
    __device__ long long operator()(int s) const { return states[s].n_buffered; }
};

struct ArrayCount {
    const long long* n;
    __device__ long long operator()(int s) const { return n[s]; }
};

__global__ void __launch_bounds__(1024) offsets_kernel(const hsc_signal_state* __restrict__ states, int S, long long* __restrict__ offsets) {
    exclusive_offsets(BufferedCount{states}, S, offsets);
}

// Block j: offsets[j][S+1] from counts[j][S] (the per-level offsets of canonical_codes_kernel).
__global__ void __launch_bounds__(1024) level_offsets_kernel(const long long* __restrict__ counts, int S, long long* __restrict__ offsets) {
    exclusive_offsets(ArrayCount{counts + (long long)blockIdx.x * S}, S, offsets + (long long)blockIdx.x * (S + 1));
}

// One block per signal: its events to their place in the flat arrays (atoms past out_capacity are dropped; the caller
// compares offsets[S] with out_capacity).
template <typename real>
__global__ void __launch_bounds__(256) compact_kernel(const int* __restrict__ evp, const int* __restrict__ evi, const real* __restrict__ evc,
                                                      long long cap, const long long* __restrict__ offsets, int* __restrict__ pos,
                                                      int* __restrict__ idx, real* __restrict__ coef, long long out_capacity) {
    const long long s = blockIdx.x;
    const long long o = offsets[s];
    long long n = offsets[s + 1] - o;
    if (o + n > out_capacity) n = out_capacity > o ? out_capacity - o : 0;
    const int* p = evp + s * cap;
    const int* i = evi + s * cap;
    const real* c = evc + s * cap;
    for (long long e = threadIdx.x; e < n; e += blockDim.x) {
        pos[o + e] = p[e];
        idx[o + e] = i[e];
        coef[o + e] = c[e];
    }
}

// Level hand-off of the hierarchical encoder (hsc/modeling.py:1489, `input = levelCoefficients.todense()`): the
// accumulated code of every signal of the encode in flight as a dense float64 map out[s][T][K] (zeroed by the caller).
// Same arithmetic as the reference's bookkeeping: the events of one (t, k) are summed in float64 in selection order
// (`coefficients[t,k] += c` on a float64 LIL matrix, :992), sums below minCoefficients are dropped (:1171-1177).
// One block per signal; the first event of every distinct (t, k) sums the later ones, so the result does not depend on
// the thread schedule (no atomics).  The event keys are staged through shared memory in tiles.
template <typename real>
__global__ void __launch_bounds__(256) events_to_dense_kernel(const hsc_signal_state* __restrict__ states, const int* __restrict__ evp,
                                                              const int* __restrict__ evi, const real* __restrict__ evc, long long cap,
                                                              int T, int K, double min_coef, double* __restrict__ out) {
    constexpr int TILE = 1024;
    __shared__ long long keys[TILE];
    const long long s = blockIdx.x;
    const long long n = states[s].n_buffered;
    const int* p = evp + s * cap;
    const int* i = evi + s * cap;
    const real* c = evc + s * cap;
    double* o = out + s * (long long)T * K;
    for (long long e0 = 0; e0 < n; e0 += blockDim.x) {
        const long long e = e0 + threadIdx.x;
        const long long key = e < n ? (long long)p[e] * K + i[e] : -1;
        bool first = e < n;
        double sum = e < n ? (double)c[e] : 0.0;
        // pass over ALL events in tiles: an earlier one with the same key -> this thread is not the owner; later ones add up
        for (long long j0 = 0; j0 < n; j0 += TILE) {
            __syncthreads();
            for (long long j = j0 + threadIdx.x; j < min(j0 + TILE, n); j += blockDim.x) keys[j - j0] = (long long)p[j] * K + i[j];
            __syncthreads();
            if (e < n) {
                const long long jn = min((long long)TILE, n - j0);
                for (long long j = 0; j < jn; ++j) {
                    if (keys[j] == key) {
                        const long long jj = j0 + j;
                        if (jj < e) first = false;
                        else if (jj > e) sum += (double)c[jj];          // ascending jj: selection order
                    }
                }
            }
        }
        if (first && sum != 0.0 && !(min_coef >= 0.0 && fabs(sum) < min_coef)) o[key] = sum;
    }
}

// Canonical code of every signal from its flat, selection-ordered events (hsc_b200_canonicalize_codes): one entry per
// distinct (t, k), valued at the float64 sum of its events in selection order - the arithmetic of events_to_dense_kernel -
// with zero sums and sums below min_coef dropped, in ascending (t, k) order within the signal (the list order of the
// decoder).  Each kept entry goes to the first level j with k < bounds[j], else to the last level; order is kept within a
// level.
//
// One block per signal.  The pairs (key = t*K + k, event index) are sorted; they are all distinct, so any sorting network
// orders equal keys by event index, i.e. in selection order.  Then the first thread of each run of equal keys sums the run
// serially (no atomics: two runs give the same bits).  Up to CANON_SMEM_EVENTS events sort in shared memory; a longer
// signal sorts in the global scratch at its own event range.  The kernel runs twice: the counting pass (SCATTER = false)
// writes the entries per (level, signal) to counts[level][s]; after level_offsets_kernel the scatter pass writes every
// entry to its place.  A long signal's scratch keeps the order of the counting pass, so the scatter pass does not sort
// again.
constexpr int CANON_THREADS = 512;
constexpr int CANON_SMEM_EVENTS = 4096;
constexpr int CANON_MAX_LEVELS = 16;

struct LevelBounds {
    long long b[CANON_MAX_LEVELS - 1];
    int n;                                   // number of bounds: n + 1 levels
};

// Ascending sort of the n pairs (key[i], ev[i]) in place, by (key, ev).  Every comparator of this form of the bitonic
// network puts the smaller pair at the lower index, so the network runs on the next power of two with virtual +inf pairs
// past n: a comparator that reaches past n never swaps and is skipped.
template <typename EvIndex>
__device__ void sort_pairs(long long* key, EvIndex* ev, long long n) {
    long long P = 1;
    while (P < n) P <<= 1;
    for (long long k = 2; k <= P; k <<= 1) {
        for (long long j = k >> 1; j > 0; j >>= 1) {
            for (long long p = threadIdx.x; p < (P >> 1); p += blockDim.x) {
                const long long i = ((p & ~(j - 1)) << 1) | (p & (j - 1));       // lower index of pair p
                const long long l = j == (k >> 1) ? (i ^ (k - 1)) : (i + j);     // the first step of a merge mirrors
                if (l >= n) continue;
                const long long ki = key[i], kl = key[l];
                const EvIndex ei = ev[i], el = ev[l];
                if (ki > kl || (ki == kl && ei > el)) {
                    key[i] = kl; key[l] = ki;
                    ev[i] = el; ev[l] = ei;
                }
            }
            __syncthreads();
        }
    }
}

// Exclusive block-wide scan of v (blockDim.x == CANON_THREADS); *total = the block's sum.  Ends with a barrier.
__device__ __forceinline__ int block_exclusive_scan(int v, int* warp_tot, int* total) {
    constexpr int NW = CANON_THREADS / 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = v;
    for (int d = 1; d < 32; d <<= 1) {
        const int o = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += o;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = lane < NW ? warp_tot[lane] : 0;
        for (int d = 1; d < 32; d <<= 1) {
            const int o = __shfl_up_sync(0xffffffffu, w, d);
            if (lane >= d) w += o;
        }
        if (lane < NW) warp_tot[lane] = w;
    }
    __syncthreads();
    const int before = (warp > 0 ? warp_tot[warp - 1] : 0) + incl - v;
    *total = warp_tot[NW - 1];
    __syncthreads();
    return before;
}

template <typename real, bool SCATTER>
__global__ void __launch_bounds__(CANON_THREADS, 1) canonical_codes_kernel(
    const long long* __restrict__ offsets, const int* __restrict__ pos, const int* __restrict__ idx, const real* __restrict__ coef,
    long long capacity, int S, long long K, LevelBounds lb, double min_coef, long long* __restrict__ gkey, int* __restrict__ gev,
    long long* __restrict__ counts, const long long* __restrict__ out_offsets, int* __restrict__ out_pos, int* __restrict__ out_idx,
    double* __restrict__ out_coef) {
    __shared__ long long skey[CANON_SMEM_EVENTS];
    __shared__ unsigned short sev[CANON_SMEM_EVENTS];
    __shared__ int warp_tot[CANON_THREADS / 32];
    __shared__ long long carry[CANON_MAX_LEVELS];
    const int s = blockIdx.x;
    const long long o = offsets[s];
    long long n = offsets[s + 1] - o;
    if (n < 0 || o < 0) n = 0;
    if (o + n > capacity) n = capacity > o ? capacity - o : 0;      // events past the arrays' capacity are not read
    const int* p = pos + o;
    const int* ix = idx + o;
    const real* c = coef + o;
    const bool in_smem = n <= CANON_SMEM_EVENTS;
    const long long* key = in_smem ? skey : gkey + o;
    if (in_smem) {
        for (int e = threadIdx.x; e < n; e += blockDim.x) {
            skey[e] = (long long)p[e] * K + ix[e];
            sev[e] = (unsigned short)e;
        }
        __syncthreads();
        sort_pairs(skey, sev, n);
    } else if (!SCATTER) {
        for (long long e = threadIdx.x; e < n; e += blockDim.x) {
            gkey[o + e] = (long long)p[e] * K + ix[e];
            gev[o + e] = (int)e;
        }
        __syncthreads();
        sort_pairs(gkey + o, gev + o, n);
    }
    if (threadIdx.x < CANON_MAX_LEVELS) carry[threadIdx.x] = 0;
    __syncthreads();
    const int L = lb.n + 1;
    for (long long r0 = 0; r0 < n; r0 += blockDim.x) {
        const long long r = r0 + threadIdx.x;
        int level = -1;                      // -1: not the first event of a kept (t, k)
        double sum = 0.0;
        long long e0 = 0;
        if (r < n && (r == 0 || key[r - 1] != key[r])) {
            const long long kr = key[r];
            e0 = in_smem ? (long long)sev[r] : (long long)gev[o + r];
            sum = (double)c[e0];
            for (long long q = r + 1; q < n && key[q] == kr; ++q) sum += (double)c[in_smem ? (long long)sev[q] : (long long)gev[o + q]];
            if (sum != 0.0 && !(min_coef >= 0.0 && fabs(sum) < min_coef)) {
                const int col = ix[e0];
                level = lb.n;
#pragma unroll
                for (int j = CANON_MAX_LEVELS - 2; j >= 0; --j) {      // constant indices: the bounds stay in the parameter bank
                    if (j < lb.n && col < lb.b[j]) level = j;
                }
            }
        }
        for (int j = 0; j < L; ++j) {
            int total;
            const int rank = block_exclusive_scan(level == j ? 1 : 0, warp_tot, &total);
            const long long base = carry[j];
            if (SCATTER && level == j) {
                const long long d = j * capacity + out_offsets[(long long)j * (S + 1) + s] + base + rank;
                out_pos[d] = p[e0];
                out_idx[d] = ix[e0];
                out_coef[d] = sum;
            }
            __syncthreads();                 // every thread has read carry[j]
            if (threadIdx.x == 0) carry[j] = base + total;
        }
    }
    if (!SCATTER) {
        __syncthreads();
        if (threadIdx.x < L) counts[(long long)threadIdx.x * S + s] = carry[threadIdx.x];
    }
}

}  // namespace events
}  // namespace hsc
