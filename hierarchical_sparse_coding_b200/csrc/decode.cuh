// Sparse decoder (reconstructSignal, hsc/modeling.py:226-245): out[s][t][f] += sum_n c_n * D[k_n][t-(p_n-off)][f].
// Gather form: the atoms of signal s are [offsets[s], offsets[s+1]) of the flat lists, sorted by centre position within
// the signal; each output sample binary-searches the contiguous range of its own signal's atoms that can cover it and sums
// them in list order (deterministic, no atomics).  offsets == nullptr: one signal, atoms [0, n).
#pragma once
#include "common.cuh"

namespace hsc {

template <typename real>
__global__ void decode_gather_kernel(const long long* __restrict__ offsets, long long n, const int* __restrict__ pos,
                                     const int* __restrict__ idx, const real* __restrict__ coef, const real* __restrict__ D,
                                     long long S, int T, int K, int L, int F, int off, real* __restrict__ out) {
    const long long per_signal = (long long)T * F;
    const long long total = S * per_signal;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total;
         e += (long long)gridDim.x * blockDim.x) {
        const long long s = e / per_signal;
        const long long r = e - s * per_signal;
        const int t = (int)(r / F);
        const int f = (int)(r - (long long)t * F);
        const long long lo = offsets ? offsets[s] : 0, hi = offsets ? offsets[s + 1] : n;
        // atom at p covers t iff p-off <= t <= p-off+L-1  <=>  t-(L-1)+off <= p <= t+off
        const int plo = t - (L - 1) + off, phi = t + off;
        long long a = lo, b = hi;         // first index of the segment with pos >= plo
        while (a < b) {
            long long m = (a + b) >> 1;
            if (pos[m] < plo) a = m + 1; else b = m;
        }
        double acc = 0.0;
        for (long long i = a; i < hi && pos[i] <= phi; ++i) {
            const int j = t - (pos[i] - off);
            acc = fma((double)coef[i], (double)D[((long long)idx[i] * L + j) * F + f], acc);
        }
        out[e] = (real)((double)out[e] + acc);
    }
}

}  // namespace hsc
