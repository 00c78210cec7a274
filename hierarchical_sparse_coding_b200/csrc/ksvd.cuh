// Dictionary-update stage of the convolutional K-SVD that consumes the MP codes
// (ConvolutionalDictionaryLearner._train_ksvd, hsc/modeling.py:593-636), Gauss-Seidel over the filters:
//   zero the column of filter k, decode WITHOUT it (:602-607), gather the length-L windows centred at its
//   atoms (:610-613), rank-1 SVD -> new filter = first left singular vector, new coefficients = s0 * v0 (:627-633).
//
// The reference decodes the whole code again for every filter (O(K * nnz * L) per sweep, a Python loop).  Here one
// running reconstruction R (float64, [S][T][F]) is kept on the device: removing filter k's atoms from R gives
// exactly the "decode without k" signal on the windows that are gathered, and the updated atoms are added
// back afterwards - O(nnz * L * F) per sweep.  The rank-1 factor is the dominant eigenvector of W^T W
// (power iteration in float64; the sign of the pair is arbitrary, as LAPACK's is in the reference).
#pragma once
#include "common.cuh"

namespace hsc {
namespace ksvd {

// Largest window q = L*F the update accepts: power_kernel keeps two q-vectors in dynamic shared memory (16 * q bytes, 48 KB
// at the limit; the launcher opts in beyond the 48 KB default), and the three q x q float64 matrices take 226 MB of scratch.
constexpr int kMaxQ = 3072;
// Eigen-solver budget.  Squaring stops, after the minimum count (HSC_KSVD_SQUARINGS, 6), once the trace-normalised power
// M = C^(2^s) / tr is numerically rank one: tr((M/tr M)^2) = ||M||_F^2 / tr(M)^2 >= 3/4 bounds the ratio of its two
// largest eigenvalues by 0.17, so that the 100 power steps converge to rounding.  This is the trace the next squaring
// computes anyway, the same in every CTA, so the test costs nothing.  kMaxSquarings = 30 (C^(2^30)) separates relative
// eigenvalue gaps down to ~2e-9; an exactly multiple top eigenvalue runs all of them and yields a vector of its eigenspace.
constexpr int kMaxSquarings = 30;
constexpr double kRankOneTrace = 0.75;

// R[s][p-off+j][f] += sign * c_i * d[j][f] for the n atoms of one filter (clipped at the signal ends).
// The per-filter kernels read the filter's slice [col_ptr[k], col_ptr[k+1]) of the code from DEVICE memory and run on fixed
// grids, so that the launch sequence of a whole sweep does not depend on the code: it is captured once in a CUDA graph.
__global__ void __launch_bounds__(256) scatter_kernel(double* __restrict__ R, const int* __restrict__ sig, const int* __restrict__ pos,
                                                      const double* __restrict__ coef, const long long* __restrict__ col_ptr, int k,
                                                      const double* __restrict__ D, int T, int L, int F, int off, double sign) {
    const int LF = L * F;
    const long long lo = col_ptr[k];
    const int n = (int)(col_ptr[k + 1] - lo);
    sig += lo; pos += lo; coef += lo;
    const double* d = D + (long long)k * LF;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < (long long)n * LF; e += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(e / LF), q = (int)(e - (long long)i * LF);
        const int j = q / F;
        const int t = pos[i] - off + j;
        if (t < 0 || t >= T) continue;
        atomicAdd(R + ((long long)sig[i] * T + t) * F + (q - j * F), sign * coef[i] * d[q]);
    }
}

// R += decode of the whole code (every filter): entry i uses filter idx[i].
__global__ void __launch_bounds__(256) scatter_all_kernel(double* __restrict__ R, const int* __restrict__ sig, const int* __restrict__ pos,
                                                          const int* __restrict__ idx, const double* __restrict__ coef,
                                                          const long long* __restrict__ col_ptr, int K,
                                                          const double* __restrict__ D, int T, int L, int F, int off) {
    const int LF = L * F;
    const long long n = col_ptr[K];
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n * LF; e += (long long)gridDim.x * blockDim.x) {
        const long long i = e / LF;
        const int q = (int)(e - i * LF);
        const int j = q / F;
        const int t = pos[i] - off + j;
        if (t < 0 || t >= T) continue;
        atomicAdd(R + ((long long)sig[i] * T + t) * F + (q - j * F), coef[i] * D[(long long)idx[i] * LF + q]);
    }
}

// W[i][q] = R[s_i][p_i-off+j][f], zero outside the signal (:610-613).
__global__ void __launch_bounds__(256) gather_kernel(const double* __restrict__ R, const int* __restrict__ sig, const int* __restrict__ pos,
                                                     const long long* __restrict__ col_ptr, int k, int T, int L, int F, int off,
                                                     double* __restrict__ W) {
    const int LF = L * F;
    const long long lo = col_ptr[k];
    const int n = (int)(col_ptr[k + 1] - lo);
    sig += lo; pos += lo;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < (long long)n * LF; e += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(e / LF), q = (int)(e - (long long)i * LF);
        const int j = q / F;
        const int t = pos[i] - off + j;
        W[e] = (t < 0 || t >= T) ? 0.0 : R[((long long)sig[i] * T + t) * F + (q - j * F)];
    }
}

// usePCA (hsc/modeling.py:52-54, :618-625): the n >= 2 window rows of filter k are mean-centred in place (the new
// coefficients are projections of the CENTRED windows); a single window is left as it is (:76-78).  32 columns per CTA,
// 8 row lanes, fixed summation order (deterministic).
__global__ void __launch_bounds__(256) center_kernel(double* __restrict__ W, const long long* __restrict__ col_ptr, int k, int q) {
    __shared__ double s_sum[8][33];
    const int n = (int)(col_ptr[k + 1] - col_ptr[k]);
    if (n < 2) return;
    const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
    const int c = blockIdx.x * 32 + cx;
    double acc = 0.0;
    if (c < q)
        for (int i = ry; i < n; i += 8) acc += W[(long long)i * q + c];
    s_sum[ry][cx] = acc;
    __syncthreads();
    double tot = 0.0;
#pragma unroll
    for (int r = 0; r < 8; ++r) tot += s_sum[r][cx];
    const double mean = tot / (double)n;
    if (c < q)
        for (int i = ry; i < n; i += 8) W[(long long)i * q + c] -= mean;
}

// C = W^T W  (q x q, q = L*F), 16x16 output tile per CTA, the n window rows streamed through shared memory.
__global__ void __launch_bounds__(256) gram_tile_kernel(const double* __restrict__ W, const long long* __restrict__ col_ptr, int k, int q,
                                                        double* __restrict__ C) {
    __shared__ double sa[16][17], sb[16][17];
    const int n = (int)(col_ptr[k + 1] - col_ptr[k]);          // 0: the zero matrix
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int a0 = blockIdx.y * 16, b0 = blockIdx.x * 16;
    double acc = 0.0;
    for (int i0 = 0; i0 < n; i0 += 16) {
        const int i = i0 + ty;
        sa[ty][tx] = (i < n && a0 + tx < q) ? W[(long long)i * q + a0 + tx] : 0.0;
        sb[ty][tx] = (i < n && b0 + tx < q) ? W[(long long)i * q + b0 + tx] : 0.0;
        __syncthreads();
#pragma unroll
        for (int r = 0; r < 16; ++r) acc = fma(sa[r][ty], sb[r][tx], acc);
        __syncthreads();
    }
    if (a0 + ty < q && b0 + tx < q) C[(long long)(a0 + ty) * q + b0 + tx] = acc;
}

// out = (in / trace(in))^2: one squaring step of the power method on a PSD matrix (eigenvalue ratios are squared,
// the trace normalisation keeps the spectrum in [0,1]).  16x16 tile per CTA.  Squaring number sq of a filter: the first
// one clears *m_final; from sq = n_min on, a squaring whose input is already numerically rank one (kRankOneTrace) or zero
// stores that input in *m_final and computes nothing, and so do the later ones (a fixed launch sequence, graph-capturable).
__global__ void __launch_bounds__(256) square_kernel(const double* __restrict__ in, int q, double* __restrict__ out, int sq, int n_min,
                                                     const double** m_final) {
    __shared__ double sa[16][17], sb[16][17];
    __shared__ double s_red[8];
    __shared__ double s_scale;
    __shared__ int s_done;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    if (tid == 0) {
        if (sq == 0 && blockIdx.x == 0 && blockIdx.y == 0) *m_final = nullptr;
        // (a CTA of this launch may store it meanwhile: that is the decision this CTA takes below as well)
        s_done = sq > 0 && sq >= n_min && *(const double* volatile*)m_final != nullptr;
    }
    __syncthreads();
    if (s_done) return;
    double tr = 0.0;
    for (int i = tid; i < q; i += 256) tr += in[(long long)i * q + i];
    tr = warp_sum(tr);
    if ((tid & 31) == 0) s_red[tid >> 5] = tr;
    __syncthreads();
    if (tid == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += s_red[w];
        s_scale = t;
    }
    __syncthreads();
    const double t = s_scale;
    if (sq >= n_min && sq > 0 && (t == 0.0 || t >= kRankOneTrace)) {
        if (tid == 0 && blockIdx.x == 0 && blockIdx.y == 0) *m_final = in;
        return;
    }
    const double sc = t > 0.0 ? 1.0 / t : 0.0;
    const int a0 = blockIdx.y * 16, b0 = blockIdx.x * 16;
    double acc = 0.0;
    for (int k0 = 0; k0 < q; k0 += 16) {
        sa[ty][tx] = (a0 + ty < q && k0 + tx < q) ? in[(long long)(a0 + ty) * q + k0 + tx] * sc : 0.0;
        sb[ty][tx] = (k0 + ty < q && b0 + tx < q) ? in[(long long)(k0 + ty) * q + b0 + tx] * sc : 0.0;
        __syncthreads();
#pragma unroll
        for (int r = 0; r < 16; ++r) acc = fma(sa[ty][r], sb[r][tx], acc);
        __syncthreads();
    }
    if (a0 + ty < q && b0 + tx < q) out[(long long)(a0 + ty) * q + b0 + tx] = acc;
}

// Dominant eigenvector of the PSD matrix C (= first left singular vector of W^T, :627-630) by power iteration with
// M = a trace-normalised power C^(2^s) of it (square_kernel), then `polish` iterations with C itself.  Single CTA.
// Start vector: the row of M with the largest diagonal entry, never orthogonal to the dominant subspace of a PSD
// matrix unless M == 0; then u = e_0 like LAPACK's SVD of a zero matrix.  The sign of a singular pair is arbitrary
// (LAPACK's choice in the reference): here <u, d_old> >= 0, the choice that keeps ||D_new - D_old|| (:636) smallest.
// block-wide sum (256 threads), result broadcast to every thread
__device__ __forceinline__ double cta_sum(double v, double* s_red) {
    v = warp_sum(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += s_red[w];
    return t;
}

// u <- u / ||u||; returns ||u_normalised - z|| (z = previous iterate) or -1 if u == 0.
__device__ __forceinline__ double normalise_step(double* u, const double* z, int q, double* s_red) {
    double acc = 0.0;
    for (int i = threadIdx.x; i < q; i += blockDim.x) acc = fma(u[i], u[i], acc);
    const double nrm = sqrt(cta_sum(acc, s_red));
    if (nrm == 0.0) return -1.0;
    const double inv = 1.0 / nrm;
    double diff = 0.0;
    for (int i = threadIdx.x; i < q; i += blockDim.x) {
        const double v = u[i] * inv;
        const double dlt = v - z[i];
        diff = fma(dlt, dlt, diff);
        u[i] = v;
    }
    return sqrt(cta_sum(diff, s_red));
}

// z <- u; u <- A z
__device__ __forceinline__ void matvec_step(const double* __restrict__ A, double* u, double* z, int q) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();
    for (int i = threadIdx.x; i < q; i += blockDim.x) z[i] = u[i];
    __syncthreads();
    for (int a = warp; a < q; a += (int)(blockDim.x >> 5)) {
        double acc = 0.0;
        for (int b = lane; b < q; b += 32) acc = fma(A[(long long)a * q + b], z[b], acc);
        acc = warp_sum(acc);
        if (lane == 0) u[a] = acc;
    }
    __syncthreads();
}

// The same iteration for small windows (q = L*F <= 64: configs 2 and 5) by ONE warp with the matrix in shared memory: lane l
// owns rows l and l + 32, the iterate lives in registers and travels through shared memory once per step, norms and
// differences are warp shuffles - no CTA barrier inside the iteration.  The CTA-wide version below spends ~2 us per
// step in its seven barriers (512-filter sweep at config 5: 36 -> 30 ms).  (Folding the six squarings into the same launch as
// well - one CTA, 4 x 4 register tiles - was built and measured: 41 ms, a single SM squares a 64 x 64 float64 matrix slower
// than the launch gaps it saves; not kept.)
constexpr int kPowerSmallQ = 64;
__device__ __forceinline__ double warp_sum_all(double v) {
    for (int m = 16; m > 0; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
    return v;
}
// one step u <- A u / ||A u|| for the warp; returns ||u_new - u_old|| or -1 when A u == 0.  As: [q][q+1] in shared memory.
__device__ __forceinline__ double power_small_step(const double* As, double* zs, int q, double& u0, double& u1) {
    const int lane = threadIdx.x & 31;
    const int r0 = lane, r1 = lane + 32;
    if (r0 < q) zs[r0] = u0;
    if (r1 < q) zs[r1] = u1;
    __syncwarp();
    double a0 = 0.0, a1 = 0.0;
    const double* row0 = As + (size_t)(r0 < q ? r0 : 0) * (q + 1);
    const double* row1 = As + (size_t)(r1 < q ? r1 : 0) * (q + 1);
    for (int c = 0; c < q; ++c) {
        const double zc = zs[c];
        a0 = fma(row0[c], zc, a0);
        a1 = fma(row1[c], zc, a1);
    }
    if (r0 >= q) a0 = 0.0;
    if (r1 >= q) a1 = 0.0;
    const double nrm = sqrt(warp_sum_all(fma(a0, a0, a1 * a1)));
    __syncwarp();                                  // every lane has read zs
    if (nrm == 0.0) return -1.0;
    const double inv = 1.0 / nrm;
    a0 *= inv; a1 *= inv;
    const double d0 = a0 - u0, d1 = a1 - u1;
    const double diff = sqrt(warp_sum_all(fma(d0, d0, d1 * d1)));
    u0 = a0; u1 = a1;
    return diff;
}

// (small windows: body shared by power_kernel and square_chain_kernel; the matrices are read through L2 - the chain kernel's
//  were written by the other CTAs of its cluster)
__device__ __forceinline__ void power_small(const double* M, const double* C, int q, int max_iter, double tol, int polish,
                                            double* d_io, double* u_out) {
    __shared__ double As[kPowerSmallQ * (kPowerSmallQ + 1)];
    __shared__ double zs[kPowerSmallQ];
    const int tid = threadIdx.x, lane = tid & 31;
    for (int e = tid; e < q * q; e += blockDim.x) As[(e / q) * (q + 1) + (e % q)] = __ldcg(M + e);
    __syncthreads();
    double u0 = 0.0, u1 = 0.0;
    bool zero = false;
    if (tid < 32) {
        // start vector: the row of M with the largest diagonal entry (lowest index among equals)
        double best = -1.0;
        int arg = 0;
        for (int i = lane; i < q; i += 32) { const double v = As[i * (q + 1) + i]; if (v > best) { best = v; arg = i; } }
        for (int m = 16; m > 0; m >>= 1) {
            const double ob = __shfl_xor_sync(0xffffffffu, best, m);
            const int oa = __shfl_xor_sync(0xffffffffu, arg, m);
            if (ob > best || (ob == best && oa < arg)) { best = ob; arg = oa; }
        }
        u0 = lane < q ? As[arg * (q + 1) + lane] : 0.0;
        u1 = lane + 32 < q ? As[arg * (q + 1) + lane + 32] : 0.0;
        const double nrm = sqrt(warp_sum_all(fma(u0, u0, u1 * u1)));
        zero = nrm == 0.0;
        if (!zero) { u0 /= nrm; u1 /= nrm; }
        for (int it = 0; it < max_iter && !zero; ++it) {
            const double d = power_small_step(As, zs, q, u0, u1);
            if (d < 0.0) zero = true;
            else if (d < tol) break;
        }
    }
    if (polish > 0) {                              // (warp-uniform condition; all threads reload the matrix: C itself now)
        __syncthreads();
        for (int e = tid; e < q * q; e += blockDim.x) As[(e / q) * (q + 1) + (e % q)] = __ldcg(C + e);
        __syncthreads();
    }
    if (tid < 32) {
        for (int it = 0; it < polish && !zero; ++it)
            if (power_small_step(As, zs, q, u0, u1) < 0.0) zero = true;
        if (zero) {
            if (lane < q) { const double v = lane == 0 ? 1.0 : 0.0; u_out[lane] = v; d_io[lane] = v; }
            if (lane + 32 < q) { u_out[lane + 32] = 0.0; d_io[lane + 32] = 0.0; }
            return;
        }
        const double o0 = lane < q ? d_io[lane] : 0.0, o1 = lane + 32 < q ? d_io[lane + 32] : 0.0;
        const double sgn = warp_sum_all(fma(u0, o0, u1 * o1)) < 0.0 ? -1.0 : 1.0;      // <u, d_old> >= 0
        if (lane < q) { u_out[lane] = sgn * u0; d_io[lane] = sgn * u0; }
        if (lane + 32 < q) { u_out[lane + 32] = sgn * u1; d_io[lane + 32] = sgn * u1; }
    }
}

// The eigen-solver after square_kernel: M = *m_final when a squaring stored the power it stopped at (m_final may be null:
// no squarings).  A filter without any atom keeps its row (hsc/modeling.py:598-599); skip_col_ptr == nullptr: the caller
// decided.  q <= kPowerSmallQ: power_small_kernel, a kernel of its own so that power_kernel does not carry power_small's
// 34 KB of static shared memory next to its 16 * q bytes of dynamic shared memory.
__global__ void __launch_bounds__(256) power_small_kernel(const double* M, const double* const* m_final, const double* C, int q,
                                                          int max_iter, double tol, int polish, double* d_io, double* u_out,
                                                          const long long* __restrict__ skip_col_ptr, int k) {
    if (skip_col_ptr && skip_col_ptr[k + 1] == skip_col_ptr[k]) return;
    if (m_final && *m_final) M = *m_final;
    power_small(M, C, q, max_iter, tol, polish, d_io, u_out);
}

__global__ void __launch_bounds__(256) power_kernel(const double* M, const double* const* m_final, const double* __restrict__ C, int q,
                                                    int max_iter, double tol, int polish, double* __restrict__ d_io,
                                                    double* __restrict__ u_out, const long long* __restrict__ skip_col_ptr, int k) {
    if (skip_col_ptr && skip_col_ptr[k + 1] == skip_col_ptr[k]) return;
    if (m_final && *m_final) M = *m_final;
    extern __shared__ double sm[];
    double* u = sm;            // [q]
    double* z = sm + q;        // [q]
    __shared__ double s_red[8];
    __shared__ int s_arg;
    const int tid = threadIdx.x;
    if (tid == 0) {
        int arg = 0;
        double best = -1.0;
        for (int i = 0; i < q; ++i) if (M[(long long)i * q + i] > best) { best = M[(long long)i * q + i]; arg = i; }
        s_arg = arg;
    }
    __syncthreads();
    for (int i = tid; i < q; i += blockDim.x) { u[i] = M[(long long)s_arg * q + i]; z[i] = 0.0; }
    __syncthreads();
    bool zero = normalise_step(u, z, q, s_red) < 0.0;
    for (int it = 0; it < max_iter && !zero; ++it) {
        matvec_step(M, u, z, q);
        const double d = normalise_step(u, z, q, s_red);
        if (d < 0.0) zero = true;
        else if (d < tol) break;
    }
    for (int it = 0; it < polish && !zero; ++it) {
        matvec_step(C, u, z, q);
        if (normalise_step(u, z, q, s_red) < 0.0) zero = true;
    }
    if (zero) {
        for (int i = tid; i < q; i += blockDim.x) { const double v = i == 0 ? 1.0 : 0.0; u_out[i] = v; d_io[i] = v; }
        return;
    }
    double dot = 0.0;
    for (int i = tid; i < q; i += blockDim.x) dot = fma(u[i], d_io[i], dot);
    const double sgn = cta_sum(dot, s_red) < 0.0 ? -1.0 : 1.0;
    __syncthreads();                                               // every thread has read the old filter
    for (int i = tid; i < q; i += blockDim.x) { const double v = sgn * u[i]; u_out[i] = v; d_io[i] = v; }     // new filter (:630)
}

// Small windows (q <= 64, i.e. at most 4 x 4 tiles): ALL squarings and the power iteration in one launch of a thread-block
// cluster that spans the grid - one 16 x 16 tile per CTA as in square_kernel, a cluster barrier (release / acquire) between
// squarings, the matrix powers through global memory read with L2-coherent loads, the power iteration on CTA 0.  The sweep is a
// chain of small dependent launches (~5 us each whatever they compute): 11 per filter with the separate kernels, 5 with this.
// Same arithmetic as square_kernel + power_kernel, element for element.  (A variant that keeps the whole matrix in every CTA's
// shared memory and broadcasts each tile with st.shared::cluster was built and measured: 26.6 ms per sweep against 24.6 ms
// - sixteen remote stores per thread and squaring cost more than the L2 round trip they replace.)
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// Squarings n_min .. n_max - 1 stop as in square_kernel: every CTA computes the same trace, so the exit is uniform.
__global__ void __launch_bounds__(256) square_chain_kernel(double* C, int q, int n_min, int n_max, double* buf0, double* buf1, int max_iter,
                                                           double tol, int polish, double* d_io, double* u_out,
                                                           const long long* __restrict__ skip_col_ptr, int k,
                                                           const double* __restrict__ W, const long long* __restrict__ w_col_ptr) {
    if (skip_col_ptr && skip_col_ptr[k + 1] == skip_col_ptr[k]) return;          // (uniform over the cluster)
    __shared__ double sa[16][17], sb[16][17];
    __shared__ double s_red[8];
    __shared__ double s_scale;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int a0 = blockIdx.y * 16, b0 = blockIdx.x * 16;
    if (W) {                                           // C = W^T W first (gram_tile_kernel's tile, same arithmetic)
        const int n = (int)(w_col_ptr[k + 1] - w_col_ptr[k]);
        double acc = 0.0;
        for (int i0 = 0; i0 < n; i0 += 16) {
            const int i = i0 + ty;
            sa[ty][tx] = (i < n && a0 + tx < q) ? W[(long long)i * q + a0 + tx] : 0.0;
            sb[ty][tx] = (i < n && b0 + tx < q) ? W[(long long)i * q + b0 + tx] : 0.0;
            __syncthreads();
#pragma unroll
            for (int r = 0; r < 16; ++r) acc = fma(sa[r][ty], sb[r][tx], acc);
            __syncthreads();
        }
        if (a0 + ty < q && b0 + tx < q) C[(long long)(a0 + ty) * q + b0 + tx] = acc;
        cluster_sync_all();
    }
    const double* in = C;
    for (int sq = 0; sq < n_max; ++sq) {
        double* out = (sq & 1) ? buf1 : buf0;
        double tr = 0.0;
        for (int i = tid; i < q; i += 256) tr += __ldcg(in + (long long)i * q + i);
        tr = warp_sum(tr);
        if ((tid & 31) == 0) s_red[tid >> 5] = tr;
        __syncthreads();
        if (tid == 0) {
            double t = 0.0;
            for (int w = 0; w < 8; ++w) t += s_red[w];
            s_scale = t;
        }
        __syncthreads();
        const double t = s_scale;
        if (sq >= n_min && sq > 0 && (t == 0.0 || t >= kRankOneTrace)) break;
        const double sc = t > 0.0 ? 1.0 / t : 0.0;
        double acc = 0.0;
        for (int k0 = 0; k0 < q; k0 += 16) {
            sa[ty][tx] = (a0 + ty < q && k0 + tx < q) ? __ldcg(in + (long long)(a0 + ty) * q + k0 + tx) * sc : 0.0;
            sb[ty][tx] = (k0 + ty < q && b0 + tx < q) ? __ldcg(in + (long long)(k0 + ty) * q + b0 + tx) * sc : 0.0;
            __syncthreads();
#pragma unroll
            for (int r = 0; r < 16; ++r) acc = fma(sa[ty][r], sb[r][tx], acc);
            __syncthreads();
        }
        if (a0 + ty < q && b0 + tx < q) out[(long long)(a0 + ty) * q + b0 + tx] = acc;
        cluster_sync_all();                            // every tile of `out` is written and visible to the whole cluster
        in = out;
    }
    if (blockIdx.x == 0 && blockIdx.y == 0) power_small(in, C, q, max_iter, tol, polish, d_io, u_out);
}

// proj[i] = <W[i], u>  (new coefficients s0 * v0, :633)
__global__ void __launch_bounds__(256) project_kernel(const double* __restrict__ W, const double* __restrict__ u, int n, int q,
                                                      double* __restrict__ proj) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int i = warp; i < n; i += nwarps) {
        double acc = 0.0;
        for (int b = lane; b < q; b += 32) acc = fma(W[(long long)i * q + b], u[b], acc);
        acc = warp_sum(acc);
        if (lane == 0) proj[i] = acc;
    }
}

// Fused: new coefficient of atom i = <W[i], u> (:633), then the atom goes back into the running reconstruction with the
// new filter u (one warp per atom; atoms of one filter may overlap: atomics).
__global__ void __launch_bounds__(256) project_scatter_kernel(const double* __restrict__ W, const double* __restrict__ u,
                                                              const long long* __restrict__ col_ptr, int k, int q,
                                                              double* __restrict__ coef, double* __restrict__ R, const int* __restrict__ sig,
                                                              const int* __restrict__ pos, int T, int L, int F, int off) {
    const long long lo = col_ptr[k];
    const int n = (int)(col_ptr[k + 1] - lo);
    coef += lo; sig += lo; pos += lo;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int i = warp; i < n; i += nwarps) {
        double acc = 0.0;
        for (int b = lane; b < q; b += 32) acc = fma(W[(long long)i * q + b], u[b], acc);
        acc = warp_sum(acc);
        if (lane == 0) coef[i] = acc;
        const long long base = (long long)sig[i] * T;
        const int p0 = pos[i] - off;
        for (int b = lane; b < q; b += 32) {
            const int j = b / F;
            const int t = p0 + j;
            if (t >= 0 && t < T) atomicAdd(R + (base + t) * F + (b - j * F), acc * u[b]);
        }
    }
}

// out[0] = sum (a - b)^2  (alpha^2 of :636), single CTA.
__global__ void __launch_bounds__(256) sqdist_kernel(const double* __restrict__ a, const double* __restrict__ b, long long n,
                                                     double* __restrict__ out) {
    __shared__ double s_red[8];
    double acc = 0.0;
    for (long long i = threadIdx.x; i < n; i += blockDim.x) { const double d = a[i] - b[i]; acc = fma(d, d, acc); }
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += s_red[w];
        out[0] = t;
    }
}

}  // namespace ksvd
}  // namespace hsc
