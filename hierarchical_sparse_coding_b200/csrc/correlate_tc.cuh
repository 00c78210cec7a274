// K1 on the 5th-generation tensor cores: the initial residual-by-dictionary cross-correlation
// (convolve1d 'same', hsc/modeling.py:149-188, called at :1077) as an IMPLICIT GEMM,
//
//     c[t][k] = sum_q A[t][q] * B[k][q],   A[t][q] = xz[(t-off)*F + q],  q = j*F + f  (Toeplitz view)
//
// with fp32 accumulators in TMEM and a three-product operand split
//     x = x_hi + x_lo  =>  c ~= A_lo*B_hi + A_hi*B_lo + A_hi*B_hi          (fp32-grade accuracy),
// so that atom selection and coefficients keep the reference's float32 precision.  Two operand formats:
//   * 3xFP16 (default, tcgen05.mma kind::f16, twice the tensor rate of tf32): hi = fp16(x*2^e), lo = fp16((x*2^e - hi)*2^11),
//     an 11 + 11 bit significand like 3xTF32.  2^e is a per-signal power of two that puts max|x| in [2^9, 2^10) (the
//     dictionary gets one global power of two), the two lo products accumulate in their own TMEM columns and the
//     epilogue forms (acc_hh + 2^-11 * acc_lo) * 2^-e: all scalings are exact.
//   * 3xTF32 (kind::tf32): hi = tf32(x*2^e), lo = tf32(x*2^e - hi) with the same powers of two (the tensor core flushes
//     subnormal tf32 operands and products, so unscaled inputs below ~2^-115 lost their map), the epilogue forms
//     (acc_hh + acc_lo) * 2^-e.  HSC_K1=tf32 selects it.
// Below, "element" is an fp16 or fp32 operand element and R = 16 / sizeof(element) is the number of elements in a
// 16-byte core-matrix row (8 or 4).
//
// No im2col, not even in shared memory.  With R elements per (super-)row the Toeplitz operand IS a
// canonical K-major / no-swizzle UMMA layout of the raw signal slab: core matrix = 8 rows x 16 B with
// a 16-byte row pitch, K-chunk stride LBO = 16 B, 8-row-group stride SBO = 128 B -- overlapping core
// matrices, which the tensor core reads like any other (probed on B200: tools/tc_probe.cu).  One
// 128-row A tile is therefore a (127*4 + Kd)-float slab (3 KB for L*F = 256) instead of 128 KB, and
// shared memory holds the whole dictionary slice B (hi and lo parts) for the life of the CTA.
//
//   F = R: rows are time steps.          F < R: s = R/F time steps are grouped in one
//   super-row m (t = s*m + i); column (i,k) of the product uses the dictionary shifted by i*F
//   elements, B'[(i,k)][q] = D[k][q - i*F]; the output [T/s][s*K] row-major is the same memory as
//   [T][K].  Kd = roundup((L+s-1)*F, elements per MMA K-step), Ntot = s*K.  (fp16, F = 4: s = 2, one MMA row
//   covers two time steps, N doubles, M halves: the same number of MACs.)
//
// CTA roles (320 threads): warp 0 fetches the pre-split signal slabs with bulk copies (6-stage ring), warp 1
// allocates TMEM and issues the MMAs (one elected lane), warps 2-9 drain the accumulators (tcgen05.ld 32x32b) to HBM
// (2-deep TMEM ring, so the epilogue of tile i overlaps the MMAs of tile i+1).  Persistent grid:
// each CTA owns one N-slice of NS columns (its B slice never leaves shared memory) and strides over
// the (signal, M-tile) list.
#pragma once
#include <cuda_fp16.h>
#include <string.h>
#include <vector>
#include "common.cuh"

namespace hsc {
namespace tc {

constexpr int kThreads = 320;   // warp 0 producer, warp 1 MMA, warps 2-9 epilogue
constexpr int kTileM = 128;
constexpr int kStages = 6;      // slab ring depth (a slab is ~3 KB per part)

struct Plan {            // host-side geometry of one dictionary
    int half;            // 1: 3xFP16 operands, 0: 3xTF32
    int esz;             // bytes per operand element (2 or 4)
    int R;               // elements per 16-byte core-matrix row (8 or 4)
    int s;               // time steps per super-row (R / F)
    int Kd;              // padded reduction length, elements
    int Ntot;            // s * K, unpadded
    int NS;              // output columns per slice (multiple of 32, <= 128: the combined [hi|lo] operand has N = 2*NS)
    int nslices;
    int slab_elems;      // R*(kTileM-1) + Kd
    int slab_stride_bytes;
    float d_scale;       // power of two applied to the dictionary before the split (max|D| in [0.5, 1))
    size_t smem_bytes;
    bool ok;
};

// Power-of-two exponent e of the operand split (3xFP16 and 3xTF32) that puts max|v| * 2^e in [2^top, 2^(top+1)): top = 9 for a signal,
// top = -1 for the dictionary.  Clamped to [-126, 127] so that 2^e and 2^-e are finite and non-zero: an input too
// small to reach the target range (max|x| < 2^-118, max|D| < 2^-128) is scaled by 2^127 instead, which still leaves
// its largest element at 2^-22 or more and every float32 subnormal exactly representable in hi + lo.  In-range
// inputs get the unclamped exponent, so their split and their map are unchanged.
__host__ __device__ inline int split_exponent(float mx, int top) {
    if (!(mx > 0.f) || !isfinite(mx)) return 0;
    const int e = top - ilogbf(mx);
    return e < -126 ? -126 : (e > 127 ? 127 : e);
}

inline Plan make_plan(int K, int L, int F, bool half, int ns_max = 128) {
    Plan p{};
    p.ok = false;
    p.half = half ? 1 : 0;
    p.esz = half ? 2 : 4;
    p.R = 16 / p.esz;
    p.d_scale = 1.f;
    if (F < 1 || F > p.R || (p.R % F) != 0) return p;
    const int kstep = half ? 16 : 8;                      // elements per MMA K-step (32 bytes)
    p.s = p.R / F;
    p.Kd = (((L + p.s - 1) * F) + kstep - 1) / kstep * kstep;
    p.Ntot = p.s * K;
    const int npad = (p.Ntot + 31) / 32 * 32;
    int best = 0;
    for (int ns = ns_max < 32 ? 32 : (ns_max > 128 ? 128 : ns_max / 32 * 32); ns >= 32; ns -= 32) {
        if (npad % ns) continue;
        size_t b = (size_t)2 * ns * p.Kd * p.esz;
        if (b <= 160 * 1024) { best = ns; break; }
    }
    if (!best) return p;
    p.NS = best;
    p.nslices = npad / best;
    if (p.nslices > 148) return p;
    p.slab_elems = p.R * (kTileM - 1) + p.Kd;
    p.slab_stride_bytes = (p.slab_elems * p.esz + 15) / 16 * 16;
    p.smem_bytes = (size_t)2 * p.NS * p.Kd * p.esz + (size_t)2 * kStages * p.slab_stride_bytes + 1024 + 256;
    if (p.smem_bytes > 227 * 1024) return p;
    p.ok = true;
    return p;
}

// fp32 -> tf32, round to nearest, ties away from zero (what cvt.rna.tf32.f32 does), host side.
inline float tf32_rna_host(float x) {
    uint32_t u;
    memcpy(&u, &x, 4);
    if ((u & 0x7f800000u) == 0x7f800000u) return x;
    u = (u + 0x1000u) & 0xffffe000u;
    float r;
    memcpy(&r, &u, 4);
    return r;
}

constexpr float kLoScale = 2048.f;      // fp16 split: the lo part is stored times 2^11

// Expanded, shifted, split dictionary in the per-slice canonical layout the CTA copies verbatim.  The hi and
// lo parts of a slice are stacked along N, [B_hi ; B_lo], so that ONE MMA of N = 2*NS computes A_hi*B_hi
// and A_hi*B_lo while reading A_hi from shared memory once:
//   out[((slice*(Kd/R) + kc)*2*NS + part*NS + n)*R + j] = part(B'[slice*NS + n][kc*R + j])
// Returns raw bytes (fp32 or fp16 elements).  p.d_scale is set to the power of two used.
inline void build_b_operand(const float* D, int K, int L, int F, Plan& p, std::vector<unsigned char>& out) {
    const size_t n = (size_t)p.nslices * 2 * p.NS * p.Kd;
    out.assign(n * p.esz, 0);
    const int LF = L * F;
    {
        float mx = 0.f;
        for (size_t i = 0; i < (size_t)K * LF; ++i) mx = fmaxf(mx, fabsf(D[i]));
        p.d_scale = ldexpf(1.f, split_exponent(mx, -1));      // max|D|*scale in [0.5, 1)
    }
    float* of = reinterpret_cast<float*>(out.data());
    __half* oh = reinterpret_cast<__half*>(out.data());
    for (int row = 0; row < p.Ntot; ++row) {
        const int i = row / K, k = row % K;
        const int sl = row / p.NS, nn = row % p.NS;
        for (int q = 0; q < p.Kd; ++q) {
            const int src = q - i * F;
            if (src < 0 || src >= LF) continue;
            const float v = D[(size_t)k * LF + src] * p.d_scale;
            const size_t o = (((size_t)sl * (p.Kd / p.R) + q / p.R) * 2 * p.NS + nn) * p.R + (q % p.R);
            if (p.half) {
                const __half h = __float2half_rn(v);
                oh[o] = h;
                oh[o + (size_t)p.NS * p.R] = __float2half_rn((v - __half2float(h)) * kLoScale);
            } else {
                const float h = tf32_rna_host(v);
                of[o] = h;
                of[o + (size_t)p.NS * p.R] = tf32_rna_host(v - h);
            }
        }
    }
}

// Device version of build_b_operand (a learning loop sets a new dictionary every iteration; the host loop costs tens of
// milliseconds at 512 filters): one thread per element of the expanded, shifted dictionary B'[row][q].
__global__ void __launch_bounds__(256) build_b_operand_kernel(const float* __restrict__ D, int K, int L, int F, int half, int R, int s_rows,
                                                              int Kd, int Ntot, int NS, float d_scale, void* __restrict__ out) {
    const long long total = (long long)Ntot * Kd;
    const int LF = L * F;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int row = (int)(e / Kd), q = (int)(e - (long long)row * Kd);
        const int i = row / K, k = row - i * K;
        const int sl = row / NS, nn = row - sl * NS;
        const int src = q - i * F;
        const float v = (src >= 0 && src < LF) ? D[(size_t)k * LF + src] * d_scale : 0.f;
        const size_t o = (((size_t)sl * (Kd / R) + q / R) * 2 * NS + nn) * R + (q % R);
        if (half) {
            __half* oh = reinterpret_cast<__half*>(out);
            const __half h = __float2half_rn(v);
            oh[o] = h;
            oh[o + (size_t)NS * R] = __float2half_rn((v - __half2float(h)) * 2048.f);
        } else {
            float* of = reinterpret_cast<float*>(out);
            uint32_t r;
            asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
            const float h = __uint_as_float(r);
            of[o] = h;
            asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v - h));
            of[o + (size_t)NS * R] = __uint_as_float(r);
        }
    }
    (void)s_rows;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;     // descriptor version 1 (sm_100); no swizzle, base offset 0
    return d;
}

__device__ __forceinline__ uint32_t idesc_tf32(int m, int n) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

__device__ __forceinline__ void mma_tf32(uint32_t tmem_c, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t}\n"
        :: "r"(tmem_c), "l"(da), "l"(db), "r"(idesc), "r"(accumulate), "r"(0), "r"(0), "r"(0), "r"(0));
}

// kind::f16 with fp16 operands (a_format = b_format = 0) and fp32 accumulators (c_format = 1)
__device__ __forceinline__ uint32_t idesc_f16(int m, int n) {
    return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

__device__ __forceinline__ void mma_f16(uint32_t tmem_c, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t}\n"
        :: "r"(tmem_c), "l"(da), "l"(db), "r"(idesc), "r"(accumulate), "r"(0), "r"(0), "r"(0), "r"(0));
}

__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(bar) : "memory");
}

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count));
}

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(bar) : "memory");
}

__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tHSC_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra HSC_DONE_%=;\n\tbra HSC_WAIT_%=;\n\tHSC_DONE_%=:\n\t}\n" :: "r"(bar), "r"(parity) : "memory");
}

__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile(
        "{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\t"
        "elect.sync rx|px, %1;\n\t"
        "@px mov.s32 %0, 1;\n\t}\n" : "+r"(pred) : "r"(0xffffffffu));
    return pred != 0;
}

__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(dst_smem), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

__device__ __forceinline__ float to_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, "
                 "%24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
                   "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
                   "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
                   "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(taddr));
}

// Zero-padded 3xTF32 split of the signals: out[s][pad_front + i] = part(x[s][i] * 2^e); everything else 0.  2^e and
// out_scale[s] as in split_signal_half_kernel below.
// pad_front = off*F makes the slab of tile m0 start at float 4*m0 of the padded signal (16-byte aligned),
// and the tail padding covers the last tile plus the reduction overhang, so every slab is one in-bounds
// contiguous chunk the TMA engine can fetch.
__global__ void __launch_bounds__(256) split_signal_kernel(const float* __restrict__ x, float* __restrict__ hi,
                                                           float* __restrict__ lo, long long n_valid, long long stride,
                                                           int pad_front, const unsigned* __restrict__ absmax,
                                                           float inv_d_scale, float* __restrict__ out_scale) {
    const long long s = blockIdx.y;
    const int e = split_exponent(__uint_as_float(absmax[s]), 9);
    const float sc = ldexpf(1.f, e);
    if (blockIdx.x == 0 && threadIdx.x == 0) out_scale[s] = ldexpf(inv_d_scale, -e);
    const float* xs = x + s * n_valid;
    float* hs = hi + s * stride;
    float* ls = lo + s * stride;
    for (long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x; j < stride; j += (long long)gridDim.x * blockDim.x) {
        const long long i = j - pad_front;
        const float v = (i >= 0 && i < n_valid) ? __ldg(xs + i) * sc : 0.f;
        const float h = to_tf32(v);
        hs[j] = h;
        ls[j] = to_tf32(v - h);
    }
}

// max|x| of every signal, as float bits (non-negative floats order like unsigned integers); absmax zero-initialised.
__global__ void __launch_bounds__(256) signal_absmax_kernel(const float* __restrict__ x, long long n_valid, unsigned* __restrict__ absmax) {
    const long long s = blockIdx.y;
    const float* xs = x + s * n_valid;
    float m = 0.f;
    for (long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x; j < n_valid; j += (long long)gridDim.x * blockDim.x)
        m = fmaxf(m, fabsf(__ldg(xs + j)));
    m = warp_max<float>(m);
    if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(absmax + s, __float_as_uint(m));
}

// Zero-padded 3xFP16 split: hi = fp16(x*2^e), lo = fp16((x*2^e - hi)*2^11) with 2^e the per-signal power of two that
// puts max|x| in [2^9, 2^10); out_scale[s] = 2^-e / d_scale is what the epilogue multiplies the accumulators by.
__global__ void __launch_bounds__(256) split_signal_half_kernel(const float* __restrict__ x, __half* __restrict__ hi,
                                                                __half* __restrict__ lo, long long n_valid, long long stride,
                                                                int pad_front, const unsigned* __restrict__ absmax,
                                                                float inv_d_scale, float* __restrict__ out_scale) {
    const long long s = blockIdx.y;
    const int e = split_exponent(__uint_as_float(absmax[s]), 9);
    const float sc = ldexpf(1.f, e);
    if (blockIdx.x == 0 && threadIdx.x == 0) out_scale[s] = ldexpf(inv_d_scale, -e);
    const float* xs = x + s * n_valid;
    __half* hs = hi + s * stride;
    __half* ls = lo + s * stride;
    for (long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x; j < stride; j += (long long)gridDim.x * blockDim.x) {
        const long long i = j - pad_front;
        const float v = (i >= 0 && i < n_valid) ? __ldg(xs + i) * sc : 0.f;
        const __half h = __float2half_rn(v);
        hs[j] = h;
        ls[j] = __float2half_rn((v - __half2float(h)) * kLoScale);
    }
}

// The same split, eight samples per thread (two 128-bit loads, one 128-bit store per part): requires pad_front and n_valid
// to be multiples of 4, stride a multiple of 8 and 16-byte aligned bases, so that each half of a group of eight is
// entirely signal or entirely padding.
__global__ void __launch_bounds__(256) split_signal_half_vec8_kernel(const float* __restrict__ x, __half* __restrict__ hi,
                                                                     __half* __restrict__ lo, long long n_valid, long long stride,
                                                                     int pad_front, const unsigned* __restrict__ absmax,
                                                                     float inv_d_scale, float* __restrict__ out_scale) {
    const long long s = blockIdx.y;
    const int e = split_exponent(__uint_as_float(absmax[s]), 9);
    const float sc = ldexpf(1.f, e);
    if (blockIdx.x == 0 && threadIdx.x == 0) out_scale[s] = ldexpf(inv_d_scale, -e);
    const float* xs = x + s * n_valid;
    uint4* hs = reinterpret_cast<uint4*>(hi + s * stride);
    uint4* ls = reinterpret_cast<uint4*>(lo + s * stride);
    const long long groups = stride >> 3;
    for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < groups; g += (long long)gridDim.x * blockDim.x) {
        const long long i = (g << 3) - pad_front;
        uint4 oh = make_uint4(0u, 0u, 0u, 0u), ol = oh;
        const bool in_a = i >= 0 && i < n_valid, in_b = i + 4 >= 0 && i + 4 < n_valid;
        if (in_a || in_b) {
            const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
            const float4 a = in_a ? __ldg(reinterpret_cast<const float4*>(xs + i)) : zero4;
            const float4 b = in_b ? __ldg(reinterpret_cast<const float4*>(xs + i + 4)) : zero4;
            const float v[8] = {a.x * sc, a.y * sc, a.z * sc, a.w * sc, b.x * sc, b.y * sc, b.z * sc, b.w * sc};
            unsigned ph[4], pl[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const __half h0 = __float2half_rn(v[2 * q]), h1 = __float2half_rn(v[2 * q + 1]);
                const __half l0 = __float2half_rn((v[2 * q] - __half2float(h0)) * kLoScale);
                const __half l1 = __float2half_rn((v[2 * q + 1] - __half2float(h1)) * kLoScale);
                ph[q] = (unsigned)__half_as_ushort(h0) | ((unsigned)__half_as_ushort(h1) << 16);
                pl[q] = (unsigned)__half_as_ushort(l0) | ((unsigned)__half_as_ushort(l1) << 16);
            }
            oh = make_uint4(ph[0], ph[1], ph[2], ph[3]);
            ol = make_uint4(pl[0], pl[1], pl[2], pl[3]);
        }
        hs[g] = oh;
        ls[g] = ol;
    }
}

// Packed level-1 keys -> the (value, filter) arrays the pursuit kernel keeps.
__global__ void __launch_bounds__(256) unpack_keys_kernel(const unsigned long long* __restrict__ keys, float* __restrict__ val1,
                                                          int* __restrict__ idx1, long long n) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const unsigned long long k = keys[i];
        val1[i] = __uint_as_float((unsigned)(k >> 32));
        idx1[i] = k == 0ull ? 0 : (int)(0xFFFFFFFFu - (unsigned)(k & 0xFFFFFFFFull));
    }
}

struct Args {
    const void* x_hi;     // [S][xpad_stride] zero-padded 'hi' part of the signal (split_signal_*_kernel), fp16 or tf32 elements
    const void* x_lo;     //                   and the 'lo' part
    long long xpad_stride;     // elements
    const void* b_op;     // [nslices][Kd/R][2*NS][R]: stacked hi / lo dictionary slices
    const float* out_scale;    // [S] factor applied to the accumulators (2^-e / d_scale)
    float* map;           // [S][T][K]
    int S, T, F, K, off;
    int s, Kd, Ntot, NS, nslices, slab_elems, slab_stride_bytes;
    int tmem_cols;        // power of two >= 4*NS (two accumulator stages of 2*NS columns)
    unsigned long long* keys;  // [S][T] packed level-1 keys (|c| bits << 32 | ~k), zero-initialised; nullptr = not fused
    long long* prof;      // HSC_PROFILE_PHASES: [grid][16] cycle counters per role, else nullptr
};

template <bool H>     // H: 3xFP16 operands (kind::f16), else 3xTF32 (kind::tf32)
// (launch bounds: 96 registers per thread - no spills - so that one correlation CTA and two pursuit CTAs fit the register
// file of an SM together: the streaming pipeline runs the correlation of batch i+1 under the pursuit of batch i)
__global__ void __launch_bounds__(kThreads, 2) correlate_tc_kernel(Args a) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    constexpr int ESZ = H ? 2 : 4;                                       // bytes per operand element
    constexpr int R = 16 / ESZ;                                          // elements per 16-byte core-matrix row
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int NS = a.NS, Kd = a.Kd;
    const int slab_stride = a.slab_stride_bytes;                         // bytes, multiple of 16
    unsigned char* sB = smem_raw;                                        // [Kd/R][2*NS][R] elements
    unsigned char* sA = sB + (size_t)2 * NS * Kd * ESZ;                  // [stage][part][slab_stride bytes]
    uint64_t* bars = reinterpret_cast<uint64_t*>(sA + (size_t)2 * kStages * slab_stride);  // 2*kStages + 4 mbarriers
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);
    const uint32_t bar_slab_full = smem_u32(bars + 0), bar_slab_empty = smem_u32(bars + kStages);
    const uint32_t bar_acc_full = smem_u32(bars + 2 * kStages), bar_acc_empty = smem_u32(bars + 2 * kStages + 2);

    const int slice = blockIdx.x % a.nslices;
    const int cta_m = blockIdx.x / a.nslices;
    const int ctas_per_slice = gridDim.x / a.nslices;
    const int Ts = (a.T + a.s - 1) / a.s;                                // super-rows per signal
    const int MT = (Ts + kTileM - 1) / kTileM;
    const long long ntiles = (long long)a.S * MT;

    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(tmem_slot)), "r"(a.tmem_cols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    if (tid == 0) {
        for (int i = 0; i < kStages; ++i) {
            mbar_init(bar_slab_full + 8 * i, 1);
            mbar_init(bar_slab_empty + 8 * i, 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(bar_acc_full + 8 * i, 1);
            mbar_init(bar_acc_empty + 8 * i, 8);
        }
        asm volatile("fence.mbarrier_init.release.cluster;");
    }
    // dictionary slice (already split and laid out): straight 16-byte copy
    {
        const float4* gb = reinterpret_cast<const float4*>(reinterpret_cast<const unsigned char*>(a.b_op) + (size_t)slice * 2 * NS * Kd * ESZ);
        float4* sb = reinterpret_cast<float4*>(sB);
        const int n4 = 2 * NS * Kd * ESZ / 16;
        for (int e = tid; e < n4; e += kThreads) sb[e] = __ldg(gb + e);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;");
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ------------------------------------------------------------ slab producer: one lane, two bulk copies
        // (TMA engine, async proxy) per tile straight out of the pre-split, zero-padded signal; completion is
        // counted in bytes on the stage's mbarrier, so no generic-proxy stores and no proxy fence sit between
        // the tensor core and its operands.
        if (lane == 0) {
            int stage = 0, phase = 0;
            const uint32_t slab_bytes = (uint32_t)a.slab_elems * (uint32_t)ESZ;
#ifdef HSC_PROFILE_PHASES
            long long pw_wait = 0, pw_work = 0;
#endif
            for (long long tile = cta_m; tile < ntiles; tile += ctas_per_slice) {
                const int sig = (int)(tile / MT);
                const int m0 = (int)(tile % MT) * kTileM;
                const long long src = ((long long)sig * a.xpad_stride + (long long)R * m0) * ESZ;     // bytes; 16-byte aligned
#ifdef HSC_PROFILE_PHASES
                long long c0_ = clock64();
#endif
                mbar_wait(bar_slab_empty + 8 * stage, phase ^ 1);
#ifdef HSC_PROFILE_PHASES
                long long c1_ = clock64();
                pw_wait += c1_ - c0_;
#endif
                const uint32_t bar = bar_slab_full + 8 * stage;
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(2u * slab_bytes) : "memory");
                bulk_g2s(smem_u32(sA + (size_t)(stage * 2 + 0) * slab_stride), reinterpret_cast<const unsigned char*>(a.x_hi) + src, slab_bytes, bar);
                bulk_g2s(smem_u32(sA + (size_t)(stage * 2 + 1) * slab_stride), reinterpret_cast<const unsigned char*>(a.x_lo) + src, slab_bytes, bar);
#ifdef HSC_PROFILE_PHASES
                pw_work += clock64() - c1_;
#endif
                if (++stage == kStages) { stage = 0; phase ^= 1; }
            }
#ifdef HSC_PROFILE_PHASES
            if (a.prof) { a.prof[blockIdx.x * 16 + 0] = pw_wait; a.prof[blockIdx.x * 16 + 1] = pw_work; }
#endif
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------ MMA issuer: warp-uniform control flow,
        // one elected lane issues (descriptors stay in uniform registers, no per-instruction lane loop)
        {
            const uint32_t idesc_wide = H ? idesc_f16(kTileM, 2 * NS) : idesc_tf32(kTileM, 2 * NS);    // A_hi x [B_hi ; B_lo]
            const uint32_t idesc_half = H ? idesc_f16(kTileM, NS) : idesc_tf32(kTileM, NS);            // A_lo x  B_hi
            const uint32_t b_lbo = (uint32_t)(2 * NS) * 16;
            const uint32_t b0 = smem_u32(sB);
            int stage = 0, phase = 0, acc = 0, acc_phase = 0;
            const int nk = Kd / (2 * R);                               // one MMA consumes 32 bytes of K per row
#ifdef HSC_PROFILE_PHASES
            long long mw_slab = 0, mw_acc = 0, mw_issue = 0;
#endif
            for (long long tile = cta_m; tile < ntiles; tile += ctas_per_slice) {
#ifdef HSC_PROFILE_PHASES
                long long c0_ = clock64();
#endif
                mbar_wait(bar_slab_full + 8 * stage, phase);
#ifdef HSC_PROFILE_PHASES
                long long c1_ = clock64();
#endif
                mbar_wait(bar_acc_empty + 8 * acc, acc_phase ^ 1);
#ifdef HSC_PROFILE_PHASES
                long long c2_ = clock64();
                mw_slab += c1_ - c0_; mw_acc += c2_ - c1_;
#endif
                asm volatile("tcgen05.fence::after_thread_sync;");
                const uint32_t ahi0 = smem_u32(sA + (size_t)(stage * 2 + 0) * slab_stride);
                const uint32_t alo0 = smem_u32(sA + (size_t)(stage * 2 + 1) * slab_stride);
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * 2 * NS);
                // per K-step: columns [0,2NS) += A_hi*[B_hi;B_lo], then columns [0,NS) += A_lo*B_hi.  A_hi is
                // fetched from shared memory once for two of the three 3xTF32 products.
                uint64_t da_hi = smem_desc(ahi0, 16, 128);              // Toeplitz slab: LBO 16 B, SBO 128 B
                uint64_t da_lo = smem_desc(alo0, 16, 128);
                uint64_t db = smem_desc(b0, b_lbo, 128);
                const uint64_t da_step = 32 >> 4, db_step = (2 * b_lbo) >> 4;
                uint32_t accum = 0;
#pragma unroll 4
                for (int kk = 0; kk < nk; ++kk) {
                    if (elect_one()) {
                        if constexpr (H) {
                            // fp16: the lo parts carry a factor 2^11, so both lo products accumulate in columns [NS, 2NS)
                            mma_f16(d_tmem, da_hi, db, idesc_wide, accum);
                            mma_f16(d_tmem + (uint32_t)NS, da_lo, db, idesc_half, 1u);
                        } else {
                            mma_tf32(d_tmem, da_hi, db, idesc_wide, accum);
                            mma_tf32(d_tmem, da_lo, db, idesc_half, 1u);
                        }
                    }
                    accum = 1;
                    da_hi += da_step;
                    da_lo += da_step;
                    db += db_step;
                }
                if (elect_one()) {
                    umma_commit(bar_slab_empty + 8 * stage);
                    umma_commit(bar_acc_full + 8 * acc);
                }
                __syncwarp();
#ifdef HSC_PROFILE_PHASES
                mw_issue += clock64() - c2_;
#endif
                if (++stage == kStages) { stage = 0; phase ^= 1; }
                acc ^= 1;
                if (acc == 0) acc_phase ^= 1;
            }
#ifdef HSC_PROFILE_PHASES
            if (lane == 0 && a.prof) { a.prof[blockIdx.x * 16 + 2] = mw_slab; a.prof[blockIdx.x * 16 + 3] = mw_acc; a.prof[blockIdx.x * 16 + 4] = mw_issue; }
#endif
        }
    } else {
        // ------------------------------------------------------------ epilogue: TMEM -> HBM
        // 8 warps: two per TMEM lane quarter, each draining half of the slice's columns.  A thread owns one
        // output row: it adds the two partial accumulators, streams its 32-column chunks out with 256-bit
        // stores and (fused level-1 key of the argmax hierarchy) folds max_k |c[t][k]| of the chunk into the
        // row's packed key with one 64-bit atomicMax, so the map is never re-read to build the keys.
        const int quarter = warp & 3;                     // TMEM lane quarter this warp may read
        const int half = (warp - 2) >> 2;                 // which half of the slice's columns
        const int chunks = NS / 32;
        const int c_begin = (half == 0 ? 0 : (chunks + 1) / 2) * 32;
        const int c_end = (half == 0 ? (chunks + 1) / 2 : chunks) * 32;
        int acc = 0, acc_phase = 0;
#ifdef HSC_PROFILE_PHASES
        long long ew_wait = 0, ew_work = 0;
#endif
        const long long row_pitch = (long long)a.Ntot;    // floats per super-row of the output
        const long long map_elems = (long long)a.T * a.K;
        const bool wide_ok = (row_pitch % 8) == 0 && (map_elems % 8) == 0;
        for (long long tile = cta_m; tile < ntiles; tile += ctas_per_slice) {
            const int sig = (int)(tile / MT);
            const int m0 = (int)(tile % MT) * kTileM;
            float* ms = a.map + (long long)sig * map_elems;
            const float osc = __ldg(a.out_scale + sig);
            constexpr float lsc = H ? (1.f / kLoScale) : 1.f;
#ifdef HSC_PROFILE_PHASES
            long long c0_ = clock64();
#endif
            mbar_wait(bar_acc_full + 8 * acc, acc_phase);
#ifdef HSC_PROFILE_PHASES
            long long c1_ = clock64();
            ew_wait += c1_ - c0_;
#endif
            asm volatile("tcgen05.fence::after_thread_sync;");
            const int row = m0 + quarter * 32 + lane;
            const uint32_t t0 = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * 2 * NS);
            if (c_begin >= c_end) {                       // NS == 32: the second warp of the pair has no columns
                if (lane == 0) mbar_arrive(bar_acc_empty + 8 * acc);
            }
            for (int c0 = c_begin; c0 < c_end; c0 += 32) {
                uint32_t v[32], w[32];
                tmem_ld32(t0 + c0, v);                    // A_hi*B_hi (tf32: + A_lo*B_hi)
                tmem_ld32(t0 + NS + c0, w);               // A_hi*B_lo (fp16: + A_lo*B_hi, both times 2^11)
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (c0 + 32 >= c_end) {                   // last read of this accumulator: hand it back
                    asm volatile("tcgen05.fence::before_thread_sync;");
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_acc_empty + 8 * acc);
                }
                float f[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    if constexpr (H) f[j] = fmaf(__uint_as_float(w[j]), lsc, __uint_as_float(v[j])) * osc;   // power-of-two scalings: exact
                    else f[j] = (__uint_as_float(v[j]) + __uint_as_float(w[j])) * osc;
                }
                const int col0 = slice * NS + c0;
                if (row < Ts && col0 < a.Ntot) {
                    const long long o = (long long)row * row_pitch + col0;
                    const bool full = col0 + 32 <= a.Ntot && o + 32 <= map_elems;
                    if (full && wide_ok) {
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            asm volatile("st.global.L1::no_allocate.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                                         :: "l"(ms + o + 8 * j), "f"(f[8 * j]), "f"(f[8 * j + 1]), "f"(f[8 * j + 2]), "f"(f[8 * j + 3]),
                                            "f"(f[8 * j + 4]), "f"(f[8 * j + 5]), "f"(f[8 * j + 6]), "f"(f[8 * j + 7]) : "memory");
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            if (col0 + j < a.Ntot && o + j < map_elems) ms[o + j] = f[j];
                    }
                    if (a.keys) {
                        // the chunk lies inside one time row (s == 1, or K % 32 == 0): time row and first filter
                        const int trow = a.s * row + col0 / a.K;
                        const int k0 = col0 % a.K;
                        if (trow < a.T) {
                            float bv = 0.f;
                            int bj = 0;
#pragma unroll
                            for (int j = 0; j < 32; ++j) {
                                const float sc = fabsf(f[j]);
                                if (sc > bv) { bv = sc; bj = j; }
                            }
                            const unsigned long long key = ((unsigned long long)__float_as_uint(bv) << 32) |
                                                           (unsigned long long)(0xFFFFFFFFu - (unsigned)(k0 + bj));
                            atomicMax(a.keys + (long long)sig * a.T + trow, key);
                        }
                    }
                }
            }
#ifdef HSC_PROFILE_PHASES
            ew_work += clock64() - c1_;
#endif
            acc ^= 1;
            if (acc == 0) acc_phase ^= 1;
        }
#ifdef HSC_PROFILE_PHASES
        if (warp == 2 && lane == 0 && a.prof) { a.prof[blockIdx.x * 16 + 5] = ew_wait; a.prof[blockIdx.x * 16 + 6] = ew_work; a.prof[blockIdx.x * 16 + 7] = (long long)((ntiles - cta_m + ctas_per_slice - 1) / ctas_per_slice); }
#endif
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(a.tmem_cols));
}

}  // namespace tc
}  // namespace hsc
