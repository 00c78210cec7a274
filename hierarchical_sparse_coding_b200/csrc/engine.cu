// Host runtime + C ABI of the B200 matching-pursuit engine (include/hsc_b200.h).
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>

#include <string>
#include <vector>

#include "../../include/hsc_b200.h"
#include "common.cuh"
#include "correlate_simt.cuh"
#include "correlate_tc.cuh"
#include "pursuit.cuh"
#include "locomp.cuh"
#include "decode.cuh"
#include "ksvd.cuh"
#include "kmeans.cuh"
#include "events.cuh"

using namespace hsc;

namespace {

size_t align_up(size_t v, size_t a = 256) { return (v + a - 1) / a * a; }

struct Layout {            // workspace carve-up for S signals of T samples
    int G1, n2, G2, n3;
    long long bitmap_words;
    size_t off_map, off_val1, off_idx1, off_val2, off_idx2, off_val3, off_idx3, off_bitmap, off_state, off_keys, off_cand_t, off_cand_k, off_cand_c, off_edge, total;
    long long edge_stride;
    int ncand_max;
};

Layout make_layout(long long S, long long T, long long K, long long L, size_t rsz, long long F = 1) {
    Layout l;
    {   // candidate lists of the block-wise selection: one entry per time block (+1 on offset passes)
        long long c = T / (4 * L) + 8;
        if (c < 1032) c = 1032;
        l.ncand_max = (int)c;
    }
    l.G1 = 128;
    l.n2 = (int)((T + l.G1 - 1) / l.G1);
    int want = (l.n2 + 63) / 64;
    l.G2 = pow2_at_least(want < 32 ? 32 : want);
    l.n3 = (l.n2 + l.G2 - 1) / l.G2;
    l.bitmap_words = (T * K + 31) / 32;
    size_t o = 0;
    l.off_map = o;    o = align_up(o + (size_t)S * T * K * rsz);
    l.off_val1 = o;   o = align_up(o + (size_t)S * T * rsz);
    l.off_idx1 = o;   o = align_up(o + (size_t)S * T * sizeof(int));
    l.off_val2 = o;   o = align_up(o + (size_t)S * l.n2 * rsz);
    l.off_idx2 = o;   o = align_up(o + (size_t)S * l.n2 * sizeof(int));
    l.off_val3 = o;   o = align_up(o + (size_t)S * l.n3 * rsz);
    l.off_idx3 = o;   o = align_up(o + (size_t)S * l.n3 * sizeof(int));
    l.off_bitmap = o; o = align_up(o + (size_t)S * l.bitmap_words * sizeof(unsigned));
    l.off_state = o;  o = align_up(o + (size_t)S * sizeof(hsc_signal_state));
    l.off_keys = o;   o = align_up(o + (size_t)S * T * sizeof(unsigned long long));   // packed level-1 keys out of the K1 epilogue
    l.off_cand_t = o; o = align_up(o + (size_t)S * 2 * l.ncand_max * sizeof(int));
    l.off_cand_k = o; o = align_up(o + (size_t)S * 2 * l.ncand_max * sizeof(int));
    l.off_cand_c = o; o = align_up(o + (size_t)S * 2 * l.ncand_max * rsz);
    l.edge_stride = (3 * L) * F;                               // reflect-padded residual slice of an edge atom (3L-2 samples)
    l.off_edge = o;   o = align_up(o + (size_t)S * l.edge_stride * rsz);
    l.total = o;
    return l;
}

}  // namespace

struct hsc_engine {
    int device = 0;
    std::string err;
    int dtype = -1;
    long long K = 0, L = 0, F = 0;
    void* D_dev = nullptr;
    void* G_dev = nullptr;
    bool gram_valid = false;   // G_dev holds the Gram tensor of the CURRENT dictionary (the buffer is kept across same-shape dictionaries)
    void* w_dev = nullptr;
    bool owns_dict = true;     // false for views (hsc_b200_create_view)
    // tensor-core K1 operand (float, F in {1,2,4}): split + shifted dictionary, per-slice canonical layout
    tc::Plan tc_plan{};
    void* tc_bop = nullptr;
    unsigned char* tc_xsplit = nullptr;   // [2][S][xpad_stride] zero-padded hi / lo parts of the signals, then [S] scales, [S] absmax
    size_t tc_xsplit_bytes = 0;
    cudaGraphExec_t ksvd_graph = nullptr;     // the captured sweep of hsc_b200_ksvd_update and what it was captured for
    unsigned char* ksvd_graph_scratch = nullptr;
    long long ksvd_graph_cap = 0, ksvd_graph_key[5] = {0, 0, 0, 0, 0}, ksvd_graph_launches = 0;
    long long ksvd_same_key_sweeps = 0;       // consecutive sweeps of the same shape: the graph is captured from the third on
    bool ksvd_graph_disabled = false;         // a capture failed once: sweeps run eagerly
    bool ksvd_chain_failed = false;           // the cluster launch of square_chain_kernel was refused once: separate kernels
    int ksvd_pca = 0;                         // hsc_b200_ksvd_set_pca: usePCA=True variant of the one-shot update (:618-625)
    unsigned char* ksvd_scratch = nullptr;    // scratch of the dictionary-update sweeps, kept between sweeps (cudaMalloc / cudaFree per sweep cost milliseconds)
    size_t ksvd_scratch_bytes = 0;
    double* locomp_scratch = nullptr;     // [S][256*257] doubles, allocated at the first LoCOMP run
    size_t locomp_scratch_signals = 0;
    unsigned char* canon_scratch = nullptr;   // hsc_b200_canonicalize_codes: sort keys of long signals, per-level counts
    size_t canon_scratch_bytes = 0;
    long long launches = 0;
    // encode in flight
    bool active = false;
    long long S = 0, T = 0;
    Layout lay{};
    unsigned char* ws = nullptr;
    void* resid = nullptr;
    hsc_mp_options opt{};
};

namespace {

int fail(hsc_engine* e, int code, const std::string& msg) {
    if (e) e->err = msg;
    return code;
}

#define HSC_CUDA(e, call)                                                                          \
    do {                                                                                           \
        cudaError_t _err = (call);                                                                 \
        if (_err != cudaSuccess)                                                                   \
            return fail((e), HSC_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(_err));    \
    } while (0)

template <typename real>
int set_dictionary_t(hsc_engine* e, const void* D_host, const void* w_host) {
    // Device buffers are kept when the new dictionary has the shape of the previous one (hsc_b200_set_dictionary): a
    // dictionary-learning loop sends a new one every iteration, and cudaFree / cudaMalloc of the 100+ MB Gram tensor next to a
    // 26 GB workspace stalled for up to a second now and then (config 5: set_dictionary 2 ms .. 1 s, tools/gpu_r2_ksvd_probe.sh).
    const size_t nD = (size_t)e->K * e->L * e->F;
    if (!e->D_dev) HSC_CUDA(e, cudaMalloc(&e->D_dev, nD * sizeof(real)));
    HSC_CUDA(e, cudaMemcpy(e->D_dev, D_host, nD * sizeof(real), cudaMemcpyHostToDevice));
    e->gram_valid = false;
    if (w_host) {
        if (!e->w_dev) HSC_CUDA(e, cudaMalloc(&e->w_dev, (size_t)e->K * sizeof(real)));
        HSC_CUDA(e, cudaMemcpy(e->w_dev, w_host, (size_t)e->K * sizeof(real), cudaMemcpyHostToDevice));
    }
    // the shift Gram tensor is built at the first pursuit (ensure_gram): decoding and plain correlation do not need it
    e->tc_plan = tc::Plan{};
    if (sizeof(real) == 4) {
        // operand format of the tensor-core K1: 3xFP16 (kind::f16, twice the tf32 rate) unless HSC_K1=tf32
        static const bool want_tf32 = getenv("HSC_K1") && !strcmp(getenv("HSC_K1"), "tf32");
        // HSC_K1_NS: columns per N-slice (multiple of 32, <= 128).  128 is the fastest stand-alone shape; 64 halves the
        // dictionary slice a CTA keeps in shared memory (70 KB at config 4), which lets two pursuit CTAs share the SM with it
        static const int ns_max = getenv("HSC_K1_NS") ? atoi(getenv("HSC_K1_NS")) : 128;
        tc::Plan p = tc::make_plan((int)e->K, (int)e->L, (int)e->F, !want_tf32, ns_max);
        if (!p.ok && !want_tf32) p = tc::make_plan((int)e->K, (int)e->L, (int)e->F, false, ns_max);
        if (p.ok) {
            // expanded / shifted / split dictionary operand, built on the device from the uploaded D (the padding of the
            // last slice stays zero); tc::build_b_operand is the host restatement of the same layout
            const size_t bytes = (size_t)p.nslices * 2 * p.NS * p.Kd * p.esz;
            {
                float mx = 0.f;
                const float* Dh = (const float*)D_host;
                for (size_t i = 0; i < nD; ++i) mx = fmaxf(mx, fabsf(Dh[i]));
                p.d_scale = ldexpf(1.f, tc::split_exponent(mx, -1));      // max|D|*scale in [0.5, 1)
            }
            if (!e->tc_bop) HSC_CUDA(e, cudaMalloc(&e->tc_bop, bytes));
            HSC_CUDA(e, cudaMemset(e->tc_bop, 0, bytes));
            const long long total = (long long)p.Ntot * p.Kd;
            unsigned blocks = (unsigned)((total + 255) / 256);
            if (blocks > 148 * 16) blocks = 148 * 16;
            tc::build_b_operand_kernel<<<blocks, 256>>>((const float*)e->D_dev, (int)e->K, (int)e->L, (int)e->F, p.half, p.R, p.s, p.Kd,
                                                        p.Ntot, p.NS, p.d_scale, e->tc_bop);
            e->launches++;
            HSC_CUDA(e, cudaGetLastError());
            HSC_CUDA(e, cudaDeviceSynchronize());
            e->tc_plan = p;
        }
    }
    return HSC_OK;
}

// Builds the shift Gram tensor G[k][tau+L-1][k'] of the current dictionary if it has not been built yet.
int ensure_gram(hsc_engine* e) {
    if (e->G_dev && (e->gram_valid || !e->owns_dict)) return HSC_OK;
    if (!e->owns_dict) return fail(e, HSC_E_STATE, "view without a Gram tensor");
    const size_t rsz = e->dtype == HSC_F32 ? 4 : 8;
    const size_t nG = (size_t)e->K * (2 * e->L - 1) * e->K;
    if (!e->G_dev) HSC_CUDA(e, cudaMalloc(&e->G_dev, nG * rsz));
    int blocks = (int)((nG + 255) / 256);
    if (blocks > 148 * 32) blocks = 148 * 32;
    if (e->dtype == HSC_F32) gram_kernel<float><<<blocks, 256>>>((const float*)e->D_dev, (float*)e->G_dev, (int)e->K, (int)e->L, (int)e->F);
    else gram_kernel<double><<<blocks, 256>>>((const double*)e->D_dev, (double*)e->G_dev, (int)e->K, (int)e->L, (int)e->F);
    e->launches++;
    HSC_CUDA(e, cudaGetLastError());
    HSC_CUDA(e, cudaDeviceSynchronize());
    e->gram_valid = true;
    return HSC_OK;
}

int correlate_tc(hsc_engine* e, const void* x, long long S, long long T, void* map, cudaStream_t st,
                 unsigned long long* keys = nullptr) {
    const tc::Plan& p = e->tc_plan;
    tc::Args a;
    const long long Ts_ = (T + p.s - 1) / p.s;
    const long long MT_ = (Ts_ + tc::kTileM - 1) / tc::kTileM;
    const long long xstride = (long long)p.R * MT_ * tc::kTileM + p.Kd;    // elements per padded signal (multiple of R)
    const size_t part_bytes = ((size_t)S * xstride * p.esz + 255) / 256 * 256;
    const size_t need = 2 * part_bytes + 2 * (((size_t)S * 4 + 255) / 256 * 256);
    if (e->tc_xsplit_bytes < need) {
        if (e->tc_xsplit) cudaFree(e->tc_xsplit);
        e->tc_xsplit = nullptr; e->tc_xsplit_bytes = 0;
        HSC_CUDA(e, cudaMalloc((void**)&e->tc_xsplit, need));
        e->tc_xsplit_bytes = need;
    }
    unsigned char* xhi = e->tc_xsplit;
    unsigned char* xlo = e->tc_xsplit + part_bytes;
    float* out_scale = (float*)(e->tc_xsplit + 2 * part_bytes);
    unsigned* absmax = (unsigned*)(e->tc_xsplit + 2 * part_bytes + (((size_t)S * 4 + 255) / 256 * 256));
    {
        unsigned bx = (unsigned)((xstride + 255) / 256);
        if (bx > 1024) bx = 1024;
        dim3 grid(bx, (unsigned)S);
        const int pad_front = centre_offset((int)e->L) * (int)e->F;
        HSC_CUDA(e, cudaMemsetAsync(absmax, 0, (size_t)S * 4, st));
        // few blocks per signal: one atomicMax per warp on the signal's slot (a (1024, S) grid spent 0.6 ms in atomics)
        const long long nval = (long long)T * e->F;
        unsigned ax = (unsigned)((nval + 256 * 64 - 1) / (256 * 64));
        if (ax < 1) ax = 1;
        if (ax > 16) ax = 16;
        tc::signal_absmax_kernel<<<dim3(ax, (unsigned)S), 256, 0, st>>>((const float*)x, nval, absmax);
        if (p.half) {
            static const bool scalar_split = getenv("HSC_K1_SPLIT_SCALAR") != nullptr;
            if (!scalar_split && pad_front % 4 == 0 && nval % 4 == 0 && xstride % 8 == 0 && ((uintptr_t)x & 15) == 0) {
                unsigned gx = (unsigned)((xstride / 8 + 255) / 256);
                if (gx > 1024) gx = 1024;
                tc::split_signal_half_vec8_kernel<<<dim3(gx, (unsigned)S), 256, 0, st>>>((const float*)x, (__half*)xhi, (__half*)xlo, nval,
                                                                                         xstride, pad_front, absmax, 1.f / p.d_scale, out_scale);
            } else {
                tc::split_signal_half_kernel<<<grid, 256, 0, st>>>((const float*)x, (__half*)xhi, (__half*)xlo, nval, xstride,
                                                                   pad_front, absmax, 1.f / p.d_scale, out_scale);
            }
        } else {
            tc::split_signal_kernel<<<grid, 256, 0, st>>>((const float*)x, (float*)xhi, (float*)xlo, nval, xstride, pad_front,
                                                          absmax, 1.f / p.d_scale, out_scale);
        }
        e->launches += 2;
        HSC_CUDA(e, cudaGetLastError());
    }
    a.x_hi = xhi; a.x_lo = xlo; a.xpad_stride = xstride; a.b_op = e->tc_bop; a.map = (float*)map;
    a.out_scale = out_scale;
    a.S = (int)S; a.T = (int)T; a.F = (int)e->F; a.K = (int)e->K; a.off = centre_offset((int)e->L);
    a.s = p.s; a.Kd = p.Kd; a.Ntot = p.Ntot; a.NS = p.NS; a.nslices = p.nslices; a.slab_elems = p.slab_elems;
    a.slab_stride_bytes = p.slab_stride_bytes;
    a.tmem_cols = pow2_at_least(4 * p.NS < 32 ? 32 : 4 * p.NS);
    if (p.half) HSC_CUDA(e, cudaFuncSetAttribute(tc::correlate_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem_bytes));
    else HSC_CUDA(e, cudaFuncSetAttribute(tc::correlate_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem_bytes));
    // CTAs per N-slice: g = 8 per SM (HSC_K1_GRID_MULT), each striding over 1/g of an SM's share of the (signal, M-tile)
    // list, so that the block scheduler hands tiles to whichever SMs are free: in the streaming pipeline the correlation of
    // batch i+1 runs under the tail of batch i's pursuit, where SMs become available one by one (a strictly persistent
    // grid would finish 11 ms after its LAST CTA found a free SM).  Stand-alone the finer grid costs nothing measurable
    // (11.2 ms either way): a CTA's set-up - 139 KB dictionary slice from L2, TMEM allocation - is ~5 us per 1.4 ms of tiles.
    static const int grid_mult = getenv("HSC_K1_GRID_MULT") ? atoi(getenv("HSC_K1_GRID_MULT")) : 8;
    int per_slice = (148 / p.nslices) * (grid_mult > 0 ? grid_mult : 1);
    const long long Ts = (T + p.s - 1) / p.s;
    const long long tiles = S * ((Ts + tc::kTileM - 1) / tc::kTileM);
    if (per_slice > tiles) per_slice = (int)tiles;
    if (per_slice < 1) per_slice = 1;
    a.keys = keys;
    a.prof = nullptr;
#ifdef HSC_PROFILE_PHASES
    static long long* tc_prof = nullptr;
    if (!tc_prof) cudaMalloc((void**)&tc_prof, 148 * 64 * 16 * sizeof(long long));
    cudaMemsetAsync(tc_prof, 0, 148 * 64 * 16 * sizeof(long long), st);
    a.prof = tc_prof;
#endif
    if (p.half) tc::correlate_tc_kernel<true><<<p.nslices * per_slice, tc::kThreads, p.smem_bytes, st>>>(a);
    else tc::correlate_tc_kernel<false><<<p.nslices * per_slice, tc::kThreads, p.smem_bytes, st>>>(a);
    e->launches++;
    HSC_CUDA(e, cudaGetLastError());
#ifdef HSC_PROFILE_PHASES
    {
        const int n = p.nslices * per_slice;
        std::vector<long long> h((size_t)n * 16);
        cudaStreamSynchronize(st);
        cudaMemcpy(h.data(), tc_prof, h.size() * sizeof(long long), cudaMemcpyDeviceToHost);
        double t[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        double pload = 0;
        for (int i = 0; i < n; ++i) { for (int j = 0; j < 8; ++j) t[j] += (double)h[(size_t)i * 16 + j]; pload += (double)h[(size_t)i * 16 + 8]; }
        const double tiles = t[7] > 0 ? t[7] : 1;
        fprintf(stderr, "[hsc K1 tc, cycles per tile] producer wait %.0f work %.0f | mma wait-slab %.0f wait-acc %.0f issue %.0f | epilogue wait %.0f work %.0f (tiles/CTA %.0f)\n",
                t[0] / tiles, t[1] / tiles, t[2] / tiles, t[3] / tiles, t[4] / tiles, t[5] / tiles, t[6] / tiles, tiles / n);
    }
#endif
    return HSC_OK;
}

template <typename real>
int correlate_t(hsc_engine* e, const void* x, long long S, long long T, void* map, cudaStream_t st) {
    static const bool force_simt = getenv("HSC_K1") && !strcmp(getenv("HSC_K1"), "simt");
    if (sizeof(real) == 4 && e->tc_plan.ok && !force_simt && T * e->K < (1ll << 31)) return correlate_tc(e, x, S, T, map, st);
    bool ok = false;
    cudaError_t err = launch_correlate<real>((const real*)x, (const real*)e->D_dev, (real*)map, S, (int)T, (int)e->K,
                                             (int)e->L, (int)e->F, st, &ok);
    if (err != cudaSuccess) return fail(e, HSC_E_CUDA, std::string("correlate launch: ") + cudaGetErrorString(err));
    if (!ok) return fail(e, HSC_E_UNSUPPORTED, "correlate: (L-1+tile)*F slab does not fit in shared memory");
    e->launches++;
    return HSC_OK;
}

template <typename real>
int run_t(hsc_engine* e, int32_t* evp, int32_t* evi, void* evc, long long cap, cudaStream_t st) {
    MpArgs<real> a;
    const Layout& l = e->lay;
    a.T = (int)e->T; a.K = (int)e->K; a.L = (int)e->L; a.F = (int)e->F; a.off = centre_offset((int)e->L);
    a.G1 = l.G1; a.n2 = l.n2; a.G2 = l.G2; a.n3 = l.n3;
    a.D = (const real*)e->D_dev; a.G = (const real*)e->G_dev;
    a.w = (e->opt.use_weights && e->w_dev) ? (const real*)e->w_dev : nullptr;
    a.map = (real*)(e->ws + l.off_map);
    a.resid = (real*)e->resid;
    a.val1 = (real*)(e->ws + l.off_val1); a.idx1 = (int*)(e->ws + l.off_idx1);
    a.val2 = (real*)(e->ws + l.off_val2); a.idx2 = (int*)(e->ws + l.off_idx2);
    a.val3 = (real*)(e->ws + l.off_val3); a.idx3 = (int*)(e->ws + l.off_idx3);
    a.bitmap = (unsigned*)(e->ws + l.off_bitmap); a.bitmap_words = l.bitmap_words;
    a.state = (hsc_signal_state*)(e->ws + l.off_state);
    a.ev_pos = evp; a.ev_idx = evi; a.ev_coef = (real*)evc; a.cap = cap;
    a.max_nnz = e->opt.nb_nonzero_coefs;
    a.has_snr = !isnan(e->opt.tolerance_snr); a.tol_snr = a.has_snr ? (real)e->opt.tolerance_snr : (real)0;
    a.has_scale = !isnan(e->opt.tolerance_residual_scale);
    a.tol_scale = a.has_scale ? (real)e->opt.tolerance_residual_scale : (real)0;
    a.null_thres = (real)e->opt.min_coefficients;
    a.eps = sizeof(real) == 4 ? (real)1.1920928955078125e-07 : (real)2.220446049250313e-16;   // np.finfo(dtype).eps (:1057)
    if (e->opt.energy_eps > 0.0) a.eps = (real)e->opt.energy_eps;                             // ... of the DICTIONARY's dtype, given by the caller
    a.coef_mode = e->opt.coef_mode;
    a.max_passes = e->opt.max_passes_per_run;
    a.max_events_total = e->opt.max_events_total;
    a.nb_blocks = e->opt.nb_blocks;
    a.ncand_max = l.ncand_max;
    a.edge_ext = (real*)(e->ws + l.off_edge); a.edge_stride = l.edge_stride;
    a.cand_t = (int*)(e->ws + l.off_cand_t); a.cand_k = (int*)(e->ws + l.off_cand_k); a.cand_c = (real*)(e->ws + l.off_cand_c);
    a.prof = nullptr;
    a.locomp_scratch = nullptr;
    {   // near-tie re-ranking window of float maps (hsc_mp_options::rerank_tolerance); HSC_RERANK overrides (0 = off)
        static const char* rr_env = getenv("HSC_RERANK");
        double tol = e->opt.rerank_tolerance < 0.0 ? 4e-6 : e->opt.rerank_tolerance;
        if (rr_env) tol = atof(rr_env);
        a.rerank_tol = sizeof(real) == 4 ? (float)tol : 0.f;
    }
    {   // HSC_K2_EARLY_ISSUE=1: the first window chunks are issued right after the pick barrier, before the bookkeeping and
        // the residual update.  Measured (interleaved A/B): no gain on the config-4 shard, 3-4 % slower per atom on the
        // latency-bound single sequences of configs 1-3; off.  (Issuing them even earlier - every warp as soon as the PICK
        // is known, handed over through a 256-thread named barrier, overlapping the coefficient's round trip - was built
        // and measured too: no gain either; not kept.)
        static const int early = getenv("HSC_K2_EARLY_ISSUE") ? atoi(getenv("HSC_K2_EARLY_ISSUE")) : 0;
        a.early_issue = early > 0 ? 1 : 0;
        // HSC_K2_NEXT_PREFETCH: the watch warp pulls the residual / map row / keys of the likely next pick (the best entry of
        // the other groups, found through the block scores) towards L2.  Measured (interleaved A/B): within noise on the
        // config-4 shard (23.1-23.5 vs 23.6 ms), 10 % slower on the single 1e6-sample sequence (6.7 -> 7.4 us per selection:
        // the lookup is on that chain), 4-5 % faster at config 5 (19.5 -> 18.6 ms: wide rows, at most two CTAs per SM, so the
        // chain of one signal is what the launch lasts).  Default: on for wide-row launches of at most two CTAs per SM.
        static const int nextpf = getenv("HSC_K2_NEXT_PREFETCH") ? atoi(getenv("HSC_K2_NEXT_PREFETCH")) : -1;
        a.next_prefetch = nextpf >= 0 ? (nextpf > 0 ? 1 : 0)
                                      : ((e->K * sizeof(real)) / 16 >= 32 && e->S > 1 && e->S <= 2 * 148 ? 1 : 0);
    }
    static const int prefetch = getenv("HSC_PREFETCH") ? atoi(getenv("HSC_PREFETCH")) : -1;
    a.prefetch = prefetch;        // -1: decided below (on for the register path, off when the window is staged by bulk copies)
    // Interior window update staged through shared memory by bulk copies (gram_update_tma): map rows of 16-byte
    // multiples only.  Per warp a ring of NS stages, each RPS*32/g map rows + the matching Gram rows (g lanes per row);
    // NS as large as fits in 48 KB per CTA (4 CTAs resident per SM), or 72 KB (3 per SM) for wide dictionaries.
    // Launch shapes: 4 = 8 warps per signal, 64 registers; 6 = 4 warps, 128 registers, two rows per lane group and step.
    static const int variant = getenv("HSC_PURSUIT_VARIANT") ? atoi(getenv("HSC_PURSUIT_VARIANT")) : 4;
    static const int tma_mode = getenv("HSC_K2_TMA") ? atoi(getenv("HSC_K2_TMA")) : 1;
    static const int tma_stages_max = getenv("HSC_K2_TMA_STAGES") ? atoi(getenv("HSC_K2_TMA_STAGES")) : 4;
    // (L2 eviction-priority hints on these copies - Gram evict_last, map evict_first - were measured twice: DRAM reads
    //  59.3 -> 50.6 GB per launch on config 4, kernel time unchanged - also with the lean window loop, where K2 is closer to
    //  the DRAM bound: 23.7 ms either way, 1.5 % at config 5; not used.)
    a.tma_rows = a.tma_stages = a.tma_bytes = 0;
    size_t dyn_smem = 0;
    int rps = 1;
    const size_t row_bytes = (size_t)e->K * sizeof(real);
    const int NW = variant == 6 ? 4 : 8;                        // warps per CTA of the launch shape
    if (tma_mode && variant != 0 && row_bytes % 16 == 0) {      // (LoCOMP: only its fast kernel uses the rings, see below)
        const int VN = 16 / (int)sizeof(real);
        const int nvec = (int)e->K / VN;
        const int gv = nvec >= 32 ? 32 : pow2_at_least(nvec);
        const int W = 2 * (int)e->L - 1;
        const int rpw = 32 / gv;
        if (variant == 6 && (size_t)NW * 3 * 2 * 2 * rpw * row_bytes <= 48 * 1024 && W >= 2 * NW * 2 * rpw) rps = 2;
        const size_t stage = (size_t)NW * 2 * rpw * rps * row_bytes;  // one stage of every warp
        const int steps = (W + NW * rpw * rps - 1) / (NW * rpw * rps);
        int ns = (int)((48 * 1024) / stage);
        if (ns < 2) ns = (int)((72 * 1024) / stage);
        // a launch of at most two CTAs per SM (config 5's 190 segments of 2 KB rows) can afford a third stage: 23.0 -> 22.3 ms
        if (ns < 3 && e->S <= 2 * 148) ns = (int)((100 * 1024) / stage) < 3 ? ns : 3;
        {   // HSC_K2_RING_KB: shared memory the stage rings of one CTA may take (default: 48 KB, i.e. 4 CTAs per SM; 72 KB when
            // that holds fewer than two stages)
            static const int ring_kb = getenv("HSC_K2_RING_KB") ? atoi(getenv("HSC_K2_RING_KB")) : 0;
            if (ring_kb > 0) ns = (int)(((size_t)ring_kb * 1024) / stage);
        }
        if (ns > tma_stages_max) ns = tma_stages_max;
        if (ns > steps) ns = steps;
        if (ns > 32 / NW) ns = 32 / NW;
        if (ns >= 1) {
            a.tma_rows = rpw * rps; a.tma_stages = ns;
            dyn_smem = stage * ns;
            a.tma_bytes = (int)dyn_smem;
        }
    }
    // Narrow maps (rows of at most 32 bytes: K <= 8 floats - config 1, level 0 of config 3): a 2L-1 row window is a KB or
    // two, and staging it through bulk copies costs more in fixed latency (mbarrier round trip, store drain, proxy fences)
    // than it saves; they take the plain register window path (cached loads / stores, no streaming hints: the whole map
    // lives in L2), still under the shared-memory argmax hierarchy.  Measured per selection, interleaved A/B: config 1
    // 9.3 -> 6.4 us, config 3 18.3 -> 15.6 ms; at 64-byte rows (config 2) the bulk-copy path is the faster one (10.2 vs
    // 11.3 us vectorised / 12.2 us scalar), hence the threshold.  HSC_K2_TINYROW=0 switches it off.
    static const int tiny_mode = getenv("HSC_K2_TINYROW") ? atoi(getenv("HSC_K2_TINYROW")) : 1;
    const size_t slot3_bytes = ((size_t)(l.n2 + 31) / 32) * sizeof(unsigned);      // block level of the shared-memory hierarchy (select_smh)
    bool tiny_row = tiny_mode && dyn_smem > 0 && sizeof(real) == 4 && row_bytes <= 32 && variant == 4;
    {   // ... only where the shared-memory hierarchy applies without the stage rings too
        const bool fits = l.n2 <= kSlotMax || (e->S <= 148 && (size_t)l.n2 * sizeof(unsigned long long) + slot3_bytes <= 200 * 1024);
        const bool smh_ok = (getenv("HSC_K2_SMH") ? atoi(getenv("HSC_K2_SMH")) : 1) && l.G1 == 128 && fits &&
                            (2 * e->L - 1 + l.G1 - 1) / l.G1 + 1 <= kDirtyMax && (long long)l.G1 * e->K < (1ll << 32);
        tiny_row = tiny_row && smh_ok;
    }
    a.scalar_window = 0;
    {   // HSC_K2_ROW32=0: wide rows through the general window loop (gram_update_tma) instead of gram_update_row32
        // (a variant with two map rows per chunk and the Gram rows read straight from global memory - half the stage bytes, one bulk
        //  load per chunk - was measured slower: K2 25.5 -> 27.3 ms at config 4, 23.2 -> 34.6 ms at config 5, whose Gram tensor
        //  does not fit L2)
        static const int row32 = getenv("HSC_K2_ROW32") ? atoi(getenv("HSC_K2_ROW32")) : 1;
        const bool wide = dyn_smem > 0 && variant == 4 && (e->K * sizeof(real)) / 16 >= 32 && !a.w;
        a.row32 = (wide && row32) ? 1 : 0;
    }
    if (tiny_row) {
        dyn_smem = 0;
        a.tma_rows = a.tma_stages = a.tma_bytes = 0;
        a.scalar_window = 1;
    }
    if (a.prefetch < 0) a.prefetch = dyn_smem > 0 ? 0 : 1;
#ifdef HSC_PROFILE_PHASES
    static long long* prof_dev = nullptr;
    if (!prof_dev) cudaMalloc((void**)&prof_dev, 65536 * 16 * sizeof(long long));
    cudaMemsetAsync(prof_dev, 0, (size_t)e->S * 16 * sizeof(long long), st);
    a.prof = prof_dev;
#endif
    if (e->opt.method == 1) {
        if (cap < 2 * kLocompMaxGroup) return fail(e, HSC_E_INVALID, "mp_run: LoCOMP needs an event capacity of at least 512 per signal");
        if (e->locomp_scratch_signals < (size_t)e->S) {
            if (e->locomp_scratch) cudaFree(e->locomp_scratch);
            e->locomp_scratch = nullptr; e->locomp_scratch_signals = 0;
            HSC_CUDA(e, cudaMalloc((void**)&e->locomp_scratch, (size_t)e->S * kLocompScratchStride * sizeof(double)));
            e->locomp_scratch_signals = (size_t)e->S;
        }
        a.locomp_scratch = e->locomp_scratch;
        // Fast kernel (locomp_fast_kernel): float maps with wide rows (32 lanes per row), no filter weights, the shared-memory
        // hierarchy within its 4-CTAs-per-SM budget and stage rings large enough for the refit scratch laid over them.
        // HSC_LOCOMP_FAST=0 keeps the original kernel (the two produce the same events: tests/test_parity_gpu.py).
        const int fast_mode = getenv("HSC_LOCOMP_FAST") ? atoi(getenv("HSC_LOCOMP_FAST")) : 1;      // (read per call: the A/B test flips it)
        bool fast = false;
        if constexpr (sizeof(real) == 4) {
            fast = fast_mode && variant == 4 && dyn_smem > 0 && !tiny_row && !a.w && (e->K * sizeof(real)) / 16 >= 32 && l.G1 == 128 &&
                   l.n2 <= kSlotMax && a.tma_bytes >= kLocompOverlayBytes && a.tma_stages >= 1 &&
                   (2 * e->L - 1 + l.G1 - 1) / l.G1 + 1 <= kDirtyMax && (long long)l.G1 * e->K < (1ll << 32);
            if (fast) {
                const size_t smem = dyn_smem + (size_t)l.n2 * sizeof(unsigned long long) + slot3_bytes;
                HSC_CUDA(e, cudaFuncSetAttribute(locomp_fast_kernel<float, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                locomp_fast_kernel<float, 256><<<(unsigned)e->S, 256, smem, st>>>(a);
            }
        }
        if (!fast) {
            a.tma_rows = a.tma_stages = a.tma_bytes = 0;
            locomp_kernel<real, 128><<<(unsigned)e->S, 128, 0, st>>>(a);      // 4 CTAs of 128 threads x 128 registers per SM
        }
        e->launches++;
        HSC_CUDA(e, cudaGetLastError());
        return HSC_OK;
    }
    // shared-memory argmax hierarchy: float scores, one packed key per 128-row group, <= kDirtyMax groups per window
    static const int smh_mode = getenv("HSC_K2_SMH") ? atoi(getenv("HSC_K2_SMH")) : 1;
    // one 8-byte key per 128-row group: up to kSlotMax groups keep 4 CTAs per SM; a launch of at most one CTA per SM
    // (few, long sequences: config 2) may spend most of the SM's shared memory on them instead
    const bool slots_fit = l.n2 <= kSlotMax || (e->S <= 148 && dyn_smem + (size_t)l.n2 * sizeof(unsigned long long) + slot3_bytes <= 200 * 1024);
    const bool smh = (dyn_smem > 0 || tiny_row) && smh_mode && sizeof(real) == 4 && l.G1 == 128 && slots_fit && (l.G1 % 32) == 0 &&
                     (2 * e->L - 1 + l.G1 - 1) / l.G1 + 1 <= kDirtyMax && (long long)l.G1 * e->K < (1ll << 32);
    if (smh) dyn_smem += (size_t)l.n2 * sizeof(unsigned long long) + slot3_bytes;
    {   // HSC_K2_SMEM_KB: request at least this much dynamic shared memory per pursuit CTA, i.e. cap the CTAs per SM from
        // the host (76 KB -> two per SM), leaving room for a correlation CTA of the next batch on every SM (streaming pipeline)
        static const int smem_kb = getenv("HSC_K2_SMEM_KB") ? atoi(getenv("HSC_K2_SMEM_KB")) : 0;
        if (smem_kb > 0 && dyn_smem > 0 && dyn_smem < (size_t)smem_kb * 1024) dyn_smem = (size_t)smem_kb * 1024;
    }
#define HSC_LAUNCH_K2(NT_, MINB_, VIF_, TMA_, SMH_, RPS_)                                                                        \
    do {                                                                                                                          \
        if (dyn_smem > 0)                                                                                                         \
            HSC_CUDA(e, cudaFuncSetAttribute(pursuit_kernel<real, NT_, MINB_, VIF_, TMA_, SMH_, RPS_>,                            \
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn_smem));                        \
        pursuit_kernel<real, NT_, MINB_, VIF_, TMA_, SMH_, RPS_><<<(unsigned)e->S, NT_, dyn_smem, st>>>(a);                       \
    } while (0)
    switch (variant) {
        case 0:            // register path, 2 CTAs per SM
            HSC_LAUNCH_K2(256, 2, 4, false, false, 1);
            break;
        case 6:            // 4 warps per signal, 128 registers per thread
            if (dyn_smem > 0 && smh && rps == 2) HSC_LAUNCH_K2(128, 4, 2, true, true, 2);
            else if (dyn_smem > 0 && smh) HSC_LAUNCH_K2(128, 4, 2, true, true, 1);
            else if (dyn_smem > 0 && rps == 2) HSC_LAUNCH_K2(128, 4, 2, true, false, 2);
            else if (dyn_smem > 0) HSC_LAUNCH_K2(128, 4, 2, true, false, 1);
            else HSC_LAUNCH_K2(128, 4, 2, false, false, 1);
            break;
        default:           // 8 warps per signal, 64 registers per thread
            if (tiny_row && smh) HSC_LAUNCH_K2(256, 4, 2, false, true, 1);
            else if (dyn_smem > 0 && smh) HSC_LAUNCH_K2(256, 4, 2, true, true, 1);
            else if (dyn_smem > 0) HSC_LAUNCH_K2(256, 4, 2, true, false, 1);
            else HSC_LAUNCH_K2(256, 4, 2, false, false, 1);
            break;
    }
#undef HSC_LAUNCH_K2
    e->launches++;
    HSC_CUDA(e, cudaGetLastError());
#ifdef HSC_PROFILE_PHASES
    {
        std::vector<long long> h((size_t)e->S * 16);
        cudaStreamSynchronize(st);
        cudaMemcpy(h.data(), a.prof, h.size() * sizeof(long long), cudaMemcpyDeviceToHost);
        double tot[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        for (long long i = 0; i < e->S; ++i) for (int j = 0; j < 8; ++j) tot[j] += (double)h[(size_t)i * 16 + j];
        fprintf(stderr, "[hsc phases, mean cycles per signal] loop-top %.0f select %.0f [book %.0f resid %.0f window %.0f wait %.0f] level2 %.0f level3 %.0f\n",
                tot[0] / e->S, tot[1] / e->S, tot[5] / e->S, tot[6] / e->S, tot[7] / e->S, tot[2] / e->S, tot[3] / e->S, tot[4] / e->S);
        // per-CTA timeline (globaltimer, ns): start skew, init time, loop time; grouped by how many CTAs share the SM
        long long t0 = h[9];
        for (long long i = 0; i < e->S; ++i) if (h[(size_t)i * 16 + 9] < t0) t0 = h[(size_t)i * 16 + 9];
        std::vector<int> per_sm(256, 0);
        for (long long i = 0; i < e->S; ++i) per_sm[(size_t)(h[(size_t)i * 16 + 8] & 255)]++;
        double sum_start[8] = {0}, sum_init[8] = {0}, sum_loop[8] = {0}, max_end[8] = {0};
        int cnt[8] = {0};
        for (long long i = 0; i < e->S; ++i) {
            const long long* r = &h[(size_t)i * 16];
            int c = per_sm[(size_t)(r[8] & 255)];
            if (c > 7) c = 7;
            cnt[c]++;
            sum_start[c] += (double)(r[9] - t0); sum_init[c] += (double)(r[10] - r[9]); sum_loop[c] += (double)(r[11] - r[10]);
            if ((double)(r[11] - t0) > max_end[c]) max_end[c] = (double)(r[11] - t0);
        }
        if (const char* dump = getenv("HSC_PROF_DUMP")) {
            FILE* f = fopen(dump, "w");
            if (f) {
                fprintf(f, "signal,smid,start_ns,init_ns,loop_ns,end_ns,looptop,select,wait,level2,level3,book,resid,window\n");
                for (long long i = 0; i < e->S; ++i) {
                    const long long* r = &h[(size_t)i * 16];
                    fprintf(f, "%lld,%lld,%lld,%lld,%lld,%lld,%lld,%lld,%lld,%lld,%lld,%lld,%lld,%lld\n", i, r[8], r[9] - t0, r[10] - r[9], r[11] - r[10],
                            r[11] - t0, r[0], r[1], r[2], r[3], r[4], r[5], r[6], r[7]);
                }
                fclose(f);
            }
        }
        {
            double ec = 0, er = 0, en = 0, ecl = 0;
            for (long long i = 0; i < e->S; ++i) { ec += (double)h[(size_t)i * 16 + 12]; er += (double)h[(size_t)i * 16 + 13]; en += (double)h[(size_t)i * 16 + 14]; ecl += (double)h[(size_t)i * 16 + 15]; }
            fprintf(stderr, "[hsc edge path] %.0f edge atoms (%.0f clipped): recompute %.0f cycles/atom, rekey %.0f cycles/atom\n", en, ecl, en > 0 ? ec / en : 0.0, en > 0 ? er / en : 0.0);
        }
        for (int c = 1; c < 8; ++c)
            if (cnt[c])
                fprintf(stderr, "[hsc timeline] CTAs on SMs holding %d: n=%d  mean start %.3f ms, init %.3f ms, loop %.3f ms, last exit %.3f ms\n",
                        c, cnt[c], sum_start[c] / cnt[c] / 1e6, sum_init[c] / cnt[c] / 1e6, sum_loop[c] / cnt[c] / 1e6, max_end[c] / 1e6);
    }
#endif
    return HSC_OK;
}

// offsets == nullptr: one signal, atoms [0, n); otherwise S signals, atoms of signal s in [offsets[s], offsets[s+1]).
template <typename real>
int decode_t(hsc_engine* e, const int64_t* offsets, const int32_t* pos, const int32_t* idx, const void* coef, long long n,
             long long S, long long T, void* out, cudaStream_t st) {
    long long total = S * T * e->F;
    long long blocks = (total + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    if (blocks < 1) blocks = 1;
    decode_gather_kernel<real><<<(unsigned)blocks, 256, 0, st>>>((const long long*)offsets, n, pos, idx, (const real*)coef,
                                                                 (const real*)e->D_dev, S, (int)T, (int)e->K, (int)e->L, (int)e->F,
                                                                 centre_offset((int)e->L), (real*)out);
    e->launches++;
    HSC_CUDA(e, cudaGetLastError());
    return HSC_OK;
}

template <typename real>
int canonicalize_t(hsc_engine* e, const int64_t* offsets, const int32_t* pos, const int32_t* idx, const void* coef, long long capacity,
                   long long S, long long K, const events::LevelBounds& lb, double min_coef, int64_t* out_offsets, int32_t* out_pos,
                   int32_t* out_idx, double* out_coef, cudaStream_t st) {
    const long long L = lb.n + 1;
    const size_t off_ev = align_up((size_t)capacity * sizeof(long long));
    const size_t off_counts = off_ev + align_up((size_t)capacity * sizeof(int));
    const size_t need = off_counts + (size_t)L * S * sizeof(long long);
    if (e->canon_scratch_bytes < need) {          // grows only (cudaFree waits for the launches that may still use it)
        if (e->canon_scratch) cudaFree(e->canon_scratch);
        e->canon_scratch = nullptr; e->canon_scratch_bytes = 0;
        HSC_CUDA(e, cudaMalloc(&e->canon_scratch, need));
        e->canon_scratch_bytes = need;
    }
    long long* gkey = (long long*)e->canon_scratch;
    int* gev = (int*)(e->canon_scratch + off_ev);
    long long* counts = (long long*)(e->canon_scratch + off_counts);
    events::canonical_codes_kernel<real, false><<<(unsigned)S, events::CANON_THREADS, 0, st>>>(
        (const long long*)offsets, pos, idx, (const real*)coef, capacity, (int)S, K, lb, min_coef, gkey, gev, counts, nullptr, nullptr,
        nullptr, nullptr);
    events::level_offsets_kernel<<<(unsigned)L, 1024, 0, st>>>(counts, (int)S, (long long*)out_offsets);
    events::canonical_codes_kernel<real, true><<<(unsigned)S, events::CANON_THREADS, 0, st>>>(
        (const long long*)offsets, pos, idx, (const real*)coef, capacity, (int)S, K, lb, min_coef, gkey, gev, counts,
        (const long long*)out_offsets, out_pos, out_idx, out_coef);
    e->launches += 3;
    HSC_CUDA(e, cudaGetLastError());
    return HSC_OK;
}

// Scratch that does not depend on the dictionary (split-signal staging of K1, LoCOMP / K-SVD scratch): kept across
// hsc_b200_set_dictionary calls - a learning loop sets a new dictionary every iteration - and released with the engine.
void free_scratch(hsc_engine* e) {
    if (e->ksvd_graph) cudaGraphExecDestroy(e->ksvd_graph);
    e->ksvd_graph = nullptr; e->ksvd_graph_scratch = nullptr; e->ksvd_graph_cap = 0;
    if (e->ksvd_scratch) cudaFree(e->ksvd_scratch);
    e->ksvd_scratch = nullptr; e->ksvd_scratch_bytes = 0;
    if (e->locomp_scratch) cudaFree(e->locomp_scratch);
    e->locomp_scratch = nullptr; e->locomp_scratch_signals = 0;
    if (e->tc_xsplit) cudaFree(e->tc_xsplit);
    e->tc_xsplit = nullptr; e->tc_xsplit_bytes = 0;
    if (e->canon_scratch) cudaFree(e->canon_scratch);
    e->canon_scratch = nullptr; e->canon_scratch_bytes = 0;
}

void free_dictionary(hsc_engine* e) {
    if (!e->owns_dict) {
        e->D_dev = e->G_dev = e->w_dev = nullptr;
        e->tc_bop = nullptr;
        e->tc_plan = tc::Plan{};
        return;
    }
    if (e->D_dev) cudaFree(e->D_dev);
    if (e->G_dev) cudaFree(e->G_dev);
    if (e->w_dev) cudaFree(e->w_dev);
    if (e->tc_bop) cudaFree(e->tc_bop);
    e->D_dev = e->G_dev = e->w_dev = nullptr;
    e->gram_valid = false;
    e->tc_bop = nullptr;
    e->tc_plan = tc::Plan{};
}

}  // namespace

extern "C" {

int hsc_b200_abi_version(void) { return HSC_B200_ABI_VERSION; }

int hsc_b200_create(int device, hsc_engine** out) {
    if (!out) return HSC_E_INVALID;
    *out = nullptr;
    int n = 0;
    cudaError_t err = cudaGetDeviceCount(&n);
    if (err != cudaSuccess || n <= 0 || device < 0 || device >= n) return HSC_E_CUDA;   // no CPU fallback
    if (cudaSetDevice(device) != cudaSuccess) return HSC_E_CUDA;
    hsc_engine* e = new hsc_engine();
    e->device = device;
    *out = e;
    return HSC_OK;
}

int hsc_b200_create_view(hsc_engine* parent, hsc_engine** out) {
    if (!parent || !out) return HSC_E_INVALID;
    if (!parent->D_dev) return fail(parent, HSC_E_STATE, "create_view: no dictionary set");
    { cudaSetDevice(parent->device); int rcg = ensure_gram(parent); if (rcg != HSC_OK) return rcg; }
    hsc_engine* e = new hsc_engine();
    e->device = parent->device;
    e->dtype = parent->dtype; e->K = parent->K; e->L = parent->L; e->F = parent->F;
    e->D_dev = parent->D_dev; e->G_dev = parent->G_dev; e->w_dev = parent->w_dev;
    e->tc_plan = parent->tc_plan; e->tc_bop = parent->tc_bop;
    e->owns_dict = false;
    *out = e;
    return HSC_OK;
}

int hsc_b200_destroy(hsc_engine* e) {
    if (!e) return HSC_E_INVALID;
    cudaSetDevice(e->device);
    free_dictionary(e);
    free_scratch(e);
    delete e;
    return HSC_OK;
}

const char* hsc_b200_last_error(const hsc_engine* e) { return e ? e->err.c_str() : "null engine"; }

int64_t hsc_b200_launch_count(const hsc_engine* e) { return e ? e->launches : 0; }

int hsc_b200_set_dictionary(hsc_engine* e, const void* D_host, int dtype, int64_t K, int64_t L, int64_t F,
                            const void* weights_host) {
    if (!e) return HSC_E_INVALID;
    if (!D_host || K <= 0 || L <= 0 || F <= 0) return fail(e, HSC_E_INVALID, "set_dictionary: D must be [K,L,F] with K,L,F > 0");
    if (dtype != HSC_F32 && dtype != HSC_F64) return fail(e, HSC_E_INVALID, "set_dictionary: dtype must be HSC_F32 or HSC_F64");
    if (K > (1 << 24) || L > (1 << 20) || F > (1 << 20)) return fail(e, HSC_E_INVALID, "set_dictionary: dimension too large");
    if (!e->owns_dict) return fail(e, HSC_E_STATE, "set_dictionary: this handle is a view; set the dictionary on its parent");
    HSC_CUDA(e, cudaSetDevice(e->device));
    // same shape, same dtype, weights present or absent as before: the device buffers (dictionary, Gram tensor, K1 operand)
    // are overwritten in place; anything else starts from scratch
    const bool same_shape = e->D_dev && e->dtype == dtype && e->K == K && e->L == L && e->F == F &&
                            ((weights_host != nullptr) == (e->w_dev != nullptr));
    if (same_shape) HSC_CUDA(e, cudaDeviceSynchronize());        // (no launch of this device may still read the old dictionary)
    else free_dictionary(e);
    e->active = false;
    e->dtype = dtype; e->K = K; e->L = L; e->F = F;
    return dtype == HSC_F32 ? set_dictionary_t<float>(e, D_host, weights_host) : set_dictionary_t<double>(e, D_host, weights_host);
}

const void* hsc_b200_dictionary_dev(const hsc_engine* e) { return e ? e->D_dev : nullptr; }
const void* hsc_b200_gram_dev(const hsc_engine* e) {
    if (!e || !e->D_dev) return nullptr;
    hsc_engine* m = const_cast<hsc_engine*>(e);
    cudaSetDevice(m->device);
    return ensure_gram(m) == HSC_OK ? m->G_dev : nullptr;
}

int hsc_b200_correlate(hsc_engine* e, const void* x_dev, int64_t S, int64_t T, void* map_dev, void* stream) {
    if (!e) return HSC_E_INVALID;
    if (!e->D_dev) return fail(e, HSC_E_STATE, "correlate: no dictionary set");
    if (!x_dev || !map_dev || S <= 0 || T <= 0 || S > 65535) return fail(e, HSC_E_INVALID, "correlate: bad arguments");
    HSC_CUDA(e, cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    return e->dtype == HSC_F32 ? correlate_t<float>(e, x_dev, S, T, map_dev, st) : correlate_t<double>(e, x_dev, S, T, map_dev, st);
}

size_t hsc_b200_workspace_bytes(const hsc_engine* e, int64_t S, int64_t T) {
    if (!e || !e->D_dev || S <= 0 || T <= 0) return 0;
    return make_layout(S, T, e->K, e->L, e->dtype == HSC_F32 ? 4 : 8, e->F).total;
}

int hsc_b200_mp_begin_part(hsc_engine* e, const void* x_dev, void* residual_dev, int64_t S, int64_t T, void* workspace_dev,
                           size_t workspace_bytes, const hsc_mp_options* opt, int64_t s_lo, int64_t s_count, void* stream) {
    if (!e) return HSC_E_INVALID;
    if (!e->D_dev) return fail(e, HSC_E_STATE, "mp_begin: no dictionary set");
    if (!x_dev || !residual_dev || !workspace_dev || !opt || S <= 0 || T <= 0 || S > 65535 || s_lo < 0 || s_count <= 0 ||
        s_lo + s_count > S)
        return fail(e, HSC_E_INVALID, "mp_begin: bad arguments");
    if (T * e->K >= (1ll << 40) || T >= (1ll << 31)) return fail(e, HSC_E_INVALID, "mp_begin: T too large for one signal; segment it");
    HSC_CUDA(e, cudaSetDevice(e->device));
    const size_t rsz = e->dtype == HSC_F32 ? 4 : 8;
    Layout l = make_layout(S, T, e->K, e->L, rsz, e->F);
    if (workspace_bytes < l.total) return fail(e, HSC_E_NOMEM, "mp_begin: workspace smaller than hsc_b200_workspace_bytes()");
    if (opt->method != 0 && opt->method != 1) return fail(e, HSC_E_INVALID, "mp_begin: method must be 0 (MP) or 1 (LoCOMP)");
    if (opt->nb_blocks != 1) {
        if (opt->nb_blocks == 0 || opt->nb_blocks < -1) return fail(e, HSC_E_INVALID, "mp_begin: nbBlocks must be 1, > 1 or -1 ('auto')");
        long long bs = opt->nb_blocks < 0 ? 4 * e->L : T / opt->nb_blocks;
        if (bs & 1) bs += 1;
        if (bs < 2) return fail(e, HSC_E_INVALID, "mp_begin: nbBlocks larger than T/2");
        if ((T + bs - 1) / bs + 1 > l.ncand_max) return fail(e, HSC_E_UNSUPPORTED, "mp_begin: too many selection blocks for the candidate lists");
    }
    cudaStream_t st = (cudaStream_t)stream;
    { int rcg = ensure_gram(e); if (rcg != HSC_OK) return rcg; }
    e->S = S; e->T = T; e->lay = l; e->ws = (unsigned char*)workspace_dev; e->resid = residual_dev; e->opt = *opt;
    // everything below touches only signals [s_lo, s_lo + s_count) of the S-signal arrays
    const size_t sig_x = (size_t)T * e->F * rsz, sig_map = (size_t)T * e->K * rsz;
    const unsigned char* xp = (const unsigned char*)x_dev + (size_t)s_lo * sig_x;
    unsigned char* rp = (unsigned char*)residual_dev + (size_t)s_lo * sig_x;
    unsigned char* mapp = e->ws + l.off_map + (size_t)s_lo * sig_map;
    unsigned char* v1p = e->ws + l.off_val1 + (size_t)s_lo * T * rsz;
    int* i1p = (int*)(e->ws + l.off_idx1) + (size_t)s_lo * T;
    const int64_t Sc = s_count;
    if ((const void*)xp != (const void*)rp)
        HSC_CUDA(e, cudaMemcpyAsync(rp, xp, (size_t)Sc * sig_x, cudaMemcpyDeviceToDevice, st));
    // Level-1 keys: fused into the tensor-core K1 epilogue when every 32-column chunk of the product lies in
    // one time row and the scores are unweighted; otherwise a grid-wide pass over the map builds them.
    static const bool force_simt = getenv("HSC_K1") && !strcmp(getenv("HSC_K1"), "simt");
    static const bool no_fuse = getenv("HSC_K1_KEYS") && !strcmp(getenv("HSC_K1_KEYS"), "separate");
    const bool tc_path = e->dtype == HSC_F32 && e->tc_plan.ok && !force_simt && T * e->K < (1ll << 31);
    const bool fused_keys = tc_path && !no_fuse && !(opt->use_weights && e->w_dev) && (e->tc_plan.s == 1 || e->K % 32 == 0);
    int rc;
    if (fused_keys) {
        unsigned long long* keys = (unsigned long long*)(e->ws + l.off_keys) + (size_t)s_lo * T;
        HSC_CUDA(e, cudaMemsetAsync(keys, 0, (size_t)Sc * T * sizeof(unsigned long long), st));
        rc = correlate_tc(e, xp, Sc, T, mapp, st, keys);
        if (rc != HSC_OK) return rc;
        const long long n = (long long)Sc * T;
        unsigned blocks = (unsigned)((n + 255) / 256);
        if (blocks > 148 * 16) blocks = 148 * 16;
        tc::unpack_keys_kernel<<<blocks, 256, 0, st>>>(keys, (float*)v1p, i1p, n);
        e->launches++;
        HSC_CUDA(e, cudaGetLastError());
    } else {
        rc = e->dtype == HSC_F32 ? correlate_t<float>(e, xp, Sc, T, mapp, st) : correlate_t<double>(e, xp, Sc, T, mapp, st);
        if (rc != HSC_OK) return rc;
        const int rows_per_cta = 64;
        dim3 grid((unsigned)((T + rows_per_cta - 1) / rows_per_cta), (unsigned)Sc);
        const void* wts = (opt->use_weights && e->w_dev) ? e->w_dev : nullptr;
        if (e->dtype == HSC_F32)
            rowkey_kernel<float><<<grid, 256, 0, st>>>((const float*)mapp, (const float*)wts, (float*)v1p, i1p, (int)T, (int)e->K, rows_per_cta);
        else
            rowkey_kernel<double><<<grid, 256, 0, st>>>((const double*)mapp, (const double*)wts, (double*)v1p, i1p, (int)T, (int)e->K, rows_per_cta);
        e->launches++;
        HSC_CUDA(e, cudaGetLastError());
    }
    HSC_CUDA(e, cudaMemsetAsync(e->ws + l.off_bitmap + (size_t)s_lo * l.bitmap_words * sizeof(unsigned), 0,
                                (size_t)Sc * l.bitmap_words * sizeof(unsigned), st));
    HSC_CUDA(e, cudaMemsetAsync(e->ws + l.off_state + (size_t)s_lo * sizeof(hsc_signal_state), 0, (size_t)Sc * sizeof(hsc_signal_state), st));
    e->active = true;
    return HSC_OK;
}

int hsc_b200_mp_begin(hsc_engine* e, const void* x_dev, void* residual_dev, int64_t S, int64_t T, void* workspace_dev,
                      size_t workspace_bytes, const hsc_mp_options* opt, void* stream) {
    return hsc_b200_mp_begin_part(e, x_dev, residual_dev, S, T, workspace_dev, workspace_bytes, opt, 0, S, stream);
}

int hsc_b200_mp_states(hsc_engine* e, hsc_signal_state* states_host, void* stream) {
    if (!e || !states_host) return HSC_E_INVALID;
    if (!e->active) return fail(e, HSC_E_STATE, "mp_states: no encode in flight");
    HSC_CUDA(e, cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    HSC_CUDA(e, cudaMemcpyAsync(states_host, e->ws + e->lay.off_state, (size_t)e->S * sizeof(hsc_signal_state),
                                cudaMemcpyDeviceToHost, st));
    HSC_CUDA(e, cudaStreamSynchronize(st));
    return HSC_OK;
}

int hsc_b200_mp_states_async(hsc_engine* e, hsc_signal_state* states_host, void* stream) {
    if (!e || !states_host) return HSC_E_INVALID;
    if (!e->active) return fail(e, HSC_E_STATE, "mp_states_async: no encode in flight");
    HSC_CUDA(e, cudaSetDevice(e->device));
    HSC_CUDA(e, cudaMemcpyAsync(states_host, e->ws + e->lay.off_state, (size_t)e->S * sizeof(hsc_signal_state),
                                cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    return HSC_OK;
}

int hsc_b200_mp_run(hsc_engine* e, int32_t* ev_pos_dev, int32_t* ev_idx_dev, void* ev_coef_dev, int64_t capacity,
                    hsc_signal_state* states_host, void* stream) {
    if (!e) return HSC_E_INVALID;
    if (!e->active) return fail(e, HSC_E_STATE, "mp_run: call hsc_b200_mp_begin first");
    if (!ev_pos_dev || !ev_idx_dev || !ev_coef_dev || capacity <= 0) return fail(e, HSC_E_INVALID, "mp_run: bad arguments");
    HSC_CUDA(e, cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    int rc = e->dtype == HSC_F32 ? run_t<float>(e, ev_pos_dev, ev_idx_dev, ev_coef_dev, capacity, st)
                                 : run_t<double>(e, ev_pos_dev, ev_idx_dev, ev_coef_dev, capacity, st);
    if (rc != HSC_OK) return rc;
    if (states_host) return hsc_b200_mp_states(e, states_host, stream);
    return HSC_OK;
}

int hsc_b200_mp_compact_events(hsc_engine* e, const int32_t* ev_pos_dev, const int32_t* ev_idx_dev, const void* ev_coef_dev,
                               int64_t capacity, int64_t* offsets_dev, int32_t* pos_out_dev, int32_t* idx_out_dev, void* coef_out_dev,
                               int64_t out_capacity, void* stream) {
    if (!e) return HSC_E_INVALID;
    if (!e->active) return fail(e, HSC_E_STATE, "mp_compact_events: no encode in flight");
    if (!ev_pos_dev || !ev_idx_dev || !ev_coef_dev || !offsets_dev || !pos_out_dev || !idx_out_dev || !coef_out_dev || capacity <= 0 ||
        out_capacity < 0)
        return fail(e, HSC_E_INVALID, "mp_compact_events: bad arguments");
    HSC_CUDA(e, cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    const hsc_signal_state* states = (const hsc_signal_state*)(e->ws + e->lay.off_state);
    events::offsets_kernel<<<1, 1024, 0, st>>>(states, (int)e->S, (long long*)offsets_dev);
    if (e->dtype == HSC_F32)
        events::compact_kernel<float><<<(unsigned)e->S, 256, 0, st>>>(ev_pos_dev, ev_idx_dev, (const float*)ev_coef_dev, capacity,
                                                                     (const long long*)offsets_dev, pos_out_dev, idx_out_dev,
                                                                     (float*)coef_out_dev, out_capacity);
    else
        events::compact_kernel<double><<<(unsigned)e->S, 256, 0, st>>>(ev_pos_dev, ev_idx_dev, (const double*)ev_coef_dev, capacity,
                                                                      (const long long*)offsets_dev, pos_out_dev, idx_out_dev,
                                                                      (double*)coef_out_dev, out_capacity);
    e->launches += 2;
    HSC_CUDA(e, cudaGetLastError());
    return HSC_OK;
}

int hsc_b200_mp_events_to_dense(hsc_engine* e, const int32_t* ev_pos_dev, const int32_t* ev_idx_dev, const void* ev_coef_dev,
                                int64_t capacity, double min_coefficients, double* dense_dev, void* stream) {
    if (!e) return HSC_E_INVALID;
    if (!e->active) return fail(e, HSC_E_STATE, "mp_events_to_dense: no encode in flight");
    if (!ev_pos_dev || !ev_idx_dev || !ev_coef_dev || !dense_dev || capacity <= 0) return fail(e, HSC_E_INVALID, "mp_events_to_dense: bad arguments");
    HSC_CUDA(e, cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    const hsc_signal_state* states = (const hsc_signal_state*)(e->ws + e->lay.off_state);
    HSC_CUDA(e, cudaMemsetAsync(dense_dev, 0, (size_t)e->S * e->T * e->K * sizeof(double), st));
    if (e->dtype == HSC_F32)
        events::events_to_dense_kernel<float><<<(unsigned)e->S, 256, 0, st>>>(states, ev_pos_dev, ev_idx_dev, (const float*)ev_coef_dev, capacity,
                                                                             (int)e->T, (int)e->K, min_coefficients, dense_dev);
    else
        events::events_to_dense_kernel<double><<<(unsigned)e->S, 256, 0, st>>>(states, ev_pos_dev, ev_idx_dev, (const double*)ev_coef_dev, capacity,
                                                                              (int)e->T, (int)e->K, min_coefficients, dense_dev);
    e->launches++;
    HSC_CUDA(e, cudaGetLastError());
    return HSC_OK;
}

const void* hsc_b200_mp_map_dev(const hsc_engine* e) { return (e && e->active) ? e->ws + e->lay.off_map : nullptr; }

int hsc_b200_decode(hsc_engine* e, const int32_t* pos_dev, const int32_t* idx_dev, const void* coef_dev, int64_t n, int64_t T,
                    void* out_dev, void* stream) {
    if (!e) return HSC_E_INVALID;
    if (!e->D_dev) return fail(e, HSC_E_STATE, "decode: no dictionary set");
    if (!out_dev || T <= 0 || n < 0 || (n > 0 && (!pos_dev || !idx_dev || !coef_dev))) return fail(e, HSC_E_INVALID, "decode: bad arguments");
    if (n == 0) return HSC_OK;
    HSC_CUDA(e, cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    return e->dtype == HSC_F32 ? decode_t<float>(e, nullptr, pos_dev, idx_dev, coef_dev, n, 1, T, out_dev, st)
                               : decode_t<double>(e, nullptr, pos_dev, idx_dev, coef_dev, n, 1, T, out_dev, st);
}

int hsc_b200_decode_batch(hsc_engine* e, const int64_t* offsets_dev, const int32_t* pos_dev, const int32_t* idx_dev,
                          const void* coef_dev, int64_t S, int64_t T, void* out_dev, void* stream) {
    if (!e) return HSC_E_INVALID;
    if (!e->D_dev) return fail(e, HSC_E_STATE, "decode_batch: no dictionary set");
    if (!out_dev || !offsets_dev || S <= 0 || T <= 0 || T >= (1ll << 31) || !pos_dev || !idx_dev || !coef_dev)
        return fail(e, HSC_E_INVALID, "decode_batch: bad arguments");
    HSC_CUDA(e, cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    return e->dtype == HSC_F32 ? decode_t<float>(e, offsets_dev, pos_dev, idx_dev, coef_dev, 0, S, T, out_dev, st)
                               : decode_t<double>(e, offsets_dev, pos_dev, idx_dev, coef_dev, 0, S, T, out_dev, st);
}

int hsc_b200_canonicalize_codes(hsc_engine* e, const int64_t* offsets_dev, const int32_t* pos_dev, const int32_t* idx_dev,
                                const void* coef_dev, int64_t capacity, int64_t S, int64_t T, int64_t K,
                                const int64_t* level_bounds_host, int64_t n_bounds, double min_coefficients, int64_t* out_offsets_dev,
                                int32_t* out_pos_dev, int32_t* out_idx_dev, double* out_coef_dev, void* stream) {
    if (!e) return HSC_E_INVALID;
    if (!e->D_dev) return fail(e, HSC_E_STATE, "canonicalize_codes: no dictionary set (it fixes the coefficient dtype)");
    if (!offsets_dev || !out_offsets_dev || S <= 0 || S > 65535 || T <= 0 || T >= (1ll << 31) || K <= 0 || K >= (1ll << 31) ||
        capacity < 0 || n_bounds < 0 || n_bounds >= events::CANON_MAX_LEVELS || (n_bounds > 0 && !level_bounds_host) ||
        (capacity > 0 && (!pos_dev || !idx_dev || !coef_dev || !out_pos_dev || !out_idx_dev || !out_coef_dev)))
        return fail(e, HSC_E_INVALID, "canonicalize_codes: bad arguments");
    events::LevelBounds lb{};
    lb.n = (int)n_bounds;
    for (int64_t j = 0; j < n_bounds; ++j) {
        if (level_bounds_host[j] < 0 || (j > 0 && level_bounds_host[j] < level_bounds_host[j - 1]))
            return fail(e, HSC_E_INVALID, "canonicalize_codes: level bounds must be non-negative and non-decreasing");
        lb.b[j] = level_bounds_host[j];
    }
    HSC_CUDA(e, cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    return e->dtype == HSC_F32 ? canonicalize_t<float>(e, offsets_dev, pos_dev, idx_dev, coef_dev, capacity, S, K, lb, min_coefficients,
                                                       out_offsets_dev, out_pos_dev, out_idx_dev, out_coef_dev, st)
                               : canonicalize_t<double>(e, offsets_dev, pos_dev, idx_dev, coef_dev, capacity, S, K, lb, min_coefficients,
                                                        out_offsets_dev, out_pos_dev, out_idx_dev, out_coef_dev, st);
}

int hsc_b200_copy_to_host(hsc_engine* e, const void* src_dev, void* dst_host, size_t bytes) {
    if (!e || !src_dev || !dst_host) return HSC_E_INVALID;
    HSC_CUDA(e, cudaSetDevice(e->device));
    HSC_CUDA(e, cudaDeviceSynchronize());
    HSC_CUDA(e, cudaMemcpy(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost));
    return HSC_OK;
}

int hsc_b200_mp_encode_host(hsc_engine* e, const void* x_host, int64_t S, int64_t T, const hsc_mp_options* opt,
                            int32_t* ev_pos_host, int32_t* ev_idx_host, void* ev_coef_host, int64_t capacity,
                            int64_t* counts_host, void* residual_host, hsc_signal_state* states_host) {
    if (!e) return HSC_E_INVALID;
    if (!e->D_dev) return fail(e, HSC_E_STATE, "mp_encode_host: no dictionary set");
    if (!x_host || !opt || !ev_pos_host || !ev_idx_host || !ev_coef_host || S <= 0 || T <= 0 || capacity <= 0)
        return fail(e, HSC_E_INVALID, "mp_encode_host: bad arguments");
    HSC_CUDA(e, cudaSetDevice(e->device));
    const size_t rsz = e->dtype == HSC_F32 ? 4 : 8;
    const size_t nx = (size_t)S * T * e->F * rsz;
    const size_t wsb = hsc_b200_workspace_bytes(e, S, T);
    void *x = nullptr, *ws = nullptr, *evc = nullptr;
    int32_t *evp = nullptr, *evi = nullptr;
    std::vector<hsc_signal_state> states((size_t)S);
    int rc = HSC_OK;
    cudaError_t ce;
#define HSC_TRYC(call)                                                                   \
    if (rc == HSC_OK && (ce = (call)) != cudaSuccess)                                    \
        rc = fail(e, HSC_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(ce));
    HSC_TRYC(cudaMalloc(&x, nx));
    HSC_TRYC(cudaMalloc(&ws, wsb));
    HSC_TRYC(cudaMalloc((void**)&evp, (size_t)S * capacity * sizeof(int32_t)));
    HSC_TRYC(cudaMalloc((void**)&evi, (size_t)S * capacity * sizeof(int32_t)));
    HSC_TRYC(cudaMalloc(&evc, (size_t)S * capacity * rsz));
    HSC_TRYC(cudaMemcpy(x, x_host, nx, cudaMemcpyHostToDevice));
    if (rc == HSC_OK) rc = hsc_b200_mp_begin(e, x, x, S, T, ws, wsb, opt, nullptr);
    if (rc == HSC_OK) rc = hsc_b200_mp_run(e, evp, evi, evc, capacity, states.data(), nullptr);
    if (rc == HSC_OK) {
        for (int64_t s = 0; s < S; ++s)
            if (states[(size_t)s].status == HSC_PAUSE_CAPACITY) {
                rc = fail(e, HSC_E_NOMEM, "mp_encode_host: event capacity exhausted before the stop rule fired");
                break;
            }
    }
    HSC_TRYC(cudaMemcpy(ev_pos_host, evp, (size_t)S * capacity * sizeof(int32_t), cudaMemcpyDeviceToHost));
    HSC_TRYC(cudaMemcpy(ev_idx_host, evi, (size_t)S * capacity * sizeof(int32_t), cudaMemcpyDeviceToHost));
    HSC_TRYC(cudaMemcpy(ev_coef_host, evc, (size_t)S * capacity * rsz, cudaMemcpyDeviceToHost));
    if (residual_host) HSC_TRYC(cudaMemcpy(residual_host, x, nx, cudaMemcpyDeviceToHost));
#undef HSC_TRYC
    if (rc == HSC_OK || rc == HSC_E_NOMEM) {
        if (counts_host) for (int64_t s = 0; s < S; ++s) counts_host[s] = states[(size_t)s].n_buffered;
        if (states_host) memcpy(states_host, states.data(), (size_t)S * sizeof(hsc_signal_state));
    }
    e->active = false;
    if (x) cudaFree(x);
    if (ws) cudaFree(ws);
    if (evp) cudaFree(evp);
    if (evi) cudaFree(evi);
    if (evc) cudaFree(evc);
    return rc;
}

// One dictionary-update sweep (hsc_b200_ksvd_begin .. _end): scratch + the per-filter state machine.
struct hsc_ksvd_sweep {
    hsc_engine* e = nullptr;
    cudaStream_t st = nullptr;
    long long K = 0, L = 0, F = 0, S = 0, T = 0, q = 0;
    int off = 0;
    std::vector<long long> col_ptr;
    const int32_t* sig = nullptr; const int32_t* pos = nullptr; const int32_t* idx = nullptr;
    double* coef = nullptr; double* D = nullptr;
    long long* col_ptr_dev = nullptr;
    double *R = nullptr, *W = nullptr, *C = nullptr, *M0 = nullptr, *M1 = nullptr, *u = nullptr, *oldD = nullptr, *acc = nullptr;
    bool owns_C = true;
    long long open_filter = -1;          // filter whose atoms are currently out of the running reconstruction
};

namespace {

constexpr unsigned kKsvdGrid = 148 * 2;  // fixed grid of the grid-stride kernels of a sweep (graph-capturable)

size_t ksvd_al(size_t v) { return (v + 255) / 256 * 256; }

// Carves the sweep's buffers out of the engine's persistent scratch: R, W (n_rows window rows), C, M0, M1, u, oldD, acc,
// col_ptr, and (stable = the graph path) engine-owned copies of the dictionary and of the code arrays.
struct KsvdCarve {
    double *R, *W, *C, *M0, *M1, *u, *oldD, *acc, *D, *coef;
    long long* col_ptr;
    int32_t *sig, *pos, *idx;
};

int ksvd_carve(hsc_engine* e, long long K, long long q, long long S, long long T, long long F, long long n_rows, long long n_code,
               KsvdCarve* c) {
    const size_t bR = ksvd_al((size_t)S * T * F * sizeof(double)), bW = ksvd_al((size_t)(n_rows > 0 ? n_rows : 1) * q * sizeof(double));
    const size_t bQ = ksvd_al((size_t)q * q * sizeof(double)), bu = ksvd_al((size_t)q * sizeof(double)), bD = ksvd_al((size_t)K * q * sizeof(double));
    const size_t bP = ksvd_al((size_t)(K + 1) * sizeof(long long));
    const size_t bI = ksvd_al((size_t)(n_code > 0 ? n_code : 1) * sizeof(int32_t)), bC = ksvd_al((size_t)(n_code > 0 ? n_code : 1) * sizeof(double));
    const size_t need = bR + bW + 3 * bQ + bu + 2 * bD + 256 + bP + 3 * bI + bC;
    if (e->ksvd_scratch_bytes < need) {
        if (e->ksvd_scratch) cudaFree(e->ksvd_scratch);
        e->ksvd_scratch = nullptr; e->ksvd_scratch_bytes = 0;
        const size_t grow = need + need / 4;                    // head room: the code size changes from sweep to sweep
        HSC_CUDA(e, cudaMalloc((void**)&e->ksvd_scratch, grow));
        e->ksvd_scratch_bytes = grow;
    }
    unsigned char* p = e->ksvd_scratch;
    // fixed-size buffers first so that their addresses survive a change of the code size
    c->C = (double*)p; p += bQ;
    c->M0 = (double*)p; p += bQ;
    c->M1 = (double*)p; p += bQ;
    c->u = (double*)p; p += bu;
    c->oldD = (double*)p; p += bD;
    c->D = (double*)p; p += bD;
    c->acc = (double*)p; p += 256;
    c->col_ptr = (long long*)p; p += bP;
    c->R = (double*)p; p += bR;
    c->W = (double*)p; p += bW;
    c->sig = (int32_t*)p; p += bI;
    c->pos = (int32_t*)p; p += bI;
    c->idx = (int32_t*)p; p += bI;
    c->coef = (double*)p; p += bC;
    return HSC_OK;
}

// The launches of one filter's update; col_ptr is read on the device, grids are fixed (eager and graph paths alike).
// (fused_gram: the Gram tile is computed by the cluster-chained eigen-solver launch of ksvd_launch_finish instead)
bool ksvd_chain_ok(const hsc_engine* e, long long q) {
    static const int chain = getenv("HSC_KSVD_CHAIN") ? atoi(getenv("HSC_KSVD_CHAIN")) : 1;
    static const int n_square = getenv("HSC_KSVD_SQUARINGS") ? atoi(getenv("HSC_KSVD_SQUARINGS")) : 6;
    return chain && q <= ksvd::kPowerSmallQ && n_square >= 1 && !e->ksvd_chain_failed;
}

void ksvd_launch_gram(hsc_engine* e, cudaStream_t st, const KsvdCarve& c, const int32_t* sig, const int32_t* pos, const double* coef,
                      const double* D, long long k, long long q, long long T, long long L, long long F, int off, bool pca = false,
                      bool fused_gram = false) {
    const unsigned qt = (unsigned)((q + 15) / 16);
    ksvd::scatter_kernel<<<kKsvdGrid, 256, 0, st>>>(c.R, sig, pos, coef, c.col_ptr, (int)k, D, (int)T, (int)L, (int)F, off, -1.0);
    ksvd::gather_kernel<<<kKsvdGrid, 256, 0, st>>>(c.R, sig, pos, c.col_ptr, (int)k, (int)T, (int)L, (int)F, off, c.W);
    if (pca) {
        ksvd::center_kernel<<<(unsigned)((q + 31) / 32), 256, 0, st>>>(c.W, c.col_ptr, (int)k, (int)q);
        e->launches += 1;
    }
    if (!fused_gram) ksvd::gram_tile_kernel<<<dim3(qt, qt), 256, 0, st>>>(c.W, c.col_ptr, (int)k, (int)q, c.C);
    e->launches += fused_gram ? 2 : 3;
}

void ksvd_launch_finish(hsc_engine* e, cudaStream_t st, const KsvdCarve& c, const int32_t* sig, const int32_t* pos, double* coef,
                        double* D, double* C, long long k, long long q, long long T, long long L, long long F, int off,
                        bool skip_empty, bool fused_gram = false) {
    // HSC_KSVD_SQUARINGS: the squarings every filter gets; more follow, up to ksvd::kMaxSquarings, until the power is
    // numerically rank one (0: power iteration on C itself)
    static const int n_square = getenv("HSC_KSVD_SQUARINGS") ? atoi(getenv("HSC_KSVD_SQUARINGS")) : 6;
    const int n_max = n_square < 1 ? 0 : (n_square > ksvd::kMaxSquarings ? n_square : ksvd::kMaxSquarings);
    const unsigned qt = (unsigned)((q + 15) / 16);
    // small windows: every squaring and the power iteration in ONE launch of a cluster spanning the grid
    // (HSC_KSVD_CHAIN=0: the separate kernels)
    static const int chain = getenv("HSC_KSVD_CHAIN") ? atoi(getenv("HSC_KSVD_CHAIN")) : 1;
    int n_finish = 0;
    bool chained = false;
    if (chain && q <= ksvd::kPowerSmallQ && n_square >= 1 && !e->ksvd_chain_failed) {
        static bool attr_set = false;
        if (!attr_set) { cudaFuncSetAttribute(ksvd::square_chain_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1); attr_set = true; }
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(qt, qt); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = 0; cfg.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = qt; at[0].val.clusterDim.y = qt; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        const long long* skip = skip_empty ? c.col_ptr : nullptr;
        const double* Wf = fused_gram ? (const double*)c.W : (const double*)nullptr;
        const cudaError_t ce = cudaLaunchKernelEx(&cfg, ksvd::square_chain_kernel, C, (int)q, n_square, n_max, c.M0, c.M1, 100, 1e-14, 2,
                                                  D + k * q, c.u, skip, (int)k, Wf, (const long long*)c.col_ptr);
        if (ce == cudaSuccess) { chained = true; n_finish = 1; }
        else { (void)cudaGetLastError(); e->ksvd_chain_failed = true; }       // (cluster launch refused: the separate kernels from now on)
    }
    if (!chained) {
        if (fused_gram) { ksvd::gram_tile_kernel<<<dim3(qt, qt), 256, 0, st>>>(c.W, c.col_ptr, (int)k, (int)q, C); e->launches += 1; }
        const double** m_final = (const double**)(c.acc + 1);      // the power the squarings stopped at (acc[0]: alpha^2)
        const double* M = C;
        double* bufs[2] = {c.M0, c.M1};
        for (int sq = 0; sq < n_max; ++sq) {
            ksvd::square_kernel<<<dim3(qt, qt), 256, 0, st>>>(M, (int)q, bufs[sq & 1], sq, n_square, m_final);
            M = bufs[sq & 1];
        }
        const long long* skip = skip_empty ? c.col_ptr : nullptr;
        const double* const* mf = n_max > 0 ? m_final : nullptr;
        if (q <= ksvd::kPowerSmallQ) {
            ksvd::power_small_kernel<<<1, 256, 0, st>>>(M, mf, C, (int)q, 100, 1e-14, 2, D + k * q, c.u, skip, (int)k);   // new filter (:630)
        } else {
            static bool smem_set = false;       // 16 * q bytes of dynamic shared memory pass the 48 KB default at q = 3072
            if (!smem_set) {
                cudaFuncSetAttribute(ksvd::power_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(2 * ksvd::kMaxQ * sizeof(double)));
                smem_set = true;
            }
            ksvd::power_kernel<<<1, 256, 2 * q * sizeof(double), st>>>(M, mf, C, (int)q, 100, 1e-14, 2, D + k * q, c.u, skip, (int)k);
        }
        n_finish = 1 + n_max;
    }
    // new coefficients (:633) and the atoms back into the running reconstruction (no-op without local atoms)
    ksvd::project_scatter_kernel<<<kKsvdGrid, 256, 0, st>>>(c.W, c.u, c.col_ptr, (int)k, (int)q, coef, c.R, sig, pos, (int)T, (int)L, (int)F, off);
    e->launches += 1 + n_finish;
}

}  // namespace

int hsc_b200_ksvd_begin(hsc_engine* e, void* D_dev_io, int64_t K, int64_t L, int64_t F, const int64_t* col_ptr_host,
                        const int32_t* sig_dev, const int32_t* pos_dev, const int32_t* idx_dev, void* coef_dev_io, int64_t S,
                        int64_t T, void* gram_dev, void* stream, hsc_ksvd_sweep** out) {
    if (!e || !out) return HSC_E_INVALID;
    *out = nullptr;
    if (!D_dev_io || !col_ptr_host || K <= 0 || L <= 0 || F <= 0 || S <= 0 || T <= 0)
        return fail(e, HSC_E_INVALID, "ksvd_begin: bad arguments");
    const long long q = L * F;
    if (q > ksvd::kMaxQ) return fail(e, HSC_E_UNSUPPORTED, "ksvd_begin: L*F > " + std::to_string(ksvd::kMaxQ));
    if (e->ksvd_pca) return fail(e, HSC_E_UNSUPPORTED, "ksvd_begin: the usePCA variant needs the global column means; use hsc_b200_ksvd_update");
    const long long n = col_ptr_host[K];
    long long n_max = 0;
    for (int64_t k = 0; k < K; ++k) {
        const long long nk = col_ptr_host[k + 1] - col_ptr_host[k];
        if (nk < 0) return fail(e, HSC_E_INVALID, "ksvd_begin: col_ptr must be non-decreasing");
        if (nk > n_max) n_max = nk;
    }
    if (n > 0 && (!sig_dev || !pos_dev || !idx_dev || !coef_dev_io)) return fail(e, HSC_E_INVALID, "ksvd_begin: null code arrays");
    HSC_CUDA(e, cudaSetDevice(e->device));
    KsvdCarve c{};
    int rc = ksvd_carve(e, K, q, S, T, F, n_max, 0, &c);
    if (rc != HSC_OK) return rc;
    hsc_ksvd_sweep* w = new hsc_ksvd_sweep();
    w->e = e; w->st = (cudaStream_t)stream;
    w->K = K; w->L = L; w->F = F; w->S = S; w->T = T; w->q = q; w->off = centre_offset((int)L);
    w->col_ptr.assign(col_ptr_host, col_ptr_host + K + 1);
    w->sig = sig_dev; w->pos = pos_dev; w->idx = idx_dev; w->coef = (double*)coef_dev_io; w->D = (double*)D_dev_io;
    w->owns_C = gram_dev == nullptr;
    w->C = w->owns_C ? c.C : (double*)gram_dev;
    w->R = c.R; w->W = c.W; w->M0 = c.M0; w->M1 = c.M1; w->u = c.u; w->oldD = c.oldD; w->acc = c.acc; w->col_ptr_dev = c.col_ptr;
    cudaError_t ce;
#define HSC_TRYK(call)                                                                   \
    if (rc == HSC_OK && (ce = (call)) != cudaSuccess)                                    \
        rc = fail(e, HSC_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(ce));
    HSC_TRYK(cudaMemcpyAsync(w->col_ptr_dev, w->col_ptr.data(), (size_t)(K + 1) * sizeof(long long), cudaMemcpyHostToDevice, w->st));
    HSC_TRYK(cudaMemcpyAsync(w->oldD, w->D, (size_t)K * q * sizeof(double), cudaMemcpyDeviceToDevice, w->st));
    HSC_TRYK(cudaMemsetAsync(w->R, 0, (size_t)S * T * F * sizeof(double), w->st));
    if (rc == HSC_OK) {
        // running reconstruction of the whole code; filter k's atoms are taken out / put back around its update
        ksvd::scatter_all_kernel<<<kKsvdGrid, 256, 0, w->st>>>(w->R, sig_dev, pos_dev, idx_dev, w->coef, w->col_ptr_dev, (int)K, w->D,
                                                               (int)T, (int)L, (int)F, w->off);
        e->launches++;
        HSC_TRYK(cudaGetLastError());
        HSC_TRYK(cudaStreamSynchronize(w->st));               // col_ptr was staged from the sweep object's own memory
    }
#undef HSC_TRYK
    if (rc != HSC_OK) { delete w; return rc; }
    *out = w;
    return HSC_OK;
}

int hsc_b200_ksvd_filter_gram(hsc_ksvd_sweep* w, int64_t k, int64_t* n_local) {
    if (!w) return HSC_E_INVALID;
    hsc_engine* e = w->e;
    if (k < 0 || k >= w->K || w->open_filter >= 0) return fail(e, HSC_E_STATE, "ksvd_filter_gram: bad filter or a filter is already open");
    HSC_CUDA(e, cudaSetDevice(e->device));
    if (n_local) *n_local = w->col_ptr[(size_t)k + 1] - w->col_ptr[(size_t)k];
    KsvdCarve c{};
    c.R = w->R; c.W = w->W; c.C = w->C; c.M0 = w->M0; c.M1 = w->M1; c.u = w->u; c.col_ptr = w->col_ptr_dev; c.acc = w->acc;
    ksvd_launch_gram(e, w->st, c, w->sig, w->pos, w->coef, w->D, k, w->q, w->T, w->L, w->F, w->off);
    HSC_CUDA(e, cudaGetLastError());
    w->open_filter = k;
    return HSC_OK;
}

int hsc_b200_ksvd_filter_finish(hsc_ksvd_sweep* w, int64_t k, int skip) {
    if (!w) return HSC_E_INVALID;
    hsc_engine* e = w->e;
    if (k != w->open_filter) return fail(e, HSC_E_STATE, "ksvd_filter_finish: call ksvd_filter_gram for this filter first");
    HSC_CUDA(e, cudaSetDevice(e->device));
    KsvdCarve c{};
    c.R = w->R; c.W = w->W; c.C = w->C; c.M0 = w->M0; c.M1 = w->M1; c.u = w->u; c.col_ptr = w->col_ptr_dev; c.acc = w->acc;
    if (!skip) {
        ksvd_launch_finish(e, w->st, c, w->sig, w->pos, w->coef, w->D, w->C, k, w->q, w->T, w->L, w->F, w->off, false);
    } else {
        // unchanged filter: its (local) atoms go back as they were
        ksvd::scatter_kernel<<<kKsvdGrid, 256, 0, w->st>>>(w->R, w->sig, w->pos, w->coef, w->col_ptr_dev, (int)k, w->D,
                                                          (int)w->T, (int)w->L, (int)w->F, w->off, 1.0);
        e->launches++;
    }
    HSC_CUDA(e, cudaGetLastError());
    w->open_filter = -1;
    return HSC_OK;
}

int hsc_b200_ksvd_end(hsc_ksvd_sweep* w, double* alpha_host) {
    if (!w) return HSC_E_INVALID;
    hsc_engine* e = w->e;
    int rc = HSC_OK;
    cudaSetDevice(e->device);
    ksvd::sqdist_kernel<<<1, 256, 0, w->st>>>(w->D, w->oldD, (long long)w->K * w->q, w->acc);
    e->launches++;
    double a2 = 0.0;
    cudaError_t ce = cudaGetLastError();
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(&a2, w->acc, sizeof(double), cudaMemcpyDeviceToHost, w->st);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(w->st);
    if (ce != cudaSuccess) rc = fail(e, HSC_E_CUDA, std::string("ksvd_end: ") + cudaGetErrorString(ce));
    if (alpha_host) *alpha_host = sqrt(a2);
    delete w;
    return rc;
}

// The whole sweep of one process.  The launch sequence (11 small dependent kernels per filter) does not depend on the code
// - the kernels read the filters' slices from device memory - so it is captured ONCE per (K, L, F, S, T, scratch) in a
// CUDA graph over engine-owned copies of the dictionary and of the code, and replayed for every sweep of a learning loop.
int hsc_b200_ksvd_set_pca(hsc_engine* e, int use_pca) {
    if (!e) return HSC_E_INVALID;
    const int v = use_pca ? 1 : 0;
    if (v != e->ksvd_pca) {      // the captured sweep belongs to the other variant
        if (e->ksvd_graph) { cudaGraphExecDestroy(e->ksvd_graph); e->ksvd_graph = nullptr; }
        e->ksvd_same_key_sweeps = 0;
        e->ksvd_pca = v;
    }
    return HSC_OK;
}

int hsc_b200_ksvd_update(hsc_engine* e, void* D_dev_io, int64_t K, int64_t L, int64_t F, const int64_t* col_ptr_host,
                         const int32_t* sig_dev, const int32_t* pos_dev, const int32_t* idx_dev, void* coef_dev_io, int64_t S,
                         int64_t T, double* alpha_host, void* stream) {
    if (!e) return HSC_E_INVALID;
    if (!D_dev_io || !col_ptr_host || K <= 0 || L <= 0 || F <= 0 || S <= 0 || T <= 0)
        return fail(e, HSC_E_INVALID, "ksvd_update: bad arguments");
    const long long q = L * F;
    if (q > ksvd::kMaxQ) return fail(e, HSC_E_UNSUPPORTED, "ksvd_update: L*F > " + std::to_string(ksvd::kMaxQ));
    const long long n = col_ptr_host[K];
    long long n_max = 0;
    for (int64_t k = 0; k < K; ++k) {
        const long long nk = col_ptr_host[k + 1] - col_ptr_host[k];
        if (nk < 0) return fail(e, HSC_E_INVALID, "ksvd_update: col_ptr must be non-decreasing");
        if (nk > n_max) n_max = nk;
    }
    if (n > 0 && (!sig_dev || !pos_dev || !idx_dev || !coef_dev_io)) return fail(e, HSC_E_INVALID, "ksvd_update: null code arrays");
    HSC_CUDA(e, cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    // window rows / code capacity in steps of 25 % so that a learning loop whose code size wobbles keeps its graph
    long long cap = e->ksvd_graph_cap;
    if (cap < n || e->ksvd_graph_key[0] != K || e->ksvd_graph_key[1] != L || e->ksvd_graph_key[2] != F || e->ksvd_graph_key[3] != S ||
        e->ksvd_graph_key[4] != T)
        cap = n + n / 4 + 1024;
    KsvdCarve c{};
    int rc = ksvd_carve(e, K, q, S, T, F, cap, cap, &c);
    if (rc != HSC_OK) return rc;
    const int off = centre_offset((int)L);
    // Capturing + instantiating the ~5600-node graph costs ~0.27 s and a replay saves ~10 ms per sweep (45 -> 35 ms at 512
    // filters): worth it for a learning loop (the reference's default is 100 iterations), not for a couple of sweeps, so
    // the first two sweeps of a shape run eagerly.  HSC_KSVD_GRAPH=0 / 1 forces never / always.
    static const int graph_mode = getenv("HSC_KSVD_GRAPH") ? atoi(getenv("HSC_KSVD_GRAPH")) : -1;
    const bool shape_same = e->ksvd_graph_key[0] == K && e->ksvd_graph_key[1] == L && e->ksvd_graph_key[2] == F &&
                            e->ksvd_graph_key[3] == S && e->ksvd_graph_key[4] == T;
    e->ksvd_same_key_sweeps = shape_same ? e->ksvd_same_key_sweeps + 1 : 1;
    const bool use_graph = !e->ksvd_graph_disabled && (graph_mode == 1 || (graph_mode != 0 && e->ksvd_same_key_sweeps >= 3));
    // stage the inputs into the engine-owned (address-stable) buffers
    HSC_CUDA(e, cudaMemcpyAsync(c.col_ptr, col_ptr_host, (size_t)(K + 1) * sizeof(long long), cudaMemcpyHostToDevice, st));
    HSC_CUDA(e, cudaMemcpyAsync(c.D, D_dev_io, (size_t)K * q * sizeof(double), cudaMemcpyDeviceToDevice, st));
    if (n > 0) {
        HSC_CUDA(e, cudaMemcpyAsync(c.sig, sig_dev, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
        HSC_CUDA(e, cudaMemcpyAsync(c.pos, pos_dev, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
        HSC_CUDA(e, cudaMemcpyAsync(c.idx, idx_dev, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
        HSC_CUDA(e, cudaMemcpyAsync(c.coef, coef_dev_io, (size_t)n * sizeof(double), cudaMemcpyDeviceToDevice, st));
    }
    auto enqueue = [&](cudaStream_t s2) {
        cudaMemcpyAsync(c.oldD, c.D, (size_t)K * q * sizeof(double), cudaMemcpyDeviceToDevice, s2);
        cudaMemsetAsync(c.R, 0, (size_t)S * T * F * sizeof(double), s2);
        ksvd::scatter_all_kernel<<<kKsvdGrid, 256, 0, s2>>>(c.R, c.sig, c.pos, c.idx, c.coef, c.col_ptr, (int)K, c.D, (int)T, (int)L, (int)F, off);
        e->launches++;
        for (int64_t k = 0; k < K; ++k) {
            const bool fuse = ksvd_chain_ok(e, q);       // Gram tile + squarings + power iteration in one cluster launch
            ksvd_launch_gram(e, s2, c, c.sig, c.pos, c.coef, c.D, k, q, T, L, F, off, e->ksvd_pca != 0, fuse);
            ksvd_launch_finish(e, s2, c, c.sig, c.pos, c.coef, c.D, c.C, k, q, T, L, F, off, true, fuse);
        }
        ksvd::sqdist_kernel<<<1, 256, 0, s2>>>(c.D, c.oldD, (long long)K * q, c.acc);
        e->launches++;
    };
    if (use_graph) {
        const bool same = e->ksvd_graph && e->ksvd_graph_scratch == e->ksvd_scratch && e->ksvd_graph_cap == cap && e->ksvd_graph_key[0] == K &&
                          e->ksvd_graph_key[1] == L && e->ksvd_graph_key[2] == F && e->ksvd_graph_key[3] == S && e->ksvd_graph_key[4] == T;
        if (!same) {
            if (e->ksvd_graph) { cudaGraphExecDestroy(e->ksvd_graph); e->ksvd_graph = nullptr; }
            cudaStream_t cs;
            HSC_CUDA(e, cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
            cudaGraph_t g = nullptr;
            cudaError_t ce = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
            if (ce == cudaSuccess) {
                const long long l0 = e->launches;
                enqueue(cs);
                e->ksvd_graph_launches = e->launches - l0;
                e->launches = l0;
                ce = cudaStreamEndCapture(cs, &g);
            }
            if (ce == cudaSuccess) ce = cudaGraphInstantiate(&e->ksvd_graph, g, 0);
            if (g) cudaGraphDestroy(g);
            cudaStreamDestroy(cs);
            if (ce != cudaSuccess) {
                // no graph on this setup: clear the error and run this and every later sweep eagerly
                e->ksvd_graph = nullptr;
                e->ksvd_graph_disabled = true;
                cudaGetLastError();
            } else {
                e->ksvd_graph_scratch = e->ksvd_scratch; e->ksvd_graph_cap = cap;
                e->ksvd_graph_key[0] = K; e->ksvd_graph_key[1] = L; e->ksvd_graph_key[2] = F; e->ksvd_graph_key[3] = S; e->ksvd_graph_key[4] = T;
            }
        }
        if (e->ksvd_graph) {
            HSC_CUDA(e, cudaGraphLaunch(e->ksvd_graph, st));
            e->launches += e->ksvd_graph_launches;
        } else {
            enqueue(st);
        }
    } else {
        enqueue(st);
        if (!shape_same) {
            if (e->ksvd_graph) { cudaGraphExecDestroy(e->ksvd_graph); e->ksvd_graph = nullptr; }
            e->ksvd_graph_key[0] = K; e->ksvd_graph_key[1] = L; e->ksvd_graph_key[2] = F; e->ksvd_graph_key[3] = S; e->ksvd_graph_key[4] = T;
        }
        e->ksvd_graph_cap = cap;
    }
    HSC_CUDA(e, cudaGetLastError());
    // results back into the caller's arrays
    HSC_CUDA(e, cudaMemcpyAsync(D_dev_io, c.D, (size_t)K * q * sizeof(double), cudaMemcpyDeviceToDevice, st));
    if (n > 0) HSC_CUDA(e, cudaMemcpyAsync(coef_dev_io, c.coef, (size_t)n * sizeof(double), cudaMemcpyDeviceToDevice, st));
    double a2 = 0.0;
    HSC_CUDA(e, cudaMemcpyAsync(&a2, c.acc, sizeof(double), cudaMemcpyDeviceToHost, st));
    HSC_CUDA(e, cudaStreamSynchronize(st));
    if (alpha_host) *alpha_host = sqrt(a2);
    return HSC_OK;
}

int hsc_b200_kmeans_assign(hsc_engine* e, const void* x_dev, int64_t B, int64_t Tw, void* map_scratch_dev, int32_t* pos_dev,
                           int32_t* idx_dev, double* sums_dev, int32_t* counts_dev, void* stream) {
    if (!e) return HSC_E_INVALID;
    if (!e->D_dev) return fail(e, HSC_E_STATE, "kmeans_assign: no dictionary (centroids) set");
    if (!x_dev || !map_scratch_dev || !pos_dev || !idx_dev || !sums_dev || !counts_dev || B <= 0 || Tw < e->L)
        return fail(e, HSC_E_INVALID, "kmeans_assign: bad arguments (windows must be at least one filter long)");
    HSC_CUDA(e, cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int off = centre_offset((int)e->L);
    const int row_lo = off, row_hi = off + (int)(Tw - e->L);              // rows of the 'same' map = 'valid' positions
    const long long LF = e->L * e->F;
    HSC_CUDA(e, cudaMemsetAsync(sums_dev, 0, (size_t)e->K * LF * sizeof(double), st));
    HSC_CUDA(e, cudaMemsetAsync(counts_dev, 0, (size_t)e->K * sizeof(int32_t), st));
    unsigned ablocks = (unsigned)((B * 32 + 255) / 256);
    if (ablocks > 148 * 8) ablocks = 148 * 8;
    for (int64_t b0 = 0; b0 < B; b0 += 65535) {                          // hsc_b200_correlate takes <= 65535 signals per call
        const int64_t nb = B - b0 < 65535 ? B - b0 : 65535;
        const size_t rsz = e->dtype == HSC_F32 ? 4 : 8;
        const unsigned char* xp = (const unsigned char*)x_dev + (size_t)b0 * Tw * e->F * rsz;
        unsigned char* mp = (unsigned char*)map_scratch_dev + (size_t)b0 * Tw * e->K * rsz;
        int rc = hsc_b200_correlate(e, xp, nb, Tw, mp, stream);
        if (rc != HSC_OK) return rc;
        if (e->dtype == HSC_F32)
            kmeans::assign_kernel<float><<<(unsigned)nb, 256, 0, st>>>((const float*)mp, (int)Tw, (int)e->K, row_lo, row_hi, pos_dev + b0, idx_dev + b0);
        else
            kmeans::assign_kernel<double><<<(unsigned)nb, 256, 0, st>>>((const double*)mp, (int)Tw, (int)e->K, row_lo, row_hi, pos_dev + b0, idx_dev + b0);
        e->launches++;
    }
    if (e->dtype == HSC_F32)
        kmeans::accumulate_kernel<float><<<ablocks, 256, 0, st>>>((const float*)x_dev, B, (int)Tw, (int)LF, (int)e->F, pos_dev, idx_dev, sums_dev, counts_dev);
    else
        kmeans::accumulate_kernel<double><<<ablocks, 256, 0, st>>>((const double*)x_dev, B, (int)Tw, (int)LF, (int)e->F, pos_dev, idx_dev, sums_dev, counts_dev);
    e->launches++;
    HSC_CUDA(e, cudaGetLastError());
    return HSC_OK;
}

}  // extern "C"
