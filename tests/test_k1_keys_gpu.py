"""K1 (the initial correlation map), its level-1 argmax keys and the float32 Gram tensor against float64.

Matching-pursuit parity hides map error (coefficients re-evaluated from the residual, near-ties re-scored in float64), so
these tests compare the kernels that feed the pursuit with their float64 definitions directly, entry by entry:

  * the map of every K1 path - 3xFP16 tensor cores at s = 1/2/4/8 time steps per super-row and N-slices of 32-128
    columns, the 3xTF32 fall-back, the SIMT kernel in float32 and float64 - at the shapes, lengths and amplitudes where
    those paths switch, within a per-entry error bound (`_bound`);
  * that K1 writes nothing past the map;
  * the level-1 keys (val1, idx1) bit for bit against the engine's own map, on every key path;
  * the float32 Gram tensor within one ulp (plus the float64 accumulation error) of float64;
  * one matching pursuit whose map has more than 2^31 entries.

Which K1 path ran: one correlate call launches 3 kernels on the tensor cores (absmax, split, MMA) and 1 on the SIMT
kernel, as the engine's launch counter shows; `_plan` restates the host plan (make_plan in csrc/correlate_tc.cuh), which
decides between the 3xFP16 and the 3xTF32 operands and shows that the shape list reaches each path.
"""
import ctypes

import numpy as np
import pytest


# ------------------------------------------------------------------ float64 reference and the per-entry bound

def centre_offset(L):
    """Centre tap (include/hsc_b200.h): L/2-1 for even L, L/2 for odd L."""
    return L // 2 - 1 if L % 2 == 0 else L // 2


def corr64(x, D):
    """'same' correlation in float64 and the sum of absolute products, for x[S,T,F] and D[K,L,F]:
    c[s,t,k] = sum_{j,f} xz[s, t-off+j, f] * D[k,j,f] (zero outside [0, T)), a[s,t,k] = the same sum of |x * D|."""
    x = np.asarray(x, np.float64)
    D = np.asarray(D, np.float64)
    S, T, F = x.shape
    K, L, _ = D.shape
    off = centre_offset(L)
    Dm = D.reshape(K, L * F).T
    Da = np.abs(Dm)
    c = np.empty((S, T, K))
    a = np.empty((S, T, K))
    for s in range(S):
        p = np.zeros((T + L - 1, F))
        p[off:off + T] = x[s]
        w = np.lib.stride_tricks.sliding_window_view(p, L, axis=0)[:T]      # [T, F, L]
        w = np.ascontiguousarray(w.transpose(0, 2, 1)).reshape(T, L * F)
        c[s] = w @ Dm
        a[s] = np.abs(w) @ Da
    return c, a


def _bound(x, D, a, dtype):
    """Per-entry error bound of K1:  |c - c64| <= eps * sum_q |x_q D_kq| + n * (2^-33 * max|x_s| * max|D| + tiny)
    with n = L*F.  float32: eps = (n + 8) * 2^-23 for the tensor-core and SIMT kernels alike; the 2^-33 term covers the
    fp16 subnormal floor of the split operands (their scale is set by the largest element of the signal and of the whole
    dictionary), tiny = 2^-149 the rounding of subnormal results.  float64: eps = (n + 8) * 2^-52, no 2^-33 term."""
    K, L, F = D.shape
    n = L * F
    if dtype == np.float32:
        eps = (n + 8) * 2.0 ** -23
        mx = np.abs(np.asarray(x, np.float64)).reshape(x.shape[0], -1).max(axis=1)
        absolute = n * (2.0 ** -33 * mx * float(np.abs(D).max()) + 2.0 ** -149)
    else:
        eps = (n + 8) * 2.0 ** -52
        absolute = np.full(x.shape[0], n * 2.0 ** -1074)
    return eps, eps * a + absolute[:, None, None]


def check_map(c, x, D, dtype, ref=None):
    """Asserts every entry of the engine map c[S,T,K] within the bound of its float64 value; returns the largest
    error / bound ratio.  An entry whose window holds no non-zero product must be exactly zero."""
    c64, a = corr64(x, D) if ref is None else ref
    eps, tol = _bound(x, D, a, dtype)
    if dtype == np.float32:
        assert eps < 2.0 ** -13, 'bound too loose to see a lost split product: eps = %.3g' % eps
    c = np.asarray(c, np.float64)
    assert c.shape == c64.shape
    assert np.all(np.isfinite(c)), 'non-finite map entries in signals %s' % sorted(set(np.nonzero(~np.isfinite(c))[0]))
    err = np.abs(c - c64)
    ratio = err / tol
    worst = np.unravel_index(np.argmax(ratio), ratio.shape)
    assert ratio[worst] <= 1.0, 'map entry %s: %r vs float64 %r, error %.3e > bound %.3e' % (
        worst, c[worst], c64[worst], err[worst], tol[worst])
    assert np.all(c[a == 0] == 0), 'non-zero map entries where every product is zero'
    return float(ratio.max())


# ------------------------------------------------------------------ host restatement of make_plan (csrc/correlate_tc.cuh)

def _plan_one(K, L, F, half):
    esz = 2 if half else 4
    R = 16 // esz
    if F < 1 or F > R or R % F:
        return None
    kstep = 16 if half else 8
    s = R // F
    Kd = -(-((L + s - 1) * F) // kstep) * kstep
    ntot = s * K
    npad = -(-ntot // 32) * 32
    best, cut = 0, False
    for ns in (128, 96, 64, 32):
        if npad % ns:
            continue
        if 2 * ns * Kd * esz <= 160 * 1024:
            best = ns
            break
        cut = True
    if not best:
        return None
    nslices = npad // best
    if nslices > 148:
        return None
    slab = (R * 127 + Kd) * esz
    smem = 2 * best * Kd * esz + 2 * 6 * (-(-slab // 16) * 16) + 1024 + 256
    if smem > 227 * 1024:
        return None
    return dict(s=s, NS=best, nslices=nslices, cut=cut)


def _plan(K, L, F, T, dtype):
    """K1 path of a float32 / float64 dictionary: ('fp16' | 'tf32' | 'simt', plan or None)."""
    if dtype != np.float32:
        return 'simt', None
    for half in (True, False):
        p = _plan_one(K, L, F, half)
        if p is not None:
            return ('simt', None) if T * K >= 2 ** 31 else ('fp16' if half else 'tf32', p)
    return 'simt', None


LAUNCHES = {'fp16': 3, 'tf32': 3, 'simt': 1}     # kernels one correlate call launches on each path


def _ilogb(v):
    return int(np.frexp(np.float64(v))[1]) - 1


def split_exponent(mx, top):
    """Host restatement of tc::split_exponent: 2^e puts max|v| in [2^top, 2^(top+1)), clamped to [-126, 127]."""
    if not mx > 0 or not np.isfinite(mx):
        return 0
    return int(min(127, max(-126, top - _ilogb(mx))))


# ------------------------------------------------------------------ inputs

# (name, S, T, F, K, L, dtype, how): how = '' | 'misaligned' (the signal view starts one float into its buffer)
MAP_CASES = [
    # 3xFP16, s = 1 (F = 8): NS = 32 / 64 / 96 / 128, L in {1, 2, odd, even}, T around one M-tile
    ('f8_k32_T1', 3, 1, 8, 32, 16, np.float32, ''),
    ('f8_k32_Tlm1', 3, 15, 8, 32, 16, np.float32, ''),
    ('f8_k32_T127', 3, 127, 8, 32, 16, np.float32, ''),
    ('f8_k32_T128', 3, 128, 8, 32, 16, np.float32, ''),
    ('f8_k32_T129', 3, 129, 8, 32, 16, np.float32, ''),
    ('f8_k64_L7', 1, 300, 8, 64, 7, np.float32, ''),
    ('f8_k96_L1', 3, 129, 8, 96, 1, np.float32, ''),
    ('f8_k128_L2', 1, 130, 8, 128, 2, np.float32, ''),
    # s = 2 (F = 4): four N-slices of 128; T % s != 0; a misaligned view takes the scalar split kernel
    ('f4_k256_T255', 3, 255, 4, 256, 64, np.float32, ''),
    ('f4_k256_T256', 1, 256, 4, 256, 64, np.float32, ''),
    ('f4_k256_T257', 3, 257, 4, 256, 64, np.float32, ''),
    ('f4_k256_T255_misaligned', 3, 255, 4, 256, 64, np.float32, 'misaligned'),
    # s = 4 (F = 2): two N-slices of 96
    ('f2_k48_T511', 3, 511, 2, 48, 5, np.float32, ''),
    ('f2_k48_T512', 1, 512, 2, 48, 5, np.float32, ''),
    ('f2_k48_T513', 3, 513, 2, 48, 5, np.float32, ''),
    # s = 8 (F = 1): 32 slices of 128, 25 or 5 slices of 32, odd T*F (scalar split kernel)
    ('f1_k512_T1023', 1, 1023, 1, 512, 64, np.float32, ''),
    ('f1_k512_T1025', 1, 1025, 1, 512, 64, np.float32, ''),
    ('f1_k100_T1001', 3, 1001, 1, 100, 16, np.float32, ''),
    ('f1_k20_T1', 3, 1, 1, 20, 9, np.float32, ''),
    ('f1_k20_Tlm1', 3, 8, 1, 20, 9, np.float32, ''),
    ('f1_k20_T1023', 3, 1023, 1, 20, 9, np.float32, ''),
    ('f1_k20_T1024', 1, 1024, 1, 20, 9, np.float32, ''),
    ('f1_k20_T1025', 3, 1025, 1, 20, 9, np.float32, ''),
    ('f1_k20_T1023_misaligned', 3, 1023, 1, 20, 9, np.float32, 'misaligned'),
    # long filter: the 160 KB rule cuts the N-slice to 32 columns
    ('f1_L1000', 1, 3001, 1, 16, 1000, np.float32, ''),
    # about 200 short signals: every CTA of a slice walks several (signal, M-tile) pairs across signal boundaries
    ('batch200', 200, 77, 1, 100, 16, np.float32, ''),
    # config 4: 4 x 65536 x 4, 256 filters of 64 taps
    ('config4', 4, 65536, 4, 256, 64, np.float32, ''),
    # 3xTF32: the FP16 plan needs more than 148 N-slices
    ('tf32_k3000_L16', 2, 257, 1, 3000, 16, np.float32, ''),
    ('tf32_k3000_L9', 1, 255, 1, 3000, 9, np.float32, ''),
    # SIMT float32: F the tensor-core layout cannot take, or too many slices for both plans
    ('simt_f3', 3, 100, 3, 10, 5, np.float32, ''),
    ('simt_f5', 1, 64, 5, 7, 1, np.float32, ''),
    ('simt_f6', 1, 65, 6, 33, 2, np.float32, ''),
    ('simt_f16', 3, 130, 16, 40, 4, np.float32, ''),
    ('simt_k5000', 1, 100, 1, 5000, 8, np.float32, ''),
    # SIMT float64
    ('f64_f1', 3, 1025, 1, 20, 9, np.float64, ''),
    ('f64_f4', 1, 257, 4, 256, 64, np.float64, ''),
]


def case_inputs(S, T, F, K, L, dtype, seed):
    """Unit-norm random filters and signals whose amplitude differs from signal to signal by up to 2^6."""
    rs = np.random.RandomState(seed)
    D = rs.randn(K, L, F)
    D /= np.sqrt(np.sum(D * D, axis=(1, 2), keepdims=True))
    x = rs.randn(S, T, F) * (2.0 ** rs.randint(-3, 4, size=(S, 1, 1)))
    return x.astype(dtype), D.astype(dtype)


def _seed(name):
    return sum(ord(ch) * (i + 1) for i, ch in enumerate(name)) % 100003


# ------------------------------------------------------------------ fixtures

@pytest.fixture(scope='module')
def eng():
    import torch
    assert torch.cuda.is_available(), 'gpu tests need a CUDA device'
    from hierarchical_sparse_coding_b200.engine import Engine
    e = Engine(0)
    yield e
    e.close()


def _device_signals(eng, x, how=''):
    import torch
    xt = torch.from_numpy(np.ascontiguousarray(x))
    if how == 'misaligned':
        buf = torch.empty(x.size + 1, dtype=xt.dtype, device=eng.device)
        buf[1:] = xt.reshape(-1).to(eng.device)
        xd = buf[1:].view(x.shape)
        assert xd.data_ptr() % 16 != 0
        return xd
    return xt.to(eng.device)


def _correlate(eng, x, D, how=''):
    """Engine map of x under dictionary D and the number of kernels the call launched."""
    import torch
    eng.set_dictionary(D, dtype=D.dtype)
    xd = _device_signals(eng, x, how)
    n0 = eng.launches
    c = eng.correlate(xd)
    n = eng.launches - n0
    torch.cuda.synchronize()
    return c.cpu().numpy(), n


def _say(capsys, text):
    with capsys.disabled():
        print('\n' + text, end='')


# ------------------------------------------------------------------ 1. the map against float64, per entry

@pytest.mark.gpu
def test_map_matches_float64_on_every_path(eng, capsys):
    worst = {}
    reached = set()
    for name, S, T, F, K, L, dtype, how in MAP_CASES:
        x, D = case_inputs(S, T, F, K, L, dtype, _seed(name))
        path, plan = _plan(K, L, F, T, dtype)
        c, n = _correlate(eng, x, D, how)
        key = path + ('' if dtype == np.float32 else '-f64')
        assert n == LAUNCHES[path], '%s: %d launches, the plan says %s (%d)' % (name, n, path, LAUNCHES[path])
        r = check_map(c, x, D, dtype)
        worst[key] = max(worst.get(key, 0.0), r)
        reached.add(key)
        if plan is not None:
            reached.add('%s s=%d' % (path, plan['s']))
            reached.add('%s NS=%d' % (path, plan['NS']))
            if plan['nslices'] > 1:
                reached.add('%s slices>1' % path)
            if plan['cut']:
                reached.add('%s cut-by-smem' % path)
        if T % (plan['s'] if plan else 1):
            reached.add('T%s!=0')
        _say(capsys, '  %-26s %-5s launches %d  S=%-3d T=%-6d F=%-2d K=%-5d L=%-5d %s  max error/bound %.3f' % (
            name, path, n, S, T, F, K, L, '' if plan is None else 's=%d NS=%d slices=%d' % (plan['s'], plan['NS'], plan['nslices']), r))
    for key, r in sorted(worst.items()):
        _say(capsys, 'K1 %-8s launch signature %d  largest error/bound %.4f' % (key, LAUNCHES[key.split('-')[0]], r))
    need = {'fp16', 'tf32', 'simt', 'simt-f64', 'fp16 s=1', 'fp16 s=2', 'fp16 s=4', 'fp16 s=8', 'fp16 NS=32', 'fp16 NS=64',
            'fp16 NS=96', 'fp16 NS=128', 'fp16 slices>1', 'fp16 cut-by-smem', 'tf32 slices>1', 'T%s!=0'}
    assert need <= reached, 'shape list misses %s' % sorted(need - reached)


# ------------------------------------------------------------------ 2. amplitudes

def amplitude_batch(T, F, dtype, seed=11):
    """One batch: signals scaled by 2^-60 ... 2^60, an all-zero signal in the middle, a single impulse, a signal of
    float32 subnormals only and one with max|x| = 1e-37."""
    rs = np.random.RandomState(seed)
    rows = [rs.randn(T, F) * 2.0 ** e for e in (-60, -30, 0)]
    rows.append(np.zeros((T, F)))
    imp = np.zeros((T, F))
    imp[T // 3, F // 2] = 1.75
    rows.append(imp)
    rows += [rs.randn(T, F) * 2.0 ** e for e in (30, 60)]
    sub = rs.randn(T, F) * 2.0 ** -140
    rows.append(sub)
    tiny = rs.randn(T, F)
    rows.append(tiny / np.abs(tiny).max() * 1e-37)
    x = np.stack(rows).astype(dtype)
    if dtype == np.float32:
        assert np.abs(x[7]).max() < 2.0 ** -126 and np.abs(x[7]).max() > 0       # subnormal only
        assert np.float32(np.abs(x[8]).max()) == np.float32(1e-37)
    return x, 3, 4                       # the batch, the zero signal, the impulse


AMPLITUDE_SHAPES = [   # (F, K, L, dtype): 3xFP16 at s = 8 and s = 1, 3xTF32, SIMT float32, float64
    (1, 64, 16, np.float32),
    (8, 32, 7, np.float32),
    (1, 3000, 16, np.float32),
    (3, 16, 5, np.float32),
    (1, 20, 9, np.float64),
]


@pytest.mark.gpu
@pytest.mark.parametrize('shape', AMPLITUDE_SHAPES, ids=lambda s: 'F%d_K%d_L%d_%s' % (s[0], s[1], s[2], np.dtype(s[3]).name))
def test_map_amplitudes_in_one_batch(eng, capsys, shape):
    F, K, L, dtype = shape
    T = 1001
    x, zero, imp = amplitude_batch(T, F, dtype)
    _, D = case_inputs(1, 1, F, K, L, dtype, 5)
    path, _ = _plan(K, L, F, T, dtype)
    c, n = _correlate(eng, x, D)
    assert n == LAUNCHES[path]
    r = check_map(c, x, D, dtype)
    assert np.all(c[zero] == 0)
    # the impulse: the map is the reversed filter times the sample, and zero away from it
    t0, f0 = T // 3, F // 2
    off = centre_offset(L)
    want = np.zeros((T, K))
    for j in range(L):
        t = t0 + off - j
        if 0 <= t < T:
            want[t] = 1.75 * D[:, j, f0].astype(np.float64)
    assert np.all((c[imp] != 0) <= (want != 0))
    _say(capsys, 'amplitudes %-5s F=%d K=%d L=%d %s: launches %d, largest error/bound %.4f' % (path, F, K, L, np.dtype(dtype).name, n, r))


@pytest.mark.gpu
@pytest.mark.parametrize('F,K,L', [(1, 64, 16), (8, 32, 7), (1, 3000, 16)])
def test_map_dictionary_amplitudes(eng, capsys, F, K, L):
    """A dictionary whose largest tap is 2^-130 (every tap a float32 subnormal) and one whose filter norms differ by 2^20."""
    T = 301
    x, D = case_inputs(3, T, F, K, L, np.float32, 17)
    path, _ = _plan(K, L, F, T, np.float32)
    tiny = (D.astype(np.float64) / np.abs(D).max() * 2.0 ** -130).astype(np.float32)
    assert np.abs(tiny).max() == np.float32(2.0 ** -130)
    wide = D.copy()
    wide[::2] *= np.float32(2.0 ** -20)
    for label, Dc in (('max|D| = 2^-130', tiny), ('norms 2^20 apart', wide)):
        c, n = _correlate(eng, x, Dc)
        assert n == LAUNCHES[path]
        r = check_map(c, x, Dc, np.float32)
        _say(capsys, 'dictionary %-17s %-5s F=%d K=%d L=%d: largest error/bound %.4f' % (label, path, F, K, L, r))


# ------------------------------------------------------------------ 3. no writes outside the map

@pytest.mark.gpu
@pytest.mark.parametrize('S,T,F,K,L,dtype', [
    (3, 1001, 1, 20, 9, np.float32),      # fp16, s = 8
    (3, 513, 2, 48, 5, np.float32),       # fp16, s = 4
    (3, 255, 4, 256, 64, np.float32),     # fp16, s = 2
    (2, 257, 1, 3000, 16, np.float32),    # tf32, s = 4
    (3, 100, 3, 10, 5, np.float32),       # SIMT
    (3, 1001, 1, 20, 9, np.float64),      # SIMT float64
])
def test_correlate_writes_only_the_map(eng, S, T, F, K, L, dtype):
    import torch
    from hierarchical_sparse_coding_b200 import _native as N
    x, D = case_inputs(S, T, F, K, L, dtype, 23)
    eng.set_dictionary(D, dtype=dtype)
    path, plan = _plan(K, L, F, T, dtype)
    assert plan is None or T % plan['s'] != 0
    xd = torch.from_numpy(x).to(eng.device)
    tdt = torch.float32 if dtype == np.float32 else torch.float64
    n_map = S * T * K
    buf = torch.full((n_map + 4096,), float('nan'), dtype=tdt, device=eng.device)
    n0 = eng.launches
    N.check(eng.lib, eng.handle, eng.lib.hsc_b200_correlate(eng.handle, ctypes.c_void_p(xd.data_ptr()), S, T,
                                                            ctypes.c_void_p(buf.data_ptr()), None))
    torch.cuda.synchronize()
    assert eng.launches - n0 == LAUNCHES[path]
    h = buf.cpu().numpy()
    assert not np.any(np.isnan(h[:n_map])), 'map entries left unwritten'
    assert np.all(np.isnan(h[n_map:])), 'K1 wrote %d elements past the map' % int(np.sum(~np.isnan(h[n_map:])))
    check_map(h[:n_map].reshape(S, T, K), x, D, dtype)


# ------------------------------------------------------------------ 4. level-1 keys, exactly

def _align256(v):
    return (v + 255) // 256 * 256


def tie_dictionary(K, L, F, dtype, seed):
    """Random unit filters with exact copies and negations, so that level-1 keys meet exact ties."""
    _, D = case_inputs(1, 1, F, K, L, np.float64, seed)
    D[1] = D[0]
    D[2] = -D[0]
    D[K - 1] = -D[3]
    if K > 40:
        D[37] = D[5]                       # a tie across two 32-column chunks of the fused epilogue
    return D.astype(dtype)


def begin_and_read_keys(eng, x, use_weights):
    """hsc_b200_mp_begin into a caller-owned workspace; returns (map, val1, idx1, launches of the call)."""
    import torch
    from hierarchical_sparse_coding_b200 import _native as N
    S, T, _ = x.shape
    K = eng.K
    rsz = np.dtype(eng.dtype).itemsize
    xd = torch.from_numpy(np.ascontiguousarray(x)).to(eng.device)
    resid = torch.empty_like(xd)
    wsb = eng.workspace_bytes(S, T)
    ws = torch.zeros((wsb,), dtype=torch.uint8, device=eng.device)
    opt = eng.make_options(nbNonzeroCoefs=1, use_weights=use_weights)
    assert eng.lib.hsc_b200_gram_dev(eng.handle)          # the Gram tensor is built by the first pursuit: not counted below
    n0 = eng.launches
    N.check(eng.lib, eng.handle, eng.lib.hsc_b200_mp_begin(eng.handle, ctypes.c_void_p(xd.data_ptr()), ctypes.c_void_p(resid.data_ptr()),
                                                           S, T, ctypes.c_void_p(ws.data_ptr()), wsb, ctypes.byref(opt), None))
    torch.cuda.synchronize()
    n = eng.launches - n0
    assert eng.lib.hsc_b200_mp_map_dev(eng.handle) == ws.data_ptr()
    tdt = torch.float32 if rsz == 4 else torch.float64
    o_val1 = _align256(S * T * K * rsz)
    o_idx1 = o_val1 + _align256(S * T * rsz)
    m = ws[:S * T * K * rsz].view(tdt).reshape(S, T, K).cpu().numpy()
    v1 = ws[o_val1:o_val1 + S * T * rsz].view(tdt).reshape(S, T).cpu().numpy()
    i1 = ws[o_idx1:o_idx1 + S * T * 4].view(torch.int32).reshape(S, T).cpu().numpy()
    return m, v1, i1, n


# (label, F, K, L, dtype, weights): key path, kernels mp_begin launches
KEY_CASES = [
    ('fused s=1', 8, 20, 7, np.float32, False, 4),               # absmax, split, MMA, unpack
    ('fused K%32=0', 1, 64, 16, np.float32, False, 4),
    ('rowkey weights', 1, 64, 16, np.float32, True, 4),          # absmax, split, MMA, rowkey
    ('rowkey s>1', 1, 20, 9, np.float32, False, 4),
    ('rowkey tf32', 1, 3000, 16, np.float32, False, 4),          # absmax, split, MMA, rowkey
    ('rowkey simt', 3, 20, 5, np.float32, True, 2),              # SIMT, rowkey
    ('rowkey f64', 1, 20, 9, np.float64, True, 2),
]


@pytest.mark.gpu
@pytest.mark.parametrize('case', KEY_CASES, ids=lambda c: c[0].replace(' ', '_').replace('%', ''))
def test_level1_keys_exact(eng, capsys, case):
    label, F, K, L, dtype, use_w, launches = case
    S, T = 3, 1001
    D = tie_dictionary(K, L, F, dtype, 31)
    x, _ = case_inputs(S, T, F, K, L, dtype, 37)
    x *= np.asarray([1.0, 2.0 ** 9, 2.0 ** -7], dtype)[:, None, None]      # unequal amplitudes
    w = None
    if use_w:
        w = np.random.RandomState(41).uniform(0.25, 2.0, K).astype(dtype)
        w[1] = w[0]
        w[2] = w[0]
    eng.set_dictionary(D, weights=w, dtype=dtype)
    path, _ = _plan(K, L, F, T, dtype)
    m, v1, i1, n = begin_and_read_keys(eng, x, use_w)
    assert n == launches, '%s: %d launches' % (label, n)
    check_map(m, x, D, dtype)
    score = np.abs(m * w[None, None, :]) if use_w else np.abs(m)
    assert score.dtype == np.dtype(dtype)
    want = score.max(axis=2)
    ui = np.uint32 if dtype == np.float32 else np.uint64
    bad = want.view(ui) != v1.view(ui)
    assert not bad.any(), '%s: val1 differs from max_k |map*w| in %d rows, first %s' % (label, int(bad.sum()), np.argwhere(bad)[0])
    first = np.argmax(score, axis=2)              # first occurrence = the lowest filter reaching the maximum
    pos = v1 > 0
    assert pos.sum() > 0.9 * S * T
    assert np.array_equal(i1[pos], first[pos]), '%s: idx1 differs in %d rows' % (label, int(np.sum(i1[pos] != first[pos])))
    ties = int(np.sum(np.sum(score == want[:, :, None], axis=2) > 1))
    if path == 'simt':
        assert ties > 0, 'the duplicated filters gave no exact tie'
    _say(capsys, 'keys %-15s %-5s launches %d: %d rows, %d exact ties, bit-exact' % (label, path, n, S * T, ties))


# ------------------------------------------------------------------ 5. float32 Gram tensor

@pytest.mark.gpu
@pytest.mark.parametrize('K,L,F', [(256, 64, 4), (512, 64, 1), (20, 7, 2), (1, 9, 3)])
def test_gram_float32_within_one_ulp(eng, K, L, F):
    """gram_kernel accumulates in double and rounds once: within one float32 ulp of float32(G64), plus the float64
    accumulation error of either side (2 (n + 2) 2^-53 sum |a b|), far below what float32 accumulation would leave."""
    _, D = case_inputs(1, 1, F, K, L, np.float32, 43 + K)
    eng.set_dictionary(D, dtype=np.float32)
    G = eng.gram()
    assert G.dtype == np.float32 and G.shape == (K, 2 * L - 1, K)
    Dd = D.astype(np.float64)
    ref = np.zeros((K, 2 * L - 1, K))
    mag = np.zeros_like(ref)
    for tau in range(-(L - 1), L):
        jlo, jhi = max(0, -tau), min(L, L - tau)
        a = Dd[:, jlo + tau:jhi + tau].reshape(K, -1)
        b = Dd[:, jlo:jhi].reshape(K, -1)
        ref[:, tau + L - 1, :] = a @ b.T
        mag[:, tau + L - 1, :] = np.abs(a) @ np.abs(b).T
    r32 = ref.astype(np.float32)
    n = L * F
    tol = np.spacing(np.abs(r32)).astype(np.float64) + 2 * (n + 2) * 2.0 ** -53 * mag
    err = np.abs(G.astype(np.float64) - r32.astype(np.float64))
    assert np.all(err <= tol), 'Gram entry off by %.3g ulp' % float(np.max(err / np.spacing(np.abs(r32)).astype(np.float64)))


# ------------------------------------------------------------------ 6. matching pursuit above 2^31 map entries

@pytest.mark.gpu
def test_pursuit_map_above_2_31_entries(eng, capsys):
    """One signal of T = 2^24 + 1001 samples and 128 filters: 2.1e9 map entries (8.6 GB).  K1 takes the SIMT kernel (the
    tensor-core path is limited to T*K < 2^31) and mp_begin builds the level-1 keys with rowkey_kernel (2 launches).  K2
    takes the global-memory argmax hierarchy: one 8-byte key per 128-row group is 131 k keys, 1 MB, which the
    shared-memory hierarchy cannot hold.  24 atoms are planted around t = 2^24, where t*K + k crosses 2^31; every other
    sample is zero, so an oracle run on a crop around the atoms is the whole pursuit."""
    import torch
    from hierarchical_sparse_coding_b200 import _native as N
    from oracle import hsc_oracle as O
    T, K, L, F = 2 ** 24 + 1001, 128, 16, 1
    assert T * K >= 2 ** 31
    rs = np.random.RandomState(47)
    D = O.normalize(rs.randn(K, L)).astype(np.float32)
    eng.set_dictionary(D[:, :, None], dtype=np.float32)
    assert eng.lib.hsc_b200_gram_dev(eng.handle)
    off = centre_offset(L)
    c0, c1 = 2 ** 24 - 1000, 2 ** 24 + 1000
    crop = np.zeros(c1 - c0, np.float32)
    n_atoms = 24
    pos = 2 ** 24 - 12 * 40 + 40 * np.arange(n_atoms) + rs.randint(0, 8, n_atoms)
    for t, k, a in zip(pos, rs.randint(0, K, n_atoms), rs.uniform(1.0, 4.0, n_atoms) * rs.choice([-1, 1], n_atoms)):
        crop[t - off - c0:t - off - c0 + L] += np.float32(a) * D[k]
    xd = torch.zeros((1, T, 1), dtype=torch.float32, device=eng.device)
    xd[0, c0:c1, 0] = torch.from_numpy(crop).to(eng.device)
    resid = torch.empty_like(xd)
    wsb = eng.workspace_bytes(1, T)
    ws = torch.empty((wsb,), dtype=torch.uint8, device=eng.device)
    opt = eng.make_options(nbNonzeroCoefs=n_atoms)
    try:
        n0 = eng.launches
        N.check(eng.lib, eng.handle, eng.lib.hsc_b200_mp_begin(eng.handle, ctypes.c_void_p(xd.data_ptr()), ctypes.c_void_p(resid.data_ptr()),
                                                               1, T, ctypes.c_void_p(ws.data_ptr()), wsb, ctypes.byref(opt), None))
        torch.cuda.synchronize()
        assert eng.launches - n0 == 2, 'expected the SIMT K1 and rowkey_kernel'
        # K1: the map rows around t = 2^24, read as device slices
        r0, r1 = 2 ** 24 - 600, 2 ** 24 + 600
        assert r0 * K < 2 ** 31 <= r1 * K
        rows = ws[r0 * K * 4:r1 * K * 4].view(torch.float32).reshape(1, r1 - r0, K).cpu().numpy()
        c64, a = corr64(crop[None, :, None], D[:, :, None])
        ref = (c64[:, r0 - c0:r1 - c0], a[:, r0 - c0:r1 - c0])
        xr = crop[None, r0 - c0 - L:r1 - c0 + L, None]          # the samples these rows see (max|x| of the bound)
        r = check_map(rows, xr, D[:, :, None], np.float32, ref=ref)
        assert np.abs(rows).max() > 1.0
        # K2
        cap = 64
        evp = torch.zeros((1, cap), dtype=torch.int32, device=eng.device)
        evi = torch.zeros((1, cap), dtype=torch.int32, device=eng.device)
        evc = torch.zeros((1, cap), dtype=torch.float32, device=eng.device)
        states = (N.SignalState * 1)()
        N.check(eng.lib, eng.handle, eng.lib.hsc_b200_mp_run(eng.handle, ctypes.c_void_p(evp.data_ptr()), ctypes.c_void_p(evi.data_ptr()),
                                                             ctypes.c_void_p(evc.data_ptr()), cap, states, None))
        m = int(states[0].n_buffered)
        _, r_ref, tr = O.mp_encode(crop, D, nbNonzeroCoefs=n_atoms, return_trace=True)
        t_ref, k_ref, c_ref = tr.arrays()
        assert m == len(t_ref) == n_atoms
        got_t = evp[0, :m].cpu().numpy()
        assert np.array_equal(got_t, t_ref + c0) and np.array_equal(evi[0, :m].cpu().numpy(), k_ref)
        assert np.allclose(evc[0, :m].cpu().numpy(), c_ref, rtol=1e-5, atol=0)
        res = resid[0, :, 0].cpu().numpy()
        assert np.allclose(res[c0:c1], r_ref, rtol=0, atol=1e-5)
        assert not np.any(res[:c0]) and not np.any(res[c1:]), 'residual differs from x outside the atoms'
        _say(capsys, 'T*K = %.3g: SIMT K1 rows across 2^31 largest error/bound %.4f; K2 %d atoms equal the oracle' % (T * K, r, m))
    finally:
        del ws, resid, xd
        torch.cuda.empty_cache()


# ------------------------------------------------------------------ 7. the bound can fail (host only)

def _split16(v):
    h = v.astype(np.float16)
    lo = ((v - h.astype(np.float32)) * np.float32(2048.0)).astype(np.float16)
    return h.astype(np.float64), lo.astype(np.float64)


def test_bound_rejects_a_lost_split_product():
    """NumPy restatement of the 3xFP16 product on inputs of the map test, once whole and once without A_lo * B_hi: the
    whole product passes the per-entry bound, the one missing a product does not."""
    for name in ('f8_k32_T129', 'f8_k96_L1', 'f2_k48_T513', 'f1_k20_T1025'):
        case = [c for c in MAP_CASES if c[0] == name][0]
        _, S, T, F, K, L, dtype, _ = case
        x, D = case_inputs(S, T, F, K, L, dtype, _seed(name))
        assert _plan(K, L, F, T, dtype)[0] == 'fp16'
        ed = split_exponent(float(np.abs(D).max()), -1)
        dh, dl = _split16(D * np.float32(2.0 ** ed))
        whole = np.empty((S, T, K))
        lost = np.empty((S, T, K))
        for s in range(S):
            ex = split_exponent(float(np.abs(x[s]).max()), 9)
            xh, xl = _split16(x[s:s + 1] * np.float32(2.0 ** ex))
            hh = corr64(xh, dh)[0]
            hl = corr64(xh, dl)[0]
            lh = corr64(xl, dh)[0]
            scale = 2.0 ** -(ex + ed)
            whole[s] = ((hh + (hl + lh) * 2.0 ** -11) * scale)[0]
            lost[s] = ((hh + hl * 2.0 ** -11) * scale)[0]
        ref = corr64(x, D)
        assert check_map(whole.astype(np.float32), x, D, np.float32, ref=ref) <= 1.0
        with pytest.raises(AssertionError, match='> bound'):
            check_map(lost.astype(np.float32), x, D, np.float32, ref=ref)

