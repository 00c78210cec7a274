#!/usr/bin/env python
"""Benchmark of the matching-pursuit hot path (BASELINE.json metric: MP atoms selected/s and signal
samples encoded/s at 1/2/4/8 B200).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c4|c2|c5] [--impl b200|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path (K1 initial correlation + K2 select/update loop to the stop
rule) over one batch of synthetic signals.  Default workload: BASELINE config 4's per-GPU shard
(512 independent signals of 65 536 samples x 4 channels, 256 filters of length 64, 655 atoms =
1 % L0 budget per signal) - the configuration the 1/2/4/8-GPU metric is quoted on; weak scaling
(every rank encodes its own 512 signals; 8 ranks = the full 4096-signal config).  Config 2 (one
1M-sample sequence, 16 filters of length 32) is a single sequence = replicas only; it is measured
with --workload c2 and reported in `extra` of the default line.

Prints ONE JSON line (rank 0).  `value` = atoms/s with inputs resident in HBM; `e2e` = the same
through the public API from pinned HOST buffers (H2D of the signals and D2H of codes + residual
inside the timed region).  `--impl reference` times the UNMODIFIED reference itself
(hsc.modeling.ConvolutionalMatchingPursuit from the git-ignored copy baseline/_ref, imported
through the Python-2 hook tests/golden/ref_loader.py) on the box's host cores: one process per core
over independent signals of the same workload - the reference's only parallel idiom - with one BLAS
thread each; `value` = atoms applied / wall time, measured (no extrapolation).  Both arms print
the same declarative `config`.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

if '--impl' in sys.argv and sys.argv[sys.argv.index('--impl') + 1:][:1] == ['reference'] or '--impl=reference' in sys.argv:
    # CPU arm: one process per host core over independent signals (the reference's only parallel idiom), so every
    # process gets ONE BLAS thread - set before NumPy loads its BLAS, the only moment it is read
    for _v in ('OPENBLAS_NUM_THREADS', 'OMP_NUM_THREADS', 'MKL_NUM_THREADS'):
        os.environ[_v] = '1'

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (S per GPU, T, F, K, L, atoms per signal)
    'c4': dict(S=512, T=65536, F=4, K=256, L=64, atoms=655, desc='config4 shard: 512 signals x 65536 x 4ch, 256 filters x 64, nbNonzeroCoefs=655'),
    'c2': dict(S=1, T=1000000, F=1, K=16, L=32, atoms=10000, desc='config2 shape: 1 sequence x 1e6, 16 filters x 32, nbNonzeroCoefs=10000'),
    'c5': dict(S=190, T=65536, F=1, K=512, L=64, atoms=655, desc='config5 segments: 190 x 65536, 512 filters x 64, nbNonzeroCoefs=655'),
    'tiny': dict(S=8, T=4096, F=4, K=32, L=16, atoms=40, desc='smoke-sized'),
}


NOISE_DB = -30.0


def centre_offset(L):
    return L // 2 - 1 if L % 2 == 0 else L // 2


def make_dictionary(w, seed=42):
    rs = np.random.RandomState(seed)
    D = rs.randn(w['K'], w['L'], w['F'])
    D /= np.sqrt(np.sum(D * D, axis=(1, 2), keepdims=True))
    return D.astype(np.float32)


def make_signals(w, D, seed, S=None):
    """Planted-atom law of the reference's generators (hsc/dataset.py:742: amplitudes U(0.25,4)),
    centres U{L, T-L}, filters uniform; float32 like the generated datasets (:456, :772)."""
    rs = np.random.RandomState(seed)
    S = w['S'] if S is None else S
    T, F, K, L, n = w['T'], w['F'], w['K'], w['L'], w['atoms']
    off = centre_offset(L)
    x = np.zeros((S, T, F), dtype=np.float32)
    for s in range(S):
        pos = rs.randint(L, T - L, size=n)
        idx = rs.randint(0, K, size=n)
        amp = rs.uniform(0.25, 4.0, size=n).astype(np.float32)
        xs = x[s]
        for p, k, a in zip(pos - off, idx, amp):
            xs[p:p + L] += a * D[k]
        # white noise 30 dB below the signal (SURVEY 8d, config 4), so the L0 budget is the binding stop rule
        sigma = math.sqrt(float(np.mean(np.square(xs, dtype=np.float64))) * 10.0 ** (NOISE_DB / 10.0))
        xs += (sigma * rs.randn(T, F)).astype(np.float32)
    return x


def per_atom_bytes(w, s=4):
    """Algorithmic bytes per selected atom (SURVEY 8d): window read+write, Gram slice, residual RMW + atom."""
    return 3 * (2 * w['L'] - 1) * w['K'] * s + 3 * w['L'] * w['F'] * s


def correlation_flops(w):
    return 2.0 * w['S'] * w['T'] * w['K'] * w['L'] * w['F']


def correlation_bytes(w, s=4):
    return float(w['S']) * w['T'] * (w['K'] + w['F']) * s


def load_traffic(workload):
    """DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) of the two kernels from the committed `ncu --set full`
    capture of this workload (profiles/traffic.json names the report): K1 per signal, K2 per applied atom."""
    p = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get(workload)
    return None


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm=float(d['hbm_gbs']), bf16=float(d['bf16_tflops']), bf16_sustained=float(d.get('bf16_tflops_sustained', d['bf16_tflops'])),
                    source='measured')
    return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, source='fallback')


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index):
        threading.Thread.__init__(self, daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop_evt = threading.Event()

    def run(self):
        q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q, '--format=csv,noheader,nounits'],
                                     stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=5).stdout.strip()
                parts = [p.strip() for p in out.split(',')]
                if len(parts) >= 6:
                    self.samples.append(float(parts[0]))
                    self.max_mhz = float(parts[1])
                    for nme, v in zip(names, parts[2:6]):
                        if v.lower().startswith('active'):
                            self.reasons.add(nme)
            except Exception:
                pass
            self._stop_evt.wait(0.02)          # nvidia-smi itself takes tens of ms: the timed region of 5 steps is ~0.2 s

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        med = float(np.median(self.samples)) if self.samples else None
        return dict(sm_mhz=med, sm_max_mhz=self.max_mhz, reasons=sorted(self.reasons), samples=len(self.samples))


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own hsc.modeling.ConvolutionalMatchingPursuit on the host cores
# ------------------------------------------------------------------------------------------------

def workload_config(w, coef_mode=1):
    """`config` of the JSON line: the declarative description of the workload, identical in both arms."""
    return {'workload': w['desc'], 'noise_db': NOISE_DB, 'signals_per_gpu': w['S'], 'T': w['T'], 'F': w['F'], 'K': w['K'], 'L': w['L'],
            'nb_nonzero_coefs': w['atoms'],
            'parallelism': 'independent signals sharded over the GPUs, one gather of the codes',
            'cache': 'inputs larger than L2 (%.1f GB map + %.2f GB signals per GPU)' % (w['S'] * w['T'] * w['K'] * 4 / 1e9, w['S'] * w['T'] * w['F'] * 4 / 1e9)}


def load_reference_modeling():
    """hsc.modeling of the UNMODIFIED reference (baseline/_ref on the GPU box, /root/reference in the dev container)
    through the Python-2 import hook; None when no copy of the reference is there."""
    sys.path.insert(0, os.path.join(ROOT, 'tests', 'golden'))
    try:
        import ref_loader
        if not ref_loader.reference_available():
            return None
        import logging
        import warnings
        warnings.simplefilter('ignore')
        mod = ref_loader.load_reference().modeling
        logging.getLogger('hsc').setLevel(logging.ERROR)
        return mod
    except Exception as e:          # noqa: BLE001
        sys.stderr.write('bench.py: reference not importable (%s)\n' % (e,))
        return None


_REF = {}


def _cpu_worker(args):
    """One signal through the CPU implementation: the reference's ConvolutionalMatchingPursuit.computeCoefficients
    (kind 'reference'), or - only when no copy of the reference is there - the oracle port.  Returns (atoms applied,
    seconds).  `n_atoms` is passed as the reference's own nbNonzeroCoefs stop rule."""
    x, D, n_atoms = args
    mod = _REF.get('modeling')
    t0 = time.perf_counter()
    if mod is not None:
        approx = mod.ConvolutionalMatchingPursuit()
        n_events = [0]
        orig = approx._updateCoefficients

        def counted(coefficients, atoms, replace=True):
            n_events[0] += len(atoms)
            return orig(coefficients, atoms, replace=replace)
        approx._updateCoefficients = counted
        approx.computeCoefficients(x, D, nbNonzeroCoefs=n_atoms)
        n = n_events[0]
    else:
        from oracle import hsc_oracle as O
        _, _, tr = O.mp_encode(x, D, nbNonzeroCoefs=n_atoms, bookkeeping='lil', return_trace=True)
        n = len(tr.events)
    return n, time.perf_counter() - t0


def _limit_blas_threads(n):
    try:
        import threadpoolctl
        return threadpoolctl.threadpool_limits(limits=n)
    except Exception:           # noqa: BLE001
        return None


def cpu_reference_step(signals, D, n_atoms, pool, procs):
    """One bounded sample: `procs` independent signals, nbNonzeroCoefs = n_atoms each, one process per signal, all
    running at once.  Returns (atoms applied by all processes, wall seconds of the step): measured, not extrapolated."""
    t0 = time.perf_counter()
    res = pool.map(_cpu_worker, [(signals[i], D, n_atoms) for i in range(procs)], chunksize=1)
    return sum(r[0] for r in res), time.perf_counter() - t0, res


def run_reference_arm(args, w):
    import multiprocessing as mp
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:           # noqa: BLE001
        cores = os.cpu_count() or 1
    procs = max(1, min(cores, 128))
    mod = load_reference_modeling()
    _REF['modeling'] = mod
    kind = 'reference' if mod is not None else 'port'
    D = make_dictionary(w)
    base = make_signals(w, D, seed=1000, S=min(procs, 8))
    signals = [base[i % len(base)] for i in range(procs)]
    budget = float(os.environ.get('HSC_BENCH_CPU_BUDGET_S', '170'))      # the whole --steps/--warmup run
    n_steps = args.steps + min(args.warmup, 1)
    ctx = mp.get_context('fork')                   # workers inherit the loaded reference and the signals
    with ctx.Pool(procs) as pool:
        # calibration (untimed): a short sample with every core busy gives the cost of the initial correlation + per atom
        n_cal = 8
        t0 = time.perf_counter()
        a1, dt1, _ = cpu_reference_step(signals, D, n_cal, pool, procs)
        a2, dt2, _ = cpu_reference_step(signals, D, 3 * n_cal, pool, procs)
        per_atom = max((dt2 - dt1) / max((a2 - a1) / procs, 1), 1e-4)
        t_init = max(dt1 - per_atom * a1 / procs, 0.0)
        left = budget - (time.perf_counter() - t0)
        per_step = max(left / max(n_steps, 1), 2.0)
        n_atoms = int(max(4, min(w['atoms'], (per_step - t_init) / per_atom)))
        for _ in range(min(args.warmup, 1)):
            cpu_reference_step(signals, D, n_atoms, pool, procs)
        atoms, tot_t = 0, 0.0
        for _ in range(args.steps):
            a, dt, _ = cpu_reference_step(signals, D, n_atoms, pool, procs)
            atoms += a
            tot_t += dt
    value = atoms / max(tot_t, 1e-9)
    full = n_atoms >= w['atoms']
    sample = ('%s on %d host cores: %d processes x 1 signal of the workload each, running concurrently with one BLAS thread each; '
              'every step each process runs computeCoefficients(x, D, nbNonzeroCoefs=%d)%s; value = atoms applied by all processes / '
              'wall time of the timed steps (measured, initial correlation included: ~%.2f s per signal, then ~%.1f ms per atom)' % (
                  'hsc.modeling.ConvolutionalMatchingPursuit of the unmodified reference (baseline/_ref via the py2 import hook)'
                  if kind == 'reference' else 'oracle port (no copy of the reference found)',
                  procs, procs, n_atoms, ' = the whole signal' if full else ' (a bounded prefix of the %d-atom budget, sized to the time limit)' % w['atoms'],
                  t_init, 1e3 * per_atom))
    line = {
        'impl': 'reference', 'metric': 'mp_atoms_per_s', 'value': value, 'unit': 'atoms/s', 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': 1000.0 * tot_t / max(args.steps, 1), 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(w),
        'cpu_baseline': {'value': value, 'unit': 'atoms/s', 'cores': procs, 'kind': kind, 'sample': sample,
                         'nb_nonzero_coefs_per_step': n_atoms, 'blas_threads_per_process': 1, 'numpy': np.__version__},
        'e2e': {'value': value, 'unit': 'atoms/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'samples_per_s': value * w['T'] / w['atoms'],
    }
    print(json.dumps(line))


def cpu_baseline_sample(w, D, budget_s=14.0):
    """The reference's own ConvolutionalMatchingPursuit (single process, one BLAS thread) on ONE signal of the workload,
    with the L0 budget cut to what fits ~budget_s (reported beside the GPU number; measured, not extrapolated)."""
    mod = load_reference_modeling()
    _REF['modeling'] = mod
    kind = 'reference' if mod is not None else 'port'
    x = make_signals(w, D, seed=1000, S=1)[0]
    lim = _limit_blas_threads(1)
    try:
        n1, dt1 = _cpu_worker((x, D, 6))
        n2, dt2 = _cpu_worker((x, D, 18))
        per = max((dt2 - dt1) / max(n2 - n1, 1), 1e-4)
        t_init = max(dt1 - per * n1, 0.0)
        n_atoms = int(max(4, min(w['atoms'], (budget_s - t_init) / per)))
        n, dt = _cpu_worker((x, D, n_atoms))
    finally:
        if lim is not None:
            lim.restore_original_limits() if hasattr(lim, 'restore_original_limits') else lim.unregister()
    return {'value': n / dt, 'unit': 'atoms/s', 'cores': 1, 'kind': kind,
            'sample': '%s, 1 process / 1 BLAS thread, 1 signal of the workload with nbNonzeroCoefs=%d%s: %d atoms in %.1f s (initial '
                      'correlation ~%.2f s included, ~%.1f ms per atom)' % (
                          'hsc.modeling.ConvolutionalMatchingPursuit of the unmodified reference' if kind == 'reference' else 'oracle port',
                          n_atoms, '' if n_atoms < w['atoms'] else ' (the whole signal)', n, dt, t_init, 1e3 * per),
            'host_cores_available': os.cpu_count()}


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------

DUMP_LIMIT_BYTES = 60 * 10 ** 6          # under 64 MB with the .npy headers, whichever megabyte is meant
DUMP_RESIDUAL_BYTES = 16 * 2 ** 20


def dump_outputs(out_dir, compact, resid, states):
    """Writes what one step of the timed path returned, as float32 / float64 .npy files under out_dir, so that two builds
    can be compared output for output on the same seeded inputs:
      code_signal, code_pos, code_filter, code_coef  the sparse codes: one entry per selected atom, signal by signal in
                                                     selection order (the engine's device compaction of the event buffers)
      energy_residual                                the final residual energy the engine reports for every signal
      residual_signals, residual                     the residual signals [n, T, F] of a fixed seeded sample of n signals
                                                     (all of them would not fit the 64 MB the dump may take)
    When the codes of all signals could not fit either (at the event-buffer capacity of every signal), a fixed seeded sample
    of signals, chosen from the number of signals and that capacity alone, keeps its codes: two builds dump the same signals.
    With several GPUs this is rank 0's own shard, as rank 0 computed it before the gather of the codes."""
    import torch
    S, T, F = resid.shape
    off = compact['offsets'].cpu().numpy()
    total = int(off[-1])
    sig = np.repeat(np.arange(S), np.diff(off))
    pos = compact['pos'][:total].cpu().numpy()
    idx = compact['idx'][:total].cpu().numpy()
    coef = compact['coef'][:total].cpu().numpy()
    n_res = max(1, min(S, DUMP_RESIDUAL_BYTES // (T * F * resid.element_size())))
    res_rows = np.sort(np.random.RandomState(0).choice(S, n_res, replace=False))
    per_atom = 3 * 8 + coef.itemsize
    budget = DUMP_LIMIT_BYTES - n_res * (8 + T * F * resid.element_size()) - 8 * S
    cap = compact['pos'].numel() // S
    if S * cap * per_atom > budget:
        keep = np.sort(np.random.RandomState(1).permutation(S)[:budget // (cap * per_atom)])
        mask = np.isin(sig, keep)
        sig, pos, idx, coef = sig[mask], pos[mask], idx[mask], coef[mask]
    arrays = {'code_signal': sig.astype(np.float64), 'code_pos': pos.astype(np.float64), 'code_filter': idx.astype(np.float64),
              'code_coef': coef, 'energy_residual': np.array([st.energy_residual for st in states], dtype=np.float64),
              'residual_signals': res_rows.astype(np.float64),
              'residual': resid[torch.as_tensor(res_rows, device=resid.device)].cpu().numpy()}
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_LIMIT_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), name
        np.save(os.path.join(out_dir, name + '.npy'), a)


def quick_workload(hsc, torch, dev, local_rank, name, steps, warmup):
    """A few resident steps of another BASELINE configuration (one step after the other, CUDA events), for the `extra` section."""
    w = dict(WORKLOADS[name])
    if name == 'c2':
        w['atoms'] = 3000                      # a 3000-atom prefix of the 1e6-sample sequence: per-atom latency is what matters
    S, T, F, K, L, n_atoms = w['S'], w['T'], w['F'], w['K'], w['L'], w['atoms']
    D = make_dictionary(w)
    x_host = make_signals(dict(w, atoms=WORKLOADS[name]['atoms']), D, seed=2000)
    eng = hsc.Engine(local_rank)
    eng.set_dictionary(D)
    opt = eng.make_options(nbNonzeroCoefs=n_atoms)
    cap = int(n_atoms * 4) + 64
    xd = torch.from_numpy(x_host).to(dev)
    resid = torch.empty_like(xd)
    evp = torch.empty((S, cap), dtype=torch.int32, device=dev)
    evi = torch.empty((S, cap), dtype=torch.int32, device=dev)
    evc = torch.empty((S, cap), dtype=torch.float32, device=dev)
    stream = torch.cuda.current_stream(dev)
    k1, k2, atoms = [], [], 0
    for it in range(warmup + steps):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        ev[0].record(stream)
        eng.begin_only(xd, opt, resid)
        ev[1].record(stream)
        states = eng.run_only(evp, evi, evc, cap, sync_states=True)
        ev[2].record(stream)
        torch.cuda.synchronize(dev)
        if it >= warmup:
            k1.append(ev[0].elapsed_time(ev[1]))
            k2.append(ev[1].elapsed_time(ev[2]))
        atoms = int(sum(st.n_events for st in states))
    k1m, k2m = float(np.mean(k1)), float(np.mean(k2))
    out = {'workload': w['desc'] if name != 'c2' else 'config2 shape: 1 sequence x 1e6, 16 filters x 32, nbNonzeroCoefs=3000',
           'atoms_per_step': atoms, 'k1_ms': k1m, 'k2_ms': k2m, 'atoms_per_s': atoms / ((k1m + k2m) / 1e3),
           'us_per_selection_per_signal': 1e3 * k2m / (atoms / S), 'k2_algorithmic_gbs': atoms * per_atom_bytes(w) / (k2m / 1e3) / 1e9,
           'mode': 'one step after the other, %d timed steps' % steps}
    if name == 'c5':
        rs = np.random.RandomState(7)
        D0 = D.astype(np.float64) + 0.3 * rs.randn(*D.shape) / math.sqrt(D.shape[1] * D.shape[2])
        D0 /= np.sqrt(np.sum(D0 * D0, axis=(1, 2), keepdims=True))
        del xd, resid, evp, evi, evc
        learner = hsc.ConvolutionalDictionaryLearner(K, L, algorithm='ksvd', device=local_rank)
        learner.train(x_host, method='cmp', maxIterations=warmup + steps, toleranceSnr=None, nbNonzeroCoefs=n_atoms, initD=D0, dtype=np.float32)
        torch.cuda.synchronize(dev)
        h = learner.history[warmup:]
        out['ksvd_loop'] = {'iterations': len(learner.history), 'encode_ms': 1e3 * float(np.mean([q['encode_s'] for q in h])),
                            'update_ms': 1e3 * float(np.mean([q['update_s'] for q in h])),
                            'per_iteration_ms': [[round(1e3 * q['encode_s'], 1), round(1e3 * q['update_s'], 1)] for q in learner.history],
                            'note': 'ConvolutionalDictionaryLearner(algorithm=ksvd).train on the 190 segments (cmp, float32 inference, float64 update); mean of iterations %d-%d' % (warmup + 1, warmup + steps)}
    eng.close()
    torch.cuda.empty_cache()
    return out


def run_b200_arm(args, w):
    import torch
    import torch.distributed as dist
    import hierarchical_sparse_coding_b200 as hsc
    from hierarchical_sparse_coding_b200 import distributed as hd

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device; the engine has no CPU fallback (use --impl reference for the CPU arm)')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)

    S, T, F, K, L, n_atoms = w['S'], w['T'], w['F'], w['K'], w['L'], w['atoms']
    D = make_dictionary(w)
    x_host = make_signals(w, D, seed=1000 + rank)
    eng = hsc.Engine(local_rank)
    eng.set_dictionary(D)
    opt = eng.make_options(nbNonzeroCoefs=n_atoms, coef_mode=args.coef_mode, rerank_tolerance=args.rerank_tol)
    cap = int(n_atoms * 4) + 64      # selections incl. re-selected (t,k); nnz counts distinct entries only

    x_pin = torch.from_numpy(x_host).pin_memory()
    xd = x_pin.to(dev)
    resid = torch.empty_like(xd)
    stream = torch.cuda.current_stream(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    gather_stream = torch.cuda.Stream(device=dev) if world > 1 else None
    ev_sets = [dict(evp=torch.empty((S, cap), dtype=torch.int32, device=dev), evi=torch.empty((S, cap), dtype=torch.int32, device=dev),
                    evc=torch.empty((S, cap), dtype=torch.float32, device=dev), compact=None) for _ in range(2)]

    def gather(es, n_atoms_rank):
        """The one collective of the path: NCCL gather of the sparse codes, straight from the device event buffers
        (compacted on the device), on a side stream - the next step's correlation does not wait for it."""
        if world == 1:
            return
        done = torch.cuda.Event()
        done.record(stream)
        with torch.cuda.stream(gather_stream):
            gather_stream.wait_event(done)
            es['compact'] = eng.compact_events(es['evp'], es['evi'], es['evc'], out=es['compact'], stream=gather_stream)
            compacted = torch.cuda.Event()
            compacted.record(gather_stream)
            stream.wait_event(compacted)            # the next step resets the per-signal states the compaction reads
            dev_codes = dict(es['compact'], total=n_atoms_rank)
            hd.gather_device_events(dev_codes, dst=0)

    # ---- resident-input step: K1 + K2 (+ gather of the codes for N > 1), CUDA events on the launch stream
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    k1_ms, k2_ms = [], []
    stop_hist = {}
    run_info = {}
    from hierarchical_sparse_coding_b200._native import STOP_NAMES
    atoms_step = 0

    def run_to_completion(evp, evi, evc):
        """K2 launches until every signal has stopped (a full event buffer pauses a signal: drain + resume)."""
        n_buffered = 0
        while True:
            states = eng.run_only(evp, evi, evc, cap, sync_states=True)
            n_buffered += int(sum(st.n_buffered for st in states))
            if not any(st.status in (0, 6, 7) for st in states):
                return states, n_buffered

    step_no = [0]
    last_step = {}

    def step_resident(record):
        nonlocal atoms_step
        es = ev_sets[step_no[0] & 1]
        step_no[0] += 1
        evp, evi, evc = es['evp'], es['evi'], es['evc']
        ev[0].record(stream)
        eng.begin_only(xd, opt, resid)
        ev[1].record(stream)
        states, n_buffered = run_to_completion(evp, evi, evc)
        ev[2].record(stream)
        gather(es, n_buffered)
        if record:
            ev[2].synchronize()
            k1_ms.append(ev[0].elapsed_time(ev[1]))
            k2_ms.append(ev[1].elapsed_time(ev[2]))
        atoms_step = int(sum(st.n_events for st in states))
        last_step.update(es=es, states=states)
        run_info['reranked_selections'] = int(sum(st.reranked for st in states))
        stop_hist.clear()
        for st in states:
            stop_hist[STOP_NAMES.get(st.status, str(st.status))] = stop_hist.get(STOP_NAMES.get(st.status, str(st.status)), 0) + 1
        bad = [st.status for st in states if st.status in (0, 6, 7)]
        assert not bad, 'some signals did not reach a stop rule: %s' % bad[:4]
        return atoms_step

    # ---- the same steps as a streaming pipeline (default): two encode slots (own workspace each), the correlation of
    # step i+1 on its own stream while the pursuit of step i is still running, pursuit launches on alternating streams so
    # that the CTAs of step i+1 move into the SMs the tail of step i frees.  No host synchronisation inside a step: the
    # states of step i are read (and its codes gathered, N > 1) after step i+1 has been enqueued.
    n_slots = max(2, args.slots)
    slots = eng.make_slots(n_slots, S, T, cap) if args.pipeline else None
    # the correlation stream has the HIGHER priority: when an SM frees resources, waiting K1 CTAs are placed before waiting
    # K2 CTAs, so K1 (one CTA per SM, tensor-bound) runs alongside two pursuit CTAs per SM instead of behind all of them
    s_k1 = torch.cuda.Stream(device=dev, priority=-1 if args.k1_priority else 0) if args.pipeline else None
    s_k2 = [torch.cuda.Stream(device=dev) for _ in range(n_slots)] if args.pipeline else None
    pipe_compact = [None] * n_slots

    def finalize(i, rec):
        """Host side of step i, after its pursuit: states -> atoms / stop reasons; N > 1: compaction + NCCL gather."""
        nonlocal atoms_step
        sl = slots[i % n_slots]
        sl.k2_done.synchronize()
        states = sl.states
        atoms_step = int(sum(st.n_events for st in states))
        run_info['reranked_selections'] = int(sum(st.reranked for st in states))
        stop_hist.clear()
        for st in states:
            nm = STOP_NAMES.get(st.status, str(st.status))
            stop_hist[nm] = stop_hist.get(nm, 0) + 1
        bad = [st.status for st in states if st.status in (0, 6, 7)]
        assert not bad, 'some signals did not reach a stop rule: %s' % bad[:4]
        if world > 1:
            with torch.cuda.stream(gather_stream):
                gather_stream.wait_event(sl.k2_done)
                pipe_compact[i % n_slots] = sl.compact(pipe_compact[i % n_slots], gather_stream)
                hd.gather_device_events(dict(pipe_compact[i % n_slots], total=int(sum(st.n_buffered for st in states))), dst=0)
                sl.gather_done = torch.cuda.Event()
                sl.gather_done.record(gather_stream)
        if rec is not None:
            k1_ms.append(rec[0].elapsed_time(rec[1]))
            k2_ms.append(rec[2].elapsed_time(rec[3]))

    def run_pipelined(n_steps, record):
        pend = []
        for i in range(n_steps):
            sl = slots[i % n_slots]
            if sl.k2_done is not None:
                s_k1.wait_event(sl.k2_done)              # this slot's workspace: the pursuit of step i-2 is done
            if getattr(sl, 'gather_done', None) is not None:
                s_k1.wait_event(sl.gather_done)          # ... and its codes have been gathered
            rec = [torch.cuda.Event(enable_timing=True) for _ in range(4)] if record else None
            if rec:
                rec[0].record(s_k1)
            with torch.cuda.stream(s_k1):
                sl.begin(xd, opt, s_k1)
            k1_done = rec[1] if rec else torch.cuda.Event()
            k1_done.record(s_k1)
            st2 = s_k2[i % n_slots]
            st2.wait_event(k1_done)
            if rec:
                rec[2].record(st2)
            with torch.cuda.stream(st2):
                sl.run(st2)
            sl.k2_done = rec[3] if rec else torch.cuda.Event()
            sl.k2_done.record(st2)
            pend.append((i, rec))
            if len(pend) >= n_slots:             # the host reads step i's states once n_slots - 1 later steps are enqueued
                finalize(*pend.pop(0))
        while pend:
            finalize(*pend.pop(0))
        for st_ in [s_k1] + s_k2 + ([gather_stream] if gather_stream is not None else []):
            stream.wait_stream(st_)

    def launches_now():
        return eng.launches + (sum(sl.launches() for sl in slots) if slots else 0)

    if args.pipeline:
        s_k1.wait_stream(stream)
        run_pipelined(args.warmup, False)
    else:
        for _ in range(args.warmup):
            step_resident(False)
    sampler = ClockSampler(local_rank)
    launches0 = launches_now()
    barrier()
    sampler.start()
    t_start = torch.cuda.Event(enable_timing=True)
    t_end = torch.cuda.Event(enable_timing=True)
    t_start.record(stream)
    if args.pipeline:
        s_k1.wait_stream(stream)
        run_pipelined(args.steps, True)
    else:
        for _ in range(args.steps):
            step_resident(True)
        if gather_stream is not None:
            stream.wait_stream(gather_stream)           # the last step's gather is inside the timed region
    t_end.record(stream)
    barrier()
    clocks = sampler.stop()
    launches = launches_now() - launches0
    total_ms = t_start.elapsed_time(t_end)
    if args.dump_outputs and rank == 0:
        if args.pipeline:
            sl = slots[(args.steps - 1) % n_slots]
            dump_outputs(args.dump_outputs, sl.compact(None, stream), sl.resid, sl.states)
        else:
            es = last_step['es']
            dump_outputs(args.dump_outputs, eng.compact_events(es['evp'], es['evi'], es['evc']), resid, last_step['states'])
    # stand-alone durations of the two kernels (outside the timed region): inside the pipeline a launch shares the GPU with
    # the tail of the previous pursuit and with the next correlation, so its event-to-event time is not its own cost
    solo_k1, solo_k2 = [], []
    if args.pipeline:
        for _ in range(args.steps):
            es = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            es[0].record(stream)
            slots[0].begin(xd, opt, stream)
            es[1].record(stream)
            slots[0].run(stream)
            es[2].record(stream)
            torch.cuda.synchronize(dev)
            solo_k1.append(es[0].elapsed_time(es[1]))
            solo_k2.append(es[1].elapsed_time(es[2]))
    slots = None                                   # the resident pipeline's workspaces make room for the host pipeline's
    pipe_compact = None
    torch.cuda.empty_cache()

    # ---- end-to-end step through the public API: pinned host -> device, encode, codes (-> rank 0) -> host
    res_pins = [torch.empty_like(x_pin).pin_memory(), torch.empty_like(x_pin).pin_memory()]

    def run_e2e(n_steps, want_residual):
        """n_steps batches through the public host API, pipelined: pinned host signals -> chunked H2D under K1 -> K2 ->
        compaction of the codes on the device -> device-to-host read of exactly the atoms (N = 1), or NCCL gather of the
        device-resident codes to rank 0, which reads them (N > 1).  want_residual adds the copy of the residuals (as large
        as the input) back to pinned host memory."""
        atoms, d2h = 0, 0
        outs = [res_pins[i & 1] for i in range(n_steps)] if want_residual else None
        hook = None
        if world > 1:
            def hook(bi, dev_codes):
                return hd.gather_device_events(dev_codes, dst=0, host_out=(rank == 0))
        for r in eng.encode_host_pipelined((x_pin for _ in range(n_steps)), opt, cap, n_chunks=args.chunks, want_residual=want_residual,
                                           residual_outs=outs, host_events=(world == 1), on_device_events=hook):
            n = r.total_events()
            atoms += n
            d2h = int(n * 12 + (S + 1) * 8 + S * 104)           # atoms (pos, idx, coef) + offsets + per-signal states
            if world > 1 and rank == 0:
                d2h = int(sum(len(p) for p in r.gathered['pos']) * 12 + world * (S + 1) * 8 + S * 104)
        return atoms, d2h

    e2e_steps = args.steps
    e2e_runs = {}
    for tag, want_res in (('codes', False), ('codes+residual', True)):
        run_e2e(min(args.warmup, 2), want_res)
        barrier()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        wall0 = time.perf_counter()
        e0.record(stream)
        n_at, d2h = run_e2e(e2e_steps, want_res)
        e1.record(stream)
        barrier()
        e2e_runs[tag] = dict(ms=max(e0.elapsed_time(e1), 1000.0 * (time.perf_counter() - wall0)), atoms=n_at,
                             d2h=d2h + (int(S * T * F * 4) if want_res else 0))
    e2e_ms, e2e_atoms, code_bytes = e2e_runs['codes']['ms'], e2e_runs['codes']['atoms'], e2e_runs['codes']['d2h']

    # ---- optional: the dictionary-learning loop that consumes the codes (BASELINE config 5), rank 0 only
    ksvd_extra = None
    if args.ksvd_iters > 0 and rank == 0:
        rs = np.random.RandomState(7)
        D0 = D.astype(np.float64) + 0.3 * rs.randn(*D.shape) / math.sqrt(D.shape[1] * D.shape[2])
        D0 /= np.sqrt(np.sum(D0 * D0, axis=(1, 2), keepdims=True))
        learner = hsc.ConvolutionalDictionaryLearner(K, L, algorithm='ksvd', device=local_rank)
        t0 = time.perf_counter()
        learner.train(x_host, method='cmp', maxIterations=args.ksvd_iters, toleranceSnr=None, nbNonzeroCoefs=n_atoms,
                      initD=D0, dtype=np.float32)
        torch.cuda.synchronize(dev)
        wall = time.perf_counter() - t0
        ksvd_extra = {'iterations': len(learner.history), 's_per_iteration': wall / max(len(learner.history), 1),
                      'segments': S, 'method': 'cmp, float32 inference + float64 dictionary update on the device',
                      'history': [{k: (round(v, 6) if isinstance(v, float) else v) for k, v in h.items()} for h in learner.history]}

    # ---- the other configurations of BASELINE.json, briefly (N = 1, default workload only): config 5's segments with the
    # dictionary-learning loop that consumes the codes, and the single 1e6-sample sequence of config 2 (latency-bound)
    others = None
    if world == 1 and args.workload == 'c4' and not args.no_extra:
        others = {}
        eng.close()
        torch.cuda.empty_cache()
        for name in ('c5', 'c2'):
            try:
                others[name] = quick_workload(hsc, torch, dev, local_rank, name, args.steps, args.warmup)
            except Exception as e:          # noqa: BLE001  (the headline line must not depend on the extras)
                others[name] = {'error': repr(e)[:300]}

    # ---- max over ranks
    solo = [float(np.mean(solo_k1)) if solo_k1 else float(np.mean(k1_ms)), float(np.mean(solo_k2)) if solo_k2 else float(np.mean(k2_ms))]
    t = torch.tensor([total_ms, e2e_ms, float(np.mean(k1_ms)), float(np.mean(k2_ms)), e2e_runs['codes+residual']['ms'], solo[0], solo[1]],
                     dtype=torch.float64, device=dev)
    a = torch.tensor([float(atoms_step), float(e2e_atoms), float(e2e_runs['codes+residual']['atoms'])], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(a, op=dist.ReduceOp.SUM)
    total_ms, e2e_ms, k1, k2, e2e_res_ms, k1_solo, k2_solo = [float(v) for v in t.cpu()]
    atoms_all, e2e_atoms_all, e2e_res_atoms_all = [float(v) for v in a.cpu()]

    if rank == 0:
        peaks = load_peaks()
        value = atoms_all * args.steps / (total_ms / 1e3)
        ms_per_step = total_ms / args.steps
        atoms_rank = atoms_all / world
        k2_bytes = atoms_rank * per_atom_bytes(w)
        k2_gbs = k2_bytes / (k2 / 1e3) / 1e9
        k1_tflops = correlation_flops(w) / (k1 / 1e3) / 1e12
        k1_gbs = correlation_bytes(w) / (k1 / 1e3) / 1e9
        # K1 operand format: 3xFP16 on tcgen05 kind::f16 (peak = the measured bf16/fp16 dense rate) unless HSC_K1=tf32
        k1_mode = os.environ.get('HSC_K1', 'f16')
        if k1_mode == 'tf32':
            k1_peak, k1_peak_src, k1_name = peaks['bf16'] / 2.0, ' bf16 burst / 2 (tf32 dense rate)', '3xTF32'
            kd_pad = 1.0
        else:
            k1_peak, k1_peak_src, k1_name = peaks['bf16'], ' bf16 burst (= fp16 dense rate)', '3xFP16'
            s_rows = max(1, 8 // F)
            kd_pad = (((L + s_rows - 1) * F + 15) // 16 * 16) / float(L * F)      # padded reduction length / L*F
        roof_k2 = {'kernel': 'pursuit_kernel (K2 select/update)', 'bound': 'hbm', 'achieved': k2_gbs, 'peak': peaks['hbm'], 'unit': 'GB/s',
                   'frac': k2_gbs / peaks['hbm'], 'traffic': None, 'ms_per_launch': k2,
                   'algorithmic_bytes_per_launch': k2_bytes, 'peak_source': peaks['source']}
        roof_k1 = {'kernel': 'correlate_tc_kernel (K1 initial correlation: tcgen05 %s implicit GEMM + split/unpack helpers)' % k1_name, 'bound': 'tensor',
                   'achieved': k1_tflops, 'peak': k1_peak,
                   'unit': 'TFLOP/s', 'frac': k1_tflops / k1_peak, 'traffic': None, 'ms_per_launch': k1,
                   'algorithmic_flops_per_launch': correlation_flops(w), 'issued_tflops': 3.0 * kd_pad * k1_tflops,
                   'issued_frac': 3.0 * kd_pad * k1_tflops / k1_peak, 'hbm_gbs': k1_gbs,
                   'note': 'achieved/frac count the useful single-pass flops 2*S*T*K*L*F; the three-product operand split issues 3x that (issued_*)',
                   'peak_source': peaks['source'] + k1_peak_src}
        # Inside the streaming pipeline a launch's event-to-event time includes the time it QUEUES behind the tail of the
        # previous pursuit and shares SMs with the next correlation; the roofline describes the kernel, so it is computed from
        # the kernel launched ALONE (same data, CUDA events on its stream, right after the timed region), which is also what the
        # serialised ncu launch list shows.  The in-pipeline times stay in pipelined_ms_per_launch / pipelined_frac.
        if args.pipeline:
            for rk, solo_ms, work in ((roof_k1, k1_solo, correlation_flops(w) / 1e12), (roof_k2, k2_solo, k2_bytes / 1e9)):
                rk['pipelined_ms_per_launch'] = rk['ms_per_launch']
                rk['pipelined_frac'] = rk['frac']
                rk['ms_per_launch'] = solo_ms
                rk['achieved'] = work / (solo_ms / 1e3)
                rk['frac'] = rk['achieved'] / rk['peak']
                rk['measured'] = ('stand-alone launch, CUDA events on its stream, right after the timed region (mean of %d); inside the '
                                  'streaming pipeline the same launch takes pipelined_ms_per_launch because it shares the GPU with the '
                                  'previous pursuit\'s tail and the next correlation' % args.steps)
            roof_k1['issued_tflops'] = 3.0 * kd_pad * roof_k1['achieved']
            roof_k1['issued_frac'] = roof_k1['issued_tflops'] / k1_peak
            roof_k1['hbm_gbs'] = correlation_bytes(w) / (k1_solo / 1e3) / 1e9
            k1, k2 = k1_solo, k2_solo           # the dominant kernel is chosen on its own duration
        step_bytes = k2_bytes + correlation_bytes(w)
        step_hbm = {'algorithmic_bytes_per_step': step_bytes, 'achieved': step_bytes / (ms_per_step / 1e3) / 1e9, 'unit': 'GB/s',
                    'frac': step_bytes / (ms_per_step / 1e3) / 1e9 / peaks['hbm'],
                    'note': 'K1 map write + signal read and K2 window / Gram / residual bytes of one step over ms_per_step (both kernels share HBM in the pipeline)'}
        tr = load_traffic(args.workload)
        if tr:
            roof_k1['traffic'] = tr['k1_dram_bytes_per_signal'] * S if tr.get('k1_dram_bytes_per_signal') else None
            roof_k2['traffic'] = tr['k2_dram_bytes_per_atom'] * atoms_rank if tr.get('k2_dram_bytes_per_atom') else None
            roof_k1['traffic_source'] = roof_k2['traffic_source'] = tr['source']
        dominant = roof_k2 if k2 >= k1 else roof_k1
        line = {
            'metric': 'mp_atoms_per_s', 'value': value, 'unit': 'atoms/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
            'data': 'synthetic',
            'config': workload_config(w),
            'run': {'stops': stop_hist, 'selections_per_signal': atoms_rank / S, 'coef_mode': args.coef_mode, 'world_size': world,
                    'mode': ('streaming pipeline: K1 of step i+1 on its own stream under K2 of step i, K2 launches on alternating streams '
                             '(kernel durations below are per-launch CUDA-event times inside the pipeline and overlap each other)')
                            if args.pipeline else 'one step after the other on one stream',
                    'reranked_selections_per_step': run_info.get('reranked_selections')},
            'samples_per_s': value * T / n_atoms,
            'e2e': {'value': e2e_atoms_all / (e2e_ms / 1e3), 'unit': 'atoms/s', 'h2d_bytes_per_step': int(S * T * F * 4),
                    'd2h_bytes_per_step': int(code_bytes), 'steps': e2e_steps, 'chunks': args.chunks,
                    'result': 'sparse codes (position, filter, coefficient per atom), compacted on the device; N > 1: NCCL gather to rank 0, which reads them',
                    'api': 'Engine.encode_host_pipelined (copies out of step i overlap H2D + K1 of step i+1; wall clock over all steps)',
                    'with_residual': {'value': e2e_res_atoms_all / (e2e_res_ms / 1e3), 'unit': 'atoms/s',
                                      'd2h_bytes_per_step': int(e2e_runs['codes+residual']['d2h']),
                                      'note': 'same call with want_residual=True: the residual signals (as large as the input) also return to pinned host memory'}},
            'gpu_launches': int(launches),
            'clocks': clocks,
            'roofline': dominant,
            'kernels': {'k1_ms': roof_k1.get('pipelined_ms_per_launch', k1), 'k2_ms': roof_k2.get('pipelined_ms_per_launch', k2),
                        'k1_solo_ms': k1_solo, 'k2_solo_ms': k2_solo, 'k1': roof_k1, 'k2': roof_k2, 'step_hbm': step_hbm,
                        'us_per_atom_per_signal': 1e3 * k2_solo / (atoms_rank / S)},
        }
        if args.ksvd_iters > 0:
            line['extra'] = {'ksvd': ksvd_extra}
        if others:
            line.setdefault('extra', {})['other_configs'] = others
        if not args.no_cpu_baseline and world == 1:
            line['cpu_baseline'] = cpu_baseline_sample(w, D)
        else:
            line['cpu_baseline'] = None
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='c4', choices=sorted(WORKLOADS))
    ap.add_argument('--signals', type=int, default=None, help='override signals per GPU')
    ap.add_argument('--coef-mode', type=int, default=1)
    ap.add_argument('--chunks', type=int, default=8, help='chunks of the host pipeline (e2e)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extra', action='store_true', help='skip the brief config-5 / config-2 measurements appended under extra.other_configs')
    ap.add_argument('--rerank-tol', type=float, default=-1.0, help='near-tie re-ranking window (hsc_mp_options.rerank_tolerance); < 0 = default, 0 = off')
    ap.add_argument('--k1-priority', type=int, default=1, help='pipeline: run the correlation on a high-priority stream')
    ap.add_argument('--slots', type=int, default=2, help='pipeline: encode slots (workspaces) in flight')
    ap.add_argument('--pipeline', type=int, default=1, help='1: steps run as a streaming pipeline on several CUDA streams (default); 0: one step after the other')
    ap.add_argument('--ksvd-iters', type=int, default=0, help='also time N K-SVD iterations (encode + dictionary update) on the workload')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last one returned (sparse codes, residual energies, a seeded sample '
                         'of residual signals) as .npy files under DIR, at most 64 MB; with several GPUs, the shard of rank 0')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be >= 1 and --warmup >= 0')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes what the GPU path computed; it has no meaning with --impl reference')
    w = dict(WORKLOADS[args.workload])
    if args.signals:
        w['S'] = args.signals
    if args.impl == 'reference':
        run_reference_arm(args, w)
    else:
        run_b200_arm(args, w)


if __name__ == '__main__':
    main()
