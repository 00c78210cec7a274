"""Throughput of batched hierarchical encoding (HierarchicalConvolutionalSparseCoder.encodeBatch and encodeBatchDevice)
against a loop of encode, on the config-3 workload: the 3-level dictionary and test signal of tests/golden/c3_complex.npz,
plus B - 1 copies of the signal rolled by seeded offsets.

    python tools/hier_batch_c3.py --out-dir DIR [--batches 1,16,148,592] [--repeats 3]

For every scripted setting (cmp / 10 blocks, cmp / 1 block, locomp / 10 blocks) and batch size B, after one warm-up call of
every shape, it times encodeBatch and encodeBatchDevice, alternating them, and splits encodeBatch into
  forward_ms   the level loop on the device: every chunk's launches up to its one synchronise and the read of its events
               (CUDA events around HierarchicalConvolutionalMatchingPursuit._forward_chunk; host clock alongside),
               including a first attempt that filled its LoCOMP event buffers (chunk_reruns counts them),
  assembly_ms  host code assembly: the per-(signal, level) csc matrices and the per-signal distributed conversion,
  residual_ms  the batched decoder, the subtraction and the read of the residuals,
and encodeBatchDevice (codes and residual left on the GPU, the call ends with a device synchronise) into
  device_forward_ms          the same level loop without the canonical-code kernels (CUDA events),
  device_canon_residual_ms   the canonical-code kernels (CUDA events around Engine.canonicalize_codes) plus everything
                             after the level loop: concatenation of the chunks, the decoder launches and the subtraction,
then times a loop of encode over min(B, --loop-max) of the same signals.  Signals/s of each, and the ratios, per row.
Prints the GPU name and power limit (read-only nvidia-smi query) and writes one JSON line to DIR/hier_batch_c3.jsonl."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SETTINGS = (('cmp_b10', 'cmp', 10), ('cmp_b1', 'cmp', 1), ('locomp_b10', 'locomp', 10))


def gpu_info():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=60).stdout.strip()
    except Exception as e:          # noqa: BLE001
        q = 'nvidia-smi unavailable: %s' % (e,)
    return q.splitlines()[0] if q else q


class Timers(object):
    """Wraps the phases of one approximator: forward (device level loop), residual, distributed conversion, and the
    canonical-code kernels of the device path; the rest of a call is host assembly (encodeBatch) or the device
    concatenation and residual (encodeBatchDevice)."""

    def __init__(self, approx, engine_cls):
        import torch
        self.torch = torch
        self.reset()
        cls = type(approx)
        fwd, res, post = cls._forward_chunk, cls._calculateResidualBatch, cls._postprocessCoefficients
        canon = getattr(engine_cls, '_untimed_canonicalize_codes', engine_cls.canonicalize_codes)
        engine_cls._untimed_canonicalize_codes = canon
        me = self

        def forward_chunk(self_, *a, **kw):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            try:
                out = fwd(self_, *a, **kw)
                me.reruns += out is None         # a chunk that filled its LoCOMP event buffers: counted, then rerun
                return out
            finally:
                e1.record()
                e1.synchronize()
                me.forward_host += time.perf_counter() - t0
                me.forward_dev += e0.elapsed_time(e1) / 1e3

        def residual(self_, *a, **kw):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = res(self_, *a, **kw)
            torch.cuda.synchronize()
            me.residual += time.perf_counter() - t0
            return out

        def postprocess(self_, *a, **kw):
            t0 = time.perf_counter()
            out = post(self_, *a, **kw)
            me.post += time.perf_counter() - t0
            return out

        def canonicalize(self_, *a, **kw):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = canon(self_, *a, **kw)
            e1.record()
            me.canon_events.append((e0, e1))     # read after the chunk's synchronise
            return out

        approx._forward_chunk = forward_chunk.__get__(approx)
        approx._calculateResidualBatch = residual.__get__(approx)
        approx._postprocessCoefficients = postprocess.__get__(approx)
        engine_cls.canonicalize_codes = canonicalize

    def canon_dev(self):
        return sum(a.elapsed_time(b) for a, b in self.canon_events) / 1e3

    def reset(self):
        self.forward_host = self.forward_dev = self.residual = self.post = 0.0
        self.reruns = 0
        self.canon_events = []


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--out-dir', required=True)
    ap.add_argument('--batches', default='1,16,148,592')
    ap.add_argument('--repeats', type=int, default=3)
    ap.add_argument('--loop-max', type=int, default=148, help='signals in the timed encode loop (its rate is per signal)')
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), 'this measurement needs a CUDA device'
    import hierarchical_sparse_coding_b200 as hsc
    gpu = gpu_info()
    print('GPU:', torch.cuda.get_device_name(0), '|', gpu, flush=True)
    z = np.load(os.path.join(ROOT, 'tests', 'golden', 'c3_complex.npz'))
    nl = int(z['nb_levels'])
    mld = hsc.MultilevelDictionary([z['raw_l%d' % i] for i in range(nl)], [int(v) for v in z['scales']],
                                   [z['rep_l%d' % i] for i in range(nl)], z['counts_no_singletons'], hasSingletonBases=True)
    x = z['x']
    batches = [int(b) for b in args.batches.split(',')]
    rs = np.random.RandomState(0)
    X = np.stack([x] + [np.roll(x, int(o)) for o in rs.randint(1, len(x), max(batches) - 1)])
    rows = []
    for tag, method, nb in SETTINGS:
        approx = hsc.HierarchicalConvolutionalMatchingPursuit(method=method)
        coder = hsc.HierarchicalConvolutionalSparseCoder(mld, approx)
        tm = Timers(approx, hsc.Engine)
        kw = dict(toleranceSnr=10.0, nbBlocks=nb, singletonWeight=0.95)
        coder.encode(X[0], **kw)                                         # warm-up: single shape
        for B in batches:
            coder.encodeBatch(X[:B], **kw)                               # warm-up: this batch shape, both paths
            coder.encodeBatchDevice(X[:B], **kw)
            torch.cuda.synchronize()
            host = dict(t=0.0, f_dev=0.0, f_host=0.0, resid=0.0, post=0.0, reruns=0)
            dev = dict(t=0.0, f_dev=0.0, f_host=0.0, canon=0.0, reruns=0)
            for _ in range(args.repeats):                                # alternating: host path, then device path
                tm.reset()
                t0 = time.perf_counter()
                codes, res = coder.encodeBatch(X[:B], **kw)
                torch.cuda.synchronize()
                host['t'] += time.perf_counter() - t0
                host['f_dev'] += tm.forward_dev
                host['f_host'] += tm.forward_host
                host['resid'] += tm.residual
                host['post'] += tm.post
                host['reruns'] += tm.reruns
                tm.reset()
                t0 = time.perf_counter()
                dcodes, dres = coder.encodeBatchDevice(X[:B], **kw)
                torch.cuda.synchronize()
                dev['t'] += time.perf_counter() - t0
                dev['f_dev'] += tm.forward_dev
                dev['f_host'] += tm.forward_host
                dev['canon'] += tm.canon_dev()
                dev['reruns'] += tm.reruns
            r = float(args.repeats)
            t_batch, f_dev, f_host, resid, post = host['t'] / r, host['f_dev'] / r, host['f_host'] / r, host['resid'] / r, host['post'] / r
            t_dev, canon = dev['t'] / r, dev['canon'] / r
            d_forward = dev['f_dev'] / r - canon
            d_canon_resid = canon + (t_dev - dev['f_host'] / r)
            n_loop = min(B, args.loop_max)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for b in range(n_loop):
                coder.encode(X[b], **kw)
            torch.cuda.synchronize()
            t_loop = (time.perf_counter() - t0) / n_loop
            row = dict(setting=tag, B=B, batch_s=t_batch, forward_ms=1e3 * f_dev, forward_host_ms=1e3 * f_host,
                       assembly_ms=1e3 * (t_batch - f_host - resid), distributed_ms=1e3 * post, residual_ms=1e3 * resid,
                       batch_signals_per_s=B / t_batch, device_batch_s=t_dev, device_forward_ms=1e3 * d_forward,
                       device_canon_ms=1e3 * canon, device_canon_residual_ms=1e3 * d_canon_resid,
                       device_batch_signals_per_s=B / t_dev, device_vs_batch=t_batch / t_dev,
                       loop_signals=n_loop, loop_s_per_signal=t_loop, loop_signals_per_s=1.0 / t_loop,
                       speedup=(B / t_batch) * t_loop, device_speedup=(B / t_dev) * t_loop,
                       chunk_reruns=host['reruns'] / r, device_chunk_reruns=dev['reruns'] / r,
                       nnz_member0=[c.nnz for c in codes[0]],
                       device_nnz_member0=[int(o[1] - o[0]) for o in dcodes.offsets])
            rows.append(row)
            print('%-10s B=%4d  encodeBatch %8.1f ms (%8.1f signals/s): forward %7.1f ms device, assembly %7.1f ms (distributed %6.1f), '
                  'residual %6.1f ms | encodeBatchDevice %8.1f ms (%8.1f signals/s): forward %7.1f ms device, canonicalize+residual '
                  '%6.1f ms (kernels %5.2f ms) | encode loop %7.2f ms/signal (%7.1f signals/s)'
                  % (tag, B, 1e3 * t_batch, B / t_batch, row['forward_ms'], row['assembly_ms'], row['distributed_ms'],
                     row['residual_ms'], 1e3 * t_dev, B / t_dev, row['device_forward_ms'], row['device_canon_residual_ms'],
                     row['device_canon_ms'], 1e3 * t_loop, 1.0 / t_loop), flush=True)
    out = dict(metric='hier_batch_c3', gpu=torch.cuda.get_device_name(0), nvidia_smi=gpu, T=int(len(x)),
               repeats=args.repeats, rows=rows)
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, 'hier_batch_c3.jsonl'), 'a') as f:
        f.write(json.dumps(out) + '\n')
    print(json.dumps(out))


if __name__ == '__main__':
    main()
