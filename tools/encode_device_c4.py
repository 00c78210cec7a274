"""Throughput of ConvolutionalSparseCoder.encodeBatchDevice at the config-4 shape (65 536 samples x 4 channels, 256 filters
of 64, nbNonzeroCoefs = 655 = 1 % L0), for batches up to the full 4096-signal config-4 workload on one GPU.

    python tools/encode_device_c4.py --out-dir DIR [--batches 512,1024,2048,4096] [--repeats 2] [--distinct 1024]

Signals: bench.py's generator (make_signals, float32), --distinct of them, tiled up to the largest batch (a signal's
pursuit time does not depend on where it sits in the batch).  For every batch size B, after one warm-up call, it times
encodeBatchDevice from a CUDA tensor, a pinned CPU tensor and a numpy array, alternating them, each call ending in a device
synchronise (host clock), with the residual returned.  At B = --compare-b it also times encodeBatch (numpy in, csc list and
numpy residual out) alternating with the device path.  Atoms/s = selected atoms (the sum of n_events over the signals)
over wall time; entries = distinct code entries returned.  Prints the GPU name and power limit (read-only nvidia-smi
query) and writes one JSON line to DIR/encode_device_c4.jsonl."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=60).stdout.strip()
    except Exception as e:          # noqa: BLE001
        q = 'nvidia-smi unavailable: %s' % (e,)
    return q.splitlines()[0] if q else q


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--out-dir', required=True)
    ap.add_argument('--batches', default='512,1024,2048,4096')
    ap.add_argument('--repeats', type=int, default=2)
    ap.add_argument('--distinct', type=int, default=1024, help='distinct signals generated, tiled up to the largest batch')
    ap.add_argument('--compare-b', type=int, default=512, help='batch size at which encodeBatch is timed too (0: none)')
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), 'this measurement needs a CUDA device'
    import bench
    import hierarchical_sparse_coding_b200 as hsc
    gpu = gpu_info()
    print('GPU:', torch.cuda.get_device_name(0), '|', gpu, flush=True)
    w = dict(bench.WORKLOADS['c4'])
    D = bench.make_dictionary(w)
    batches = [int(b) for b in args.batches.split(',')]
    base = bench.make_signals(w, D, seed=1000, S=min(args.distinct, max(batches)))
    X = np.ascontiguousarray(np.concatenate([base] * (-(-max(batches) // len(base))))[:max(batches)])
    del base
    coder = hsc.ConvolutionalSparseCoder(D, hsc.ConvolutionalMatchingPursuit())
    kw = dict(nbNonzeroCoefs=w['atoms'])
    rows = []
    for B in batches:
        forms = dict(cuda=torch.from_numpy(X[:B]).cuda(), pinned=torch.from_numpy(X[:B]).pin_memory(), numpy=X[:B])
        codes, res = coder.encodeBatchDevice(forms['cuda'], **kw)          # warm-up of this shape
        del codes, res
        torch.cuda.synchronize()
        for rep in range(args.repeats):
            names = list(forms) + (['encodeBatch'] if B == args.compare_b else [])
            for name in names:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                if name == 'encodeBatch':
                    codes, res = coder.encodeBatch(forms['numpy'], **kw)
                    torch.cuda.synchronize()
                    dt = time.perf_counter() - t0
                    events = coder.approximator.last_result.total_events()
                    entries = int(sum(c.nnz for c in codes))
                else:
                    codes, res = coder.encodeBatchDevice(forms[name], **kw)
                    torch.cuda.synchronize()
                    dt = time.perf_counter() - t0
                    events = int(sum(st.n_events for st in codes.states))
                    entries = int(codes.offsets[-1])
                del codes, res
                row = dict(B=B, input=name, repeat=rep, wall_s=dt, events=events, entries=entries, atoms_per_s=events / dt,
                           signals_per_s=B / dt)
                rows.append(row)
                print('B=%4d %-11s rep %d: %8.1f ms  %6.2f M atoms/s  %7.1f signals/s  events %d entries %d'
                      % (B, name, rep, 1e3 * dt, events / dt / 1e6, B / dt, events, entries), flush=True)
        del forms
        torch.cuda.empty_cache()
    out = dict(metric='encode_device_c4', gpu=torch.cuda.get_device_name(0), nvidia_smi=gpu, workload=w, distinct=args.distinct,
               repeats=args.repeats, rows=rows)
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, 'encode_device_c4.jsonl'), 'a') as f:
        f.write(json.dumps(out) + '\n')
    print(json.dumps(out))


if __name__ == '__main__':
    main()
