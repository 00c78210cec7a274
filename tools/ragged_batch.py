"""Ragged batch on the config-4 dictionary (256 filters x 64 x 4 channels, float32): 512 signals whose lengths are drawn,
seeded, from 8 values between 8192 and 65536, encoded to toleranceSnr from a CUDA tensor.  Times, alternated `--rounds`
times with a device synchronisation around each call:

  (a) one ragged ConvolutionalSparseCoder.encodeBatchDevice(X, lengths=...) call;
  (b) the correct alternative without lengths: one encodeBatchDevice call per distinct length;
  (c) the padded tensor encoded as a uniform batch - a cost reference only, its results differ (atoms in the padding).

Prints the card name and power limit, then one JSON line per arm with the median time, sequences/s and atoms/s (atoms:
the selections of every signal, SignalState.n_events).

    python tools/ragged_batch.py [--signals 512] [--rounds 3] [--snr 20] [--out ragged_batch.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def card():
    try:
        return subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                              stdout=subprocess.PIPE, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                  # noqa: BLE001
        return 'unknown (%s)' % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--signals', type=int, default=512)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--snr', type=float, default=20.0)
    ap.add_argument('--seed', type=int, default=7)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()

    import torch
    import bench
    import hierarchical_sparse_coding_b200 as hsc
    assert torch.cuda.is_available(), 'tools/ragged_batch.py measures on the GPU'

    w = dict(bench.WORKLOADS['c4'])
    w['S'] = args.signals
    T = w['T']
    D = bench.make_dictionary(w, seed=42)
    X = bench.make_signals(w, D, seed=43)
    rs = np.random.RandomState(args.seed)
    choices = np.sort(rs.choice(np.arange(8192, T + 1, 1024), 8, replace=False))
    choices[-1] = T
    lengths = rs.choice(choices, args.signals).astype(np.int64)
    Xp = X.copy()
    for b, n in enumerate(lengths):
        Xp[b, n:] = 0.0
    xd = torch.from_numpy(Xp).cuda()
    groups = [(int(n), torch.from_numpy(np.flatnonzero(lengths == n)).cuda()) for n in np.unique(lengths)]
    parts = [(n, xd[ix, :n].contiguous()) for n, ix in groups]
    coder = hsc.ConvolutionalSparseCoder(D, hsc.ConvolutionalMatchingPursuit())
    kw = dict(toleranceSnr=args.snr)

    def arm_a():
        codes, _ = coder.encodeBatchDevice(xd, lengths=lengths, **kw)
        return sum(codes.stats(b)['n_events'] for b in range(codes.B))

    def arm_b():
        n_ev = 0
        for _, xpart in parts:
            codes, _ = coder.encodeBatchDevice(xpart, **kw)
            n_ev += sum(codes.stats(b)['n_events'] for b in range(codes.B))
        return n_ev

    def arm_c():
        codes, _ = coder.encodeBatchDevice(xd, **kw)
        return sum(codes.stats(b)['n_events'] for b in range(codes.B))

    arms = [('a_ragged_one_call', arm_a), ('b_one_call_per_length', arm_b), ('c_padded_uniform', arm_c)]
    for _, f in arms:                       # warm-up: module loads, buffers, pinned staging
        f()
    times = {name: [] for name, _ in arms}
    atoms = {}
    for _ in range(args.rounds):
        for name, f in arms:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            atoms[name] = f()
            torch.cuda.synchronize()
            times[name].append(time.perf_counter() - t0)
    info = dict(card=card(), signals=args.signals, T_max=T, lengths=[int(n) for n in choices],
                samples=int(lengths.sum()), padded_samples=int(args.signals * T), toleranceSnr=args.snr)
    print(json.dumps(info))
    lines = [info]
    for name, _ in arms:
        med = float(np.median(times[name]))
        line = dict(arm=name, seconds=[round(t, 4) for t in times[name]], median_s=round(med, 4),
                    sequences_per_s=round(args.signals / med, 1), atoms=int(atoms[name]),
                    atoms_per_s=round(atoms[name] / med, 1))
        print(json.dumps(line))
        lines.append(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write('\n'.join(json.dumps(l) for l in lines) + '\n')


if __name__ == '__main__':
    main()
