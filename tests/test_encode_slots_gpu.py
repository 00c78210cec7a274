"""The encode slots an Engine keeps between calls: encode_host_pipelined with both slots on one shared workspace, and the
engine's slot, pipeline slots and streams shared by encode, encode_host, encode_host_pipelined and encode_stream_device
without one call's state reaching another's result."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

S, T, F, K, L, ATOMS, CAP = 12, 4096, 4, 64, 32, 30, 256


@pytest.fixture(scope='module')
def hsc():
    import torch
    assert torch.cuda.is_available(), 'gpu tests need a CUDA device'
    import hierarchical_sparse_coding_b200 as pkg
    return pkg


@pytest.fixture(scope='module')
def data():
    """A float32 dictionary and five pinned batches of S signals, each a sum of ATOMS scaled atoms."""
    import torch
    from oracle import hsc_oracle as O
    rs = np.random.RandomState(13)
    D = O.normalize(rs.randn(K, L, F)).astype(np.float32)
    batches = []
    for _ in range(5):
        x = np.zeros((S, T, F), np.float32)
        for s in range(S):
            for p, k, a in zip(rs.randint(0, T - L, ATOMS), rs.randint(0, K, ATOMS), rs.uniform(0.25, 4.0, ATOMS)):
                x[s, p:p + L] += np.float32(a) * D[k]
        batches.append(torch.from_numpy(x).pin_memory())
    return D, batches


def _engine(hsc, D):
    eng = hsc.Engine(0)
    eng.set_dictionary(D)
    return eng


def _same_result(a, b):
    import torch
    assert a.S == b.S and (a.residual is None) == (b.residual is None)
    for s in range(a.S):
        assert np.array_equal(a.pos[s], b.pos[s]) and np.array_equal(a.idx[s], b.idx[s]), s
        assert np.array_equal(a.coef[s].view(np.int32), b.coef[s].view(np.int32)), s
    assert [bytes(st) for st in a.states] == [bytes(st) for st in b.states]
    if a.residual is not None:
        assert torch.equal(a.residual, b.residual)


@pytest.mark.gpu
def test_pipeline_with_one_shared_workspace_equals_encode_host(hsc, data, monkeypatch):
    """No room for a second workspace: both pipeline slots share one, on the engine's own handle, and every batch is
    still exactly what encode_host returns, with and without the residual."""
    D, batches = data
    eng = _engine(hsc, D)
    opt = eng.make_options(nbNonzeroCoefs=ATOMS)
    refs = [eng.encode_host(b, opt, capacity=CAP, n_chunks=3) for b in batches]
    for r in refs:
        r.residual = r.residual.clone()
    monkeypatch.setattr(eng, '_free_device_bytes', lambda: 0)
    for want_residual in (True, False):
        got = list(eng.encode_host_pipelined(batches, opt, capacity=CAP, n_chunks=3, want_residual=want_residual))
        slots = next(iter(eng._pipe_slots.values()))
        assert slots[0].ws is slots[1].ws and slots[0].handle is slots[1].handle is eng.handle
        assert [g.batch_index for g in got] == list(range(len(batches)))
        for r, g in zip(refs, got):
            if not want_residual:
                assert g.residual is None
                g.residual = r.residual
            _same_result(r, g)
            assert np.array_equal(g.counts, [len(p) for p in r.pos])
    eng.close()


@pytest.mark.gpu
def test_calls_sharing_an_engine_equal_calls_on_fresh_engines(hsc, data):
    """One engine runs encode, encode_host, an abandoned encode_host_pipelined, encode_stream_device and a full pipeline,
    interleaved and at shapes that share the engine's cached slot; every result is bit for bit that of the same call on a
    fresh engine."""
    import torch
    D, batches = data
    shared = _engine(hsc, D)
    opt = shared.make_options(nbNonzeroCoefs=ATOMS)
    x0 = batches[0].numpy()
    calls = [
        ('encode', lambda e: e.encode(x0, opt, capacity=CAP)),
        ('encode_host', lambda e: e.encode_host(batches[1], opt, capacity=CAP, n_chunks=3)),
        ('abandoned pipeline', lambda e: [next(iter(e.encode_host_pipelined(batches[:4], opt, capacity=CAP, want_residual=True)))]),
        ('encode, paused', lambda e: e.encode(batches[2], opt, capacity=7)),
        ('encode_stream_device', lambda e: e.encode_stream_device(batches[3], opt, capacity=CAP)),
        ('encode_host, fewer signals', lambda e: e.encode_host(batches[4][:5], opt, capacity=CAP, n_chunks=2)),
        ('pipeline', lambda e: list(e.encode_host_pipelined(batches, opt, capacity=CAP, n_chunks=2, want_residual=True))),
        ('encode_host', lambda e: e.encode_host(batches[0], opt, capacity=CAP, n_chunks=4)),
        ('encode, residual in place', lambda e: e.encode(batches[1].cuda(), opt, capacity=CAP, residual_inplace=True)),
    ]
    for name, call in calls:
        got = call(shared)
        fresh = _engine(hsc, D)
        ref = call(fresh)
        torch.cuda.synchronize()
        if name == 'encode_stream_device':
            for a, b in zip(got[:4] + got[5:], ref[:4] + ref[5:]):
                assert torch.equal(a, b), name
            assert [bytes(st) for st in got[4]] == [bytes(st) for st in ref[4]], name
        else:
            got, ref = (r if isinstance(r, list) else [r] for r in (got, ref))
            assert len(got) == len(ref), name
            for a, b in zip(got, ref):
                _same_result(a, b)
        fresh.close()
    shared.close()
