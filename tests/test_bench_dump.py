"""bench.py --dump-outputs: what the last timed step returned, as float64 .npy files of bounded total size, with the trajectories
of a fixed seeded sample of the OCPs (CPU tensors in the shapes of the quadrotor path stand in for the device arrays)."""
import os

import numpy as np
import torch

import bench


def _step_outputs(B, N=50, n=13, m=4, r=7):
    g = torch.Generator().manual_seed(3)

    def f(*s):
        return torch.randn(*s, generator=g, dtype=torch.float64)

    def i(*s):
        return torch.randint(-5, 50, s, generator=g, dtype=torch.int32)
    sol = dict(X=f(B, N + 1, n), U=f(B, N + 1, m), Lam=f(B, N + 1, n), status=i(B), iters=i(B), kkt=f(B), cost=f(B))
    aux = dict(Xa=f(B, N + 1, n * r), Ua=f(B, N + 1, m * r), loss=f(B), dtheta=f(B, r), aux_status=i(B), counters=i(B, 8))
    return f(r + 2), sol, aux


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def _check(d, red, sol, aux, idx):
    assert all(v.dtype == np.float64 for v in d.values())
    assert np.array_equal(d["reduced"], red.numpy())
    for k in ("status", "iters", "kkt", "cost"):
        assert np.array_equal(d[k], sol[k].numpy()), k
    for k in ("loss", "dtheta", "aux_status", "counters"):
        assert np.array_equal(d[k], aux[k].numpy()), k
    for k in ("X", "U", "Lam"):
        assert np.array_equal(d[k], sol[k].numpy()[idx]), k
    for k in ("Xa", "Ua"):
        assert np.array_equal(d[k], aux[k].numpy()[idx]), k


def test_small_batch_is_dumped_whole(tmp_path):
    red, sol, aux = _step_outputs(8)
    bench.dump_outputs(str(tmp_path), red, sol, aux, first=0)
    d = _load(str(tmp_path))
    assert np.array_equal(d["sample_index"], np.arange(8))
    _check(d, red, sol, aux, np.arange(8))


def test_large_batch_is_sampled_within_the_bound_and_the_same_every_run(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    red, sol, aux = _step_outputs(64)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), red, sol, aux, first=128)
    a, b = _load(str(tmp_path / "a")), _load(str(tmp_path / "b"))
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)
    files = os.listdir(tmp_path / "a")
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= (1 << 20) + 256 * len(files)     # + .npy headers
    idx = a["sample_index"].astype(np.int64) - 128
    assert 0 < len(idx) < 64 and np.all(np.diff(idx) > 0) and idx[-1] < 64
    _check(a, red, sol, aux, idx)
