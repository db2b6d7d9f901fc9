"""The Newton-solve linear algebra of the backward BDF sweep on the B200: the probe kernel (tests/bdf_probe/bdf_probe.cuh)
built with nvcc for sm_100a runs the inputs of tests/test_bdf_linalg.py.  On the device the code differs from the emulation
in bdf_rcp / bdf_rsqrt (approximate seed + two Newton steps), bdf_argmax (__reduce_max_sync on the high word), the shuffle
butterflies, bdf_sweep's stepped addressing and the 128-bit loads, so the device outputs are held to the same bounds as the
emulation's, take the same path (dk, FLAG[1], FLAG[3]) wherever the reference is not within 1e-6 of a threshold, and their
largest difference from the emulation is printed (bit equality is not expected)."""
import numpy as np
import pytest

from tests import bdf_linalg_reference as ref
from tests import test_bdf_linalg as T

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


@pytest.fixture(scope="module", autouse=True)
def _print_ratios(request):
    T.RATIOS.clear()
    yield
    T.report(request.config, "test_bdf_linalg_gpu (B200)")


@pytest.fixture(scope="module")
def probes(torch_mod):
    return T.build_all(device=True), T.build_all(device=False)


def _same_path(dev, emu, idx, L):
    for key in ("dk", "flag1", "flag3", "fok"):
        if dev[key][idx] != emu[key][idx]:
            kv = ref.kappa_v(L)
            assert abs(kv / T.KAPPA - 1.0) <= 1e-6, (key, idx, dev[key][idx], emu[key][idx], kv)


def _diff(dev, emu, idx, n, tag):
    d = np.abs(dev["R"][idx] - emu["R"][idx]).max() / max(np.abs(emu["R"][idx]).max(), 1e-300)
    T.record("device - emulation (rel)", tag, n, d)


@pytest.mark.parametrize("dim", T.DIMS, ids=T.DIM_IDS)
def test_device_schur_eigen_gate_and_newton_solve(probes, dim):
    dev, emu = probes
    n = dim[0]
    fam, recs, rece = T.schur_and_solve(dev[dim][0], dev[dim][1], n)
    Ls = [f[1] for f in fam]
    cs = [T.c_for(L) for L in Ls]
    erec, _ = T.run_cases(emu[dim][0], Ls, cs, seed=n)
    esw, _ = T.run_cases(emu[dim][1], Ls, cs, seed=n)
    for k, L in enumerate(Ls):
        _same_path(rece, erec, (k, 0), L)
        _same_path(recs, esw, (k, 0), L)
        _diff(rece, erec, (k, 0), n, "eig" if erec["flag3"][k, 0] else "sweep")
        _diff(recs, esw, (k, 0), n, "sweep")


@pytest.mark.parametrize("dim", T.DIMS, ids=T.DIM_IDS)
def test_device_singular_operator_and_gauss_jordan(probes, dim):
    dev, emu = probes
    n = dim[0]
    cases = T.singular_cases(n)
    for pd, pe in zip(dev[dim], emu[dim]):
        rd, inp = T.run_cases(pd, [c[0] for c in cases], [c[1] for c in cases], seed=3)
        re_, _ = T.run_cases(pe, [c[0] for c in cases], [c[1] for c in cases], seed=3)
        T.check_singular(rd, inp, cases)
        for k, (L, c, sing) in enumerate(cases):
            if sing is not None:
                assert rd["fok"][k, 0] == re_["fok"][k, 0], c
    rng = np.random.default_rng(90 + n)
    mats = T.gj_matrices(n, rng)
    ok, inv = dev[dim][0].gj(np.stack(mats))
    for k, A in enumerate(mats):
        assert ok[k] == 1 and np.all(np.isfinite(inv[k]))
        r = ref.inv_residual(A, inv[k]) / (n * T.U * np.linalg.cond(A, "fro"))
        T.record("gauss-jordan A A^-1 - I", "-", n, r)
        assert r <= T.C_GJ, (k, r)
    z = np.zeros((1, n, n))
    ok, inv = dev[dim][0].gj(z)
    assert ok[0] == 0 and np.all(inv == 0.0)


@pytest.mark.parametrize("dim", [d for d in T.DIMS if d[0] >= 2], ids=[i for d, i in zip(T.DIMS, T.DIM_IDS) if d[0] >= 2])
def test_device_warm_refinement(probes, dim):
    dev, emu = probes
    n = dim[0]
    seqs = T.warm_sequences(n, np.random.default_rng(300 + n))
    rec2, inp2, rec1 = T.run_warm(dev[dim][0], seqs)
    T.check_warm(rec2, inp2, rec1, n, [s[3] for s in seqs], [s[0] for s in seqs])
    e2, _, _ = T.run_warm(emu[dim][0], seqs)
    assert np.array_equal(rec2["dk"], e2["dk"]) and np.array_equal(rec2["flag3"], e2["flag3"])


def test_device_quadrotor_jacobians(probes):
    dev, _ = probes
    T.test_quadrotor_jacobians({(13, 12): dev[(13, 12)]}, T.quad_jacobians())


def test_device_scale_sweep(probes):
    """Power-of-two scalings on the device: the Schur form scales within rounding (rsqrt / rcp seeds)."""
    dev, _ = probes
    for dim in ((4, 3), (13, 12)):
        n = dim[0]
        L = ref.mixed_spectrum(n, np.random.default_rng(7 + n), 1.0)
        ks = list(range(-40, 41, 20))
        rec, _ = T.run_cases(dev[dim][1], [L * 2.0 ** k for k in ks], [0.1 * 2.0 ** -k for k in ks])
        base = ks.index(0)
        for i, k in enumerate(ks):
            d = np.abs(rec["TD"][i, 0] * 2.0 ** -k - rec["TD"][base, 0]).max() / np.abs(rec["TD"][base, 0]).max()
            T.record("scale sweep TD (rel)", "sweep", n, d)
            assert d <= 64 * n * T.U


def test_device_one_state_model_bdf_matches_oracle(torch_mod):
    """NX = 1 built by nvcc for sm_100a: the BDF sweep on the device against the oracle."""
    _, oc = T.one_state_models()
    oc.build(name="onestate")
    T.one_state_check(oc)
