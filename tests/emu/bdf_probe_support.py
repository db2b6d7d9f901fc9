"""Builds and runs the probe of the BDF sweep's Newton-solve linear algebra (tests/bdf_probe/bdf_probe.cuh) for a synthetic
linear-quadratic model with NX = n states and NP = r parameters: the thread emulation (g++, tests/emu/emu_bdf_probe.cpp) and
the device build (nvcc for sm_100a, tests/bdf_probe/bdf_probe.cu).  Libraries are cached by content hash in tests/emu/_build.
TEST INFRASTRUCTURE — the product never imports this."""
import ctypes
import hashlib
import os
import subprocess

import numpy as np

import lfsd_b200  # noqa: F401
from lfsd_b200 import _capi, codegen
from lfsd_b200.sx import SX, vertcat
from tests.emu.build_emu import CSRC
from tests.emu.support import _BUILD

_HERE = os.path.dirname(os.path.abspath(__file__))
_PROBE = os.path.join(os.path.dirname(_HERE), "bdf_probe")
_BDF_SOURCES = ("cpdp_port.h", "cpdp_kernels.cuh", "cpdp_aux.cuh", "cpdp_bdf.cuh")
LAYOUT_KEYS = ("NX", "NP", "NC", "QS", "TW", "IN_STEP", "OUT_STEP", "SMEM_BYTES", "OUT_Q", "OUT_QT", "OUT_TD", "OUT_ROT",
               "OUT_T2S", "OUT_WT", "OUT_R", "OUT_PV", "EIG", "WARM")


def lq_model_header(n, r):
    """Model header of x' = A x + b u with a path cost weighted by the r parameters (only the layout constants matter)."""
    x, u, th = SX.sym('x', n), SX.sym('u', 1), SX.sym('th', r)
    A = np.random.default_rng(n).normal(size=(n, n)) * 0.5
    dyn = vertcat(*[sum(float(A[i, j]) * x[j] for j in range(n)) + (u[0] if i == n - 1 else 0) for i in range(n)])
    pc = sum(th[k] * x[k % n] * x[k % n] for k in range(r)) + 0.1 * u[0] * u[0]
    fc = sum(x[i] * x[i] for i in range(n))
    text, _ = codegen.generate_model_header("lq%d_%d" % (n, r), x, u, th, dyn, pc, fc)
    return text


def _sources():
    src = "".join(open(os.path.join(CSRC, fn)).read() for fn in _BDF_SOURCES)
    for fn in ("bdf_probe.cuh", "bdf_probe_api.inl", "bdf_probe.cu"):
        src += open(os.path.join(_PROBE, fn)).read()
    return src + open(os.path.join(_HERE, "emu_bdf_probe.cpp")).read()


def build_probe(n, r, device=False, flags=()):
    """Path of the probe library for the LQ model (n, r); `flags` are extra -D options of the kernel (mutant builds)."""
    text = lq_model_header(n, r)
    kind = "dev" if device else "emu"
    cmd_flags = " ".join(_capi.NVCC_FLAGS) if device else ""
    tag = hashlib.sha1((text + _sources() + kind + cmd_flags + " ".join(flags)).encode()).hexdigest()[:12]
    os.makedirs(_BUILD, exist_ok=True)
    so = os.path.join(_BUILD, "libbdfprobe_%s_%d_%d_%s.so" % (kind, n, r, tag))
    if os.path.exists(so):
        return so
    hdr = os.path.join(_BUILD, "model_lq%d_%d_%s.cuh" % (n, r, tag))
    with open(hdr, "w") as f:
        f.write(text)
    tmp = "%s.tmp%d" % (so, os.getpid())
    ns = "cpdp_probe_%s_%d_%d" % (kind, n, r)
    if device:
        nvcc = "/usr/local/cuda/bin/nvcc" if os.path.exists("/usr/local/cuda/bin/nvcc") else "nvcc"
        cmd = [nvcc] + _capi.NVCC_FLAGS + ["-I", CSRC, "-I", _PROBE, "-DCPDP_NS=%s" % ns, "-DCPDP_MODEL_HEADER=\"%s\"" % hdr]
        cmd += list(flags) + [os.path.join(_PROBE, "bdf_probe.cu"), "-o", tmp]
    else:
        cmd = ["g++", "-std=c++20", "-O2", "-fPIC", "-shared", "-pthread", "-fvisibility=hidden", "-fno-gnu-unique",
               "-DCPDP_NS=%s" % ns, "-I", CSRC, "-I", _PROBE, "-DCPDP_MODEL_HEADER_PORT=\"cpdp_port.h\"",
               "-DCPDP_MODEL_HEADER=\"%s\"" % hdr] + list(flags) + [os.path.join(_HERE, "emu_bdf_probe.cpp"), "-o", tmp]
    subprocess.check_call(cmd)
    os.replace(tmp, so)
    return so


class Probe:
    """One loaded probe library.  run(L, C, c, B) takes arrays with a leading (cases, steps) shape and returns per-step
    records as a dict of arrays; gj(A) inverts a stack of matrices with bdf_gauss_jordan."""

    def __init__(self, so, device=False):
        self.lib = ctypes.CDLL(so)
        self.device = device
        v = (ctypes.c_int * len(LAYOUT_KEYS))()
        self.lib.bdf_probe_layout(v)
        self.lay = dict(zip(LAYOUT_KEYS, list(v)))
        self.lib.bdf_probe_kappa.restype = ctypes.c_double
        self.kappa = self.lib.bdf_probe_kappa()
        for fn in (self.lib.bdf_probe_run, self.lib.bdf_probe_gj):
            fn.restype = ctypes.c_int
        self.lib.bdf_probe_run.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
        self.lib.bdf_probe_gj.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
        self.n, self.np_, self.nc = self.lay["NX"], self.lay["NP"], self.lay["NC"]

    def _call(self, fn, inp, out_size, *args):
        inp = np.ascontiguousarray(inp, dtype=np.float64)
        if not self.device:
            out = np.zeros(out_size)
            rc = fn(inp.ctypes.data, out.ctypes.data, *args, None)
            assert rc == 0, rc
            return out
        import torch
        ti = torch.from_numpy(inp).cuda()
        to = torch.zeros(out_size, dtype=torch.float64, device="cuda")
        rc = fn(ti.data_ptr(), to.data_ptr(), *args, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0, rc
        torch.cuda.synchronize()
        return to.cpu().numpy()

    def run(self, L, C, c, B):
        lay, n, nc = self.lay, self.n, self.nc
        L = np.asarray(L, dtype=np.float64)
        cases, S = L.shape[:2]
        inp = np.zeros((cases, S, lay["IN_STEP"]))
        inp[:, :, :n * n] = L.reshape(cases, S, n * n)
        inp[:, :, n * n:n * n + n * self.np_] = np.asarray(C, dtype=np.float64).reshape(cases, S, -1)
        inp[:, :, n * n + n * self.np_] = np.asarray(c, dtype=np.float64).reshape(cases, S)
        inp[:, :, n * n + n * self.np_ + 1:] = np.asarray(B, dtype=np.float64).reshape(cases, S, -1)
        o = self._call(self.lib.bdf_probe_run, inp, cases * S * lay["OUT_STEP"], cases, S).reshape(cases, S, lay["OUT_STEP"])
        tw = lay["TW"]
        sl = lambda k, size: o[:, :, lay[k]:lay[k] + size]  # noqa: E731
        return {
            "dk": o[:, :, 0].astype(int), "flag1": o[:, :, 1].astype(int), "flag3": o[:, :, 2].astype(int),
            "fok": o[:, :, 3].astype(int),
            "Q": sl("OUT_Q", n * n).reshape(cases, S, n, n),          # Q slot, [k][i]
            "QT": sl("OUT_QT", n * n).reshape(cases, S, n, n),        # QT slot, [k][i]
            "TD": sl("OUT_TD", 2 * n).reshape(cases, S, n, 2),
            "ROT": sl("OUT_ROT", 4 * n).reshape(cases, S, 4, n),
            "T2S": sl("OUT_T2S", 2 * n * tw).reshape(cases, S, n, tw, 2),
            "PV": sl("OUT_PV", 2 * n * n).reshape(cases, S, 2, n, n),   # Tr | Ti
            "WT": sl("OUT_WT", n * n).reshape(cases, S, n, n),        # [k][i] = Winv[i][k]
            "R": sl("OUT_R", n * nc).reshape(cases, S, n, nc),
            "raw": o,
        }

    def gj(self, A):
        n = self.n
        A = np.asarray(A, dtype=np.float64).reshape(-1, n, n)
        o = self._call(self.lib.bdf_probe_gj, A, A.shape[0] * (1 + n * n), A.shape[0]).reshape(-1, 1 + n * n)
        return o[:, 0].astype(int), o[:, 1:].reshape(-1, n, n)


def schur_T(rec, idx):
    """Complex upper-triangular T of a sweep-path record (idx = (case, step)): the diagonal from TD, the strict upper triangle
    from the skewed rows of T2S."""
    TD, T2S = rec["TD"][idx], rec["T2S"][idx]
    n, tw = T2S.shape[0], T2S.shape[1]
    T = np.zeros((n, n), dtype=complex)
    for r in range(n):
        T[r, r] = TD[r, 0] + 1j * TD[r, 1]
        for t in range(tw):
            k = r + 1 + t
            if k < n:
                T[r, k] = T2S[r, t, 0] + 1j * T2S[r, t, 1]
    return T
