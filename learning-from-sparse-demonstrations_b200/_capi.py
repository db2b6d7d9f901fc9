"""ctypes binding of the C ABI in ``include/cpdp.h`` and the nvcc build of one model library.

The library is the product path: nothing here falls back to a CPU implementation.  If the shared object is
missing it is compiled with nvcc for sm_100a (in-tree, under ``lib/``); if that is impossible the call raises.
"""
import ctypes
import hashlib
import os
import shutil
import subprocess

_PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_PKG, "csrc")
GEN_DIR = os.path.join(CSRC, "generated")
LIB_DIR = os.path.join(_PKG, "lib")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC,-fvisibility=hidden"]
# developer knob for tuning experiments (e.g. -DCPDP_HESS_MINB=2): forces a rebuild here and is deliberately NOT part of the
# build digest, so that a variant built in this container is used as it is on a GPU box that does not set the variable
EXTRA_NVCC_FLAGS = os.environ.get("CPDP_EXTRA_NVCC_FLAGS", "").split()

STATUS_NAMES = {0: "running", 1: "converged", 2: "max_iter", 3: "linesearch_fail", 4: "numeric", 5: "infeasible"}

_vp = ctypes.c_void_p
_i = ctypes.c_int
_d = ctypes.c_double
_sz = ctypes.c_size_t


_DIGEST_MARK = "CPDP_BUILD_DIGEST="


class CpdpError(RuntimeError):
    pass


def _sources_digest():
    h = hashlib.sha1()
    for fn in sorted(os.listdir(CSRC)):
        p = os.path.join(CSRC, fn)
        if os.path.isfile(p):
            h.update(fn.encode())
            with open(p, "rb") as f:
                h.update(f.read())
    return h.hexdigest()[:16]


def build_model_library(name, header_text, force=False, verbose=False, pd_header_text=None):
    """Writes csrc/generated/model_<name>.cuh (and, given ``pd_header_text``, the companion model_<name>_pd.cuh with the pdata
    derivatives, codegen.generate_pdata_header) and compiles lib/libcpdp_<name>.so (skipped when up to date)."""
    os.makedirs(GEN_DIR, exist_ok=True)
    os.makedirs(LIB_DIR, exist_ok=True)
    hdr = os.path.join(GEN_DIR, "model_%s.cuh" % name)
    pd_hdr = os.path.join(GEN_DIR, "model_%s_pd.cuh" % name)
    so = os.path.join(LIB_DIR, "libcpdp_%s.so" % name)
    stamp = so + ".stamp"
    digest = hashlib.sha1((header_text + (pd_header_text or "") + _sources_digest() +
                           " ".join(NVCC_FLAGS + EXTRA_NVCC_FLAGS)).encode()).hexdigest()

    def up_to_date():
        # The digest of (model header, kernel sources, all flags) is compiled INTO the library (cpdp_build_digest), so a prebuilt
        # .so is recognised wherever it travels without any side file (git-ignored stamp files do not reach a GPU box), and a
        # tuning build (CPDP_EXTRA_NVCC_FLAGS) is never mistaken for the default one.
        if force or not os.path.exists(so):
            return False
        with open(so, "rb") as f:
            return (_DIGEST_MARK + digest).encode() in f.read()

    if up_to_date():
        return so
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise CpdpError("libcpdp_%s.so is missing and nvcc was not found; the CUDA extension is required "
                        "(there is no CPU fallback)" % name)
    # One builder at a time per library (every rank of a torchrun job calls build()): the others wait on the lock and then find
    # the finished file.  The compiler writes to a temporary name; the rename is atomic, so no process ever maps a partial file.
    import fcntl
    with open(so + ".lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and up_to_date():
                return so
            with open(hdr, "w") as f:
                f.write(header_text)
            pd_flags = []
            if pd_header_text is not None:
                with open(pd_hdr, "w") as f:
                    f.write(pd_header_text)
                pd_flags = ["-DCPDP_PD_HEADER=\"%s\"" % pd_hdr]
            ns = "cpdp_" + "".join(ch if ch.isalnum() else "_" for ch in name)
            tmp = "%s.tmp%d" % (so, os.getpid())
            cmd = [nvcc] + NVCC_FLAGS + EXTRA_NVCC_FLAGS + ["-I", CSRC, "-DCPDP_NS=%s" % ns, "-DCPDP_MODEL_HEADER=\"%s\"" % hdr,
                                         "-DCPDP_BUILD_DIGEST=\"%s%s\"" % (_DIGEST_MARK, digest)] + pd_flags + [
                                         os.path.join(CSRC, "cpdp_lib.cu"), "-o", tmp]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
                print(" ".join(cmd))
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                if os.path.exists(tmp):
                    os.remove(tmp)
                raise CpdpError("nvcc failed for model %s:\n%s\n%s" % (name, r.stdout, r.stderr))
            if verbose:
                print(r.stderr)
            os.replace(tmp, so)
            with open(stamp, "w") as f:
                f.write(digest)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return so


class CpdpLib:
    """Thin typed wrapper over one libcpdp_<model>.so.  All pointer arguments are integer addresses."""

    def __init__(self, so_path):
        if not os.path.exists(so_path):
            raise CpdpError("CUDA extension %s not found (no CPU fallback exists)" % so_path)
        self.path = so_path
        L = self.L = ctypes.CDLL(so_path)
        L.cpdp_model_dims.argtypes = [ctypes.POINTER(_i)] * 4
        L.cpdp_model_dims.restype = _i
        L.cpdp_riccati_state_dim.restype = _i
        L.cpdp_last_rounds.restype = _i
        L.cpdp_workspace_bytes.argtypes = [_i, _i, _i]
        L.cpdp_workspace_bytes.restype = _sz
        L.cpdp_solve.argtypes = [_vp, _sz, _i, _i, _i, _d, _vp, _vp, _i, _vp, _d, _i, _i,
                                 _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]
        L.cpdp_solve.restype = _i
        L.cpdp_solve_warm.argtypes = L.cpdp_solve.argtypes + [_vp, _vp, _vp, _vp, _vp, _vp, _i, _d]
        L.cpdp_solve_warm.restype = _i
        L.cpdp_aux.argtypes = [_vp, _sz, _i, _i, _i, _d, _vp, _i, _vp, _vp, _vp, _vp, _vp,
                               _i, _d, _d, _d, _d, _i, _i, ctypes.POINTER(_i), _vp, _i, _vp,
                               _vp, _vp, _vp, _vp, _vp, _vp, _vp]
        L.cpdp_aux.restype = _i
        L.cpdp_aux_phases.argtypes = L.cpdp_aux.argtypes + [_i]
        L.cpdp_aux_phases.restype = _i
        L.cpdp_aux_adjoint.argtypes = [_vp, _sz, _i, _i, _i, _d, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]
        L.cpdp_aux_adjoint.restype = _i
        L.cpdp_pdata_workspace_bytes.argtypes = [_i, _i]
        L.cpdp_pdata_workspace_bytes.restype = _sz
        L.cpdp_aux_adjoint_pd.argtypes = [_vp, _sz, _vp, _sz, _i, _i, _i, _d, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                          _vp, _vp, _vp]
        L.cpdp_aux_adjoint_pd.restype = _i
        L.cpdp_dfma_probe.argtypes = [_vp, _i, _i, _vp]
        L.cpdp_dfma_probe.restype = _i
        L.cpdp_reduce.argtypes = [_vp, _vp, _i, _vp, _vp, _vp]
        L.cpdp_reduce.restype = _i
        L.cpdp_pack_rows.argtypes = [_vp, _vp, _vp, _vp, _i, _vp, _vp]
        L.cpdp_pack_rows.restype = _i
        L.cpdp_reduce_rows.argtypes = [_vp, _i, _i, _vp, _vp, _vp]
        L.cpdp_reduce_rows.restype = _i
        L.cpdp_optim_step.argtypes = [_i, _i, _d, _d, _d, _d, _d, _d, _d, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp]
        L.cpdp_optim_step.restype = _i
        L.cpdp_bounds.argtypes = [ctypes.POINTER(_d), ctypes.POINTER(_d)]
        L.cpdp_bounds.restype = _i
        L.cpdp_eval_bounds.argtypes = [_vp, _i, _vp, _vp, _vp]
        L.cpdp_eval_bounds.restype = _i
        for fn in (L.cpdp_get_bound_multipliers, L.cpdp_set_bound_multipliers):
            fn.argtypes = [_vp, _sz, _i, _i, _i, _vp, _vp, _vp, _vp]
            fn.restype = _i
        if hasattr(L, "cpdp_error_string"):
            L.cpdp_error_string.argtypes = [_i]
            L.cpdp_error_string.restype = ctypes.c_char_p
        n, m, r, q = _i(), _i(), _i(), _i()
        L.cpdp_model_dims(ctypes.byref(n), ctypes.byref(m), ctypes.byref(r), ctypes.byref(q))
        self.n, self.m, self.r, self.q = n.value, m.value, r.value, q.value
        self.nyr = L.cpdp_riccati_state_dim()
        L.cpdp_num_counters.restype = _i
        L.cpdp_has_bdf.restype = _i
        self.ncounters = int(L.cpdp_num_counters())
        self.has_bdf = bool(L.cpdp_has_bdf())
        lb, ub = (_d * (self.n + self.m))(), (_d * (self.n + self.m))()
        nb = L.cpdp_bounds(lb, ub)
        self.has_bounds = bool(nb)
        self.bounds_pd = nb == 2                       # some bound depends on pdata (those entries read NaN)
        self.lb, self.ub = list(lb), list(ub)          # states then controls, +-1e20 for none

    def check(self, rc, what):
        if rc != 0:
            msg = self.L.cpdp_error_string(rc).decode() if hasattr(self.L, "cpdp_error_string") else ""
            raise CpdpError("%s failed with code %d (%s)" % (what, rc, msg))

    def last_rounds(self):
        return int(self.L.cpdp_last_rounds())

    def workspace_bytes(self, B, N, S):
        return int(self.L.cpdp_workspace_bytes(B, N, S))

    def solve(self, ws, ws_bytes, B, N, S, T, x0, theta, theta_stride, pdata, tol, max_iter, rounds,
              X, U, Lam, status, iters, kkt, cost, stream):
        self.check(self.L.cpdp_solve(ws, ws_bytes, B, N, S, T, x0, theta, theta_stride, pdata, tol, max_iter, rounds,
                                     X, U, Lam, status, iters, kkt, cost, stream), "cpdp_solve")

    def solve_warm(self, ws, ws_bytes, B, N, S, T, x0, theta, theta_stride, pdata, tol, max_iter, rounds,
                   X, U, Lam, status, iters, kkt, cost, stream, Xg, Ug, Lg, Zlg, Zug, init_status, shift, mu_init):
        self.check(self.L.cpdp_solve_warm(ws, ws_bytes, B, N, S, T, x0, theta, theta_stride, pdata, tol, max_iter, rounds,
                                          X, U, Lam, status, iters, kkt, cost, stream, Xg, Ug, Lg, Zlg, Zug, init_status, shift,
                                          mu_init), "cpdp_solve_warm")

    def aux(self, ws, ws_bytes, B, N, S, T, theta, theta_stride, pdata, X, U, Lam, solve_status,
            mode, rtol_b, atol_b, rtol_f, atol_f, W, D, sel, taus, taus_stride, wp,
            Xa, Ua, loss, dtheta, aux_status, counters, stream, phases=3):
        sel_arr = (_i * max(1, len(sel)))(*sel) if sel else (_i * 1)(0)
        args = (ws, ws_bytes, B, N, S, T, theta, theta_stride, pdata, X, U, Lam, solve_status,
                mode, rtol_b, atol_b, rtol_f, atol_f, W, D, sel_arr, taus, taus_stride, wp,
                Xa, Ua, loss, dtheta, aux_status, counters, stream)
        if phases == 3:
            self.check(self.L.cpdp_aux(*args), "cpdp_aux")
        else:
            self.check(self.L.cpdp_aux_phases(*(args + (phases,))), "cpdp_aux_phases")

    def aux_adjoint(self, ws, ws_bytes, B, N, S, T, theta, theta_stride, pdata, X, U, Lam, solve_status, Xbar, Ubar,
                    theta_bar, x0_bar, aux_status, stream):
        self.check(self.L.cpdp_aux_adjoint(ws, ws_bytes, B, N, S, T, theta, theta_stride, pdata, X, U, Lam, solve_status, Xbar,
                                           Ubar, theta_bar, x0_bar, aux_status, stream), "cpdp_aux_adjoint")

    def pdata_workspace_bytes(self, B, N):
        return int(self.L.cpdp_pdata_workspace_bytes(B, N))

    def aux_adjoint_pd(self, ws, ws_bytes, pd_ws, pd_ws_bytes, B, N, S, T, theta, theta_stride, pdata, X, U, Lam, solve_status,
                       Xbar, Ubar, theta_bar, x0_bar, pdata_bar, aux_status, stream):
        self.check(self.L.cpdp_aux_adjoint_pd(ws, ws_bytes, pd_ws, pd_ws_bytes, B, N, S, T, theta, theta_stride, pdata, X, U, Lam,
                                              solve_status, Xbar, Ubar, theta_bar, x0_bar, pdata_bar, aux_status, stream),
                   "cpdp_aux_adjoint_pd")

    def eval_bounds(self, pdata, B, lb, ub, stream):
        self.check(self.L.cpdp_eval_bounds(pdata, B, lb, ub, stream), "cpdp_eval_bounds")

    def get_bound_multipliers(self, ws, ws_bytes, B, N, S, Zl, Zu, mu, stream):
        self.check(self.L.cpdp_get_bound_multipliers(ws, ws_bytes, B, N, S, Zl, Zu, mu, stream), "cpdp_get_bound_multipliers")

    def set_bound_multipliers(self, ws, ws_bytes, B, N, S, Zl, Zu, mu, stream):
        self.check(self.L.cpdp_set_bound_multipliers(ws, ws_bytes, B, N, S, Zl, Zu, mu, stream), "cpdp_set_bound_multipliers")

    def dfma_probe(self, sink, blocks, iters, stream):
        self.check(self.L.cpdp_dfma_probe(sink, blocks, iters, stream), "cpdp_dfma_probe")

    def pack_rows(self, loss, dtheta, solve_status, aux_status, B, rows, stream):
        self.check(self.L.cpdp_pack_rows(loss, dtheta, solve_status, aux_status, B, rows, stream), "cpdp_pack_rows")

    def reduce_rows(self, rows, B, C, scratch, out, stream):
        self.check(self.L.cpdp_reduce_rows(rows, B, C, scratch, out, stream), "cpdp_reduce_rows")

    def optim_step(self, phase, method, lr, mu, beta1, beta2, eps, loss_stop, grad_stop, theta, theta_eval, state, red, it,
                   loss_trace, param_trace, cap, defer_close, stream):
        self.check(self.L.cpdp_optim_step(phase, method, lr, mu, beta1, beta2, eps, loss_stop, grad_stop, theta, theta_eval,
                                          state, red, it, loss_trace, param_trace, cap, defer_close, stream), "cpdp_optim_step")

    def reduce(self, loss, dtheta, B, scratch, out, stream):
        self.check(self.L.cpdp_reduce(loss, dtheta, B, scratch, out, stream), "cpdp_reduce")
