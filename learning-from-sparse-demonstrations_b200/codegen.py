"""sympy -> CUDA C code generation for one optimal-control model.

Replaces CasADi's expression VM + AD (SURVEY.md §2 "Third-party: CasADi"; call sites
``/root/reference/CPDP/CPDP.py:53-79,107-124,209-248``): the dynamics, path cost, final cost and every
derivative the CPDP iteration needs are differentiated symbolically here, run through common-subexpression
elimination and emitted as ``__host__ __device__`` inline functions of a ``struct Model`` that the kernel
templates in ``csrc/cpdp_kernels.cuh`` are instantiated with.

Emitted members (n states, m controls, r parameters, nz = n+m):
  fc(x,u,th, f[n], &c)                       dynamics and path cost                    (CPDP.py:112)
  hgrad(x,u,th,mu,w, gx[n], gu[m])           gradient of  Ham = w*c + mu'f             (adjoint of one RK4 stage)
  dir(x,u,th,mu,w,dx,du, df[n], hz[nz])      df = fx dx + fu du ; hz = Hess_z(Ham) [dx;du]
  pmp(x,u,lam,th, M)                         dense, row-major matrices of CPDP.py:209-239 with H = c + lam'f,
                                             written at the PMP_* offsets; structural zeros are NOT written
                                             (the caller zero-fills the buffer once)
  term(x,th, &h, hx[n])                      final cost and gradient                   (CPDP.py:77-79,242)
  term2(x,th, hxx[n*n], hxe[n*r])            CPDP.py:245-248
  dir_th(x,u,th,mu,w,dx,du,dth, df[n], hz[nz])   df = fx dx + fu du + fth dth ; hz = Hess_z(Ham) [dx;du] + Hess_ztheta(Ham) dth
                                             (discrete auxiliary mode: theta-sensitivities of the RK4 stages)
plus static sparsity tables (CSR and CSC) of fx and fu used by the Riccati / auxiliary right-hand sides.
"""
import hashlib

import sympy as sp
from sympy.printing.c import C99CodePrinter

from .sx import SX, _to_matrix


class _Printer(C99CodePrinter):
    """C printer: integer powers as products, doubles with 17 significant digits."""

    def _print_Pow(self, expr):
        b, e = expr.base, expr.exp
        if e.is_Integer and 2 <= int(e) <= 4:
            s = self.parenthesize(b, 1000)
            return "(" + "*".join([s] * int(e)) + ")"
        if e.is_Integer and -4 <= int(e) <= -1:
            s = self.parenthesize(b, 1000)
            return "(1.0/(" + "*".join([s] * (-int(e))) + "))"
        return super()._print_Pow(expr)

    def _print_Float(self, expr):
        return repr(float(expr))

    def _print_Rational(self, expr):
        return "(%d.0/%d.0)" % (expr.p, expr.q)

    def _print_Integer(self, expr):
        return "%d.0" % int(expr) if abs(int(expr)) < 2 ** 53 else repr(float(expr))


_pr = _Printer()


def _vec(m):
    M = _to_matrix(m)
    return list(M) if M.shape[1] == 1 else list(M.T)


def _emit_body(assignments, indent="    "):
    """assignments: list of (c_lvalue, sympy expr). Returns C statements with CSE temporaries."""
    exprs = [sp.sympify(e) for _, e in assignments]
    repl, red = sp.cse(exprs, symbols=sp.numbered_symbols("t_"), optimizations="basic", order="none")
    lines = []
    for s, e in repl:
        lines.append("%sconst double %s = %s;" % (indent, _pr.doprint(s), _pr.doprint(e)))
    for (lhs, _), e in zip(assignments, red):
        lines.append("%s%s = %s;" % (indent, lhs, _pr.doprint(e)))
    nops = sum(int(sp.count_ops(e)) for _, e in repl) + sum(int(sp.count_ops(e)) for e in red)
    return "\n".join(lines), nops


def _sparse_tables(name, M):
    """CSR + CSC index tables of the structural non-zeros of sympy matrix M (row-major dense storage)."""
    nr, nc = M.shape
    rowptr, colidx = [0], []
    for i in range(nr):
        for j in range(nc):
            if M[i, j] != 0:
                colidx.append(j)
        rowptr.append(len(colidx))
    colptr, rowidx = [0], []
    for j in range(nc):
        for i in range(nr):
            if M[i, j] != 0:
                rowidx.append(i)
        colptr.append(len(rowidx))
    coor = [i for i in range(nr) for j in range(nc) if M[i, j] != 0]      # COO list in row-major order: folds to constants
    cooc = [j for i in range(nr) for j in range(nc) if M[i, j] != 0]      # in fully unrolled loops (straight-line products)
    def arr(nm, v):
        v = v if v else [0]
        return ("    CPDP_HD static constexpr int %s_%s(int i) { constexpr int t[%d] = {%s}; return t[i]; }"
                % (name, nm, len(v), ", ".join(map(str, v))))
    return "\n".join([arr("rowptr", rowptr), arr("colidx", colidx), arr("colptr", colptr), arr("rowidx", rowidx),
                      arr("coor", coor), arr("cooc", cooc),
                      "    static constexpr int %s_nnz = %d;" % (name, len(colidx))])


BOUND_INF = 1e20          # the reference's "no bound" (CPDP.py:24-29); |bound| >= 1e19 counts as none


def is_symbolic(v):
    """True for a bound entry that is an expression (of the per-problem constants), not a number."""
    return isinstance(v, sp.Basic)


def bound_entry(v):
    """One bound entry as a float, or as a sympy expression when it has free symbols (an SX / sympy scalar)."""
    if isinstance(v, SX):
        assert v.m.shape == (1, 1), "a bound entry is a scalar"
        v = v.m[0, 0]
    if isinstance(v, sp.Basic):
        return v if v.free_symbols else float(v)
    return float(v)


def bound_entries(v):
    """A bound vector (list / array of numbers or scalar expressions, or an SX / sympy column) as a flat list of bound_entry."""
    if isinstance(v, SX):
        v = v.m
    if isinstance(v, sp.MatrixBase):
        return [bound_entry(e) for e in v]
    if isinstance(v, (list, tuple)) or hasattr(v, "__array__"):
        out = []
        for e in (v.ravel() if hasattr(v, "ravel") else v):
            out.extend(bound_entries(e) if isinstance(e, (list, tuple, SX, sp.MatrixBase)) else [bound_entry(e)])
        return out
    return [bound_entry(v)]


def normalize_bounds(lb, ub, n):
    """Lists of n lower / upper bounds with every absent or infinite entry replaced by -/+BOUND_INF (expressions as they are)."""
    lb = [v if is_symbolic(v) else -BOUND_INF if v <= -1e19 else float(v) for v in (lb if len(lb) == n else [-BOUND_INF] * n)]
    ub = [v if is_symbolic(v) else BOUND_INF if v >= 1e19 else float(v) for v in (ub if len(ub) == n else [BOUND_INF] * n)]
    return lb, ub


def bounds_symbolic(bounds):
    """True when some entry of (state_lb, state_ub, control_lb, control_ub) is an expression."""
    return bounds is not None and any(is_symbolic(v) for part in bounds for v in part)


def _bound_exprs(bounds, e):
    """The four bound lists with every expression in the generated code's names (pd[i]); rejects an expression that uses
    anything but the per-problem constants."""
    names = ("state_lb", "state_ub", "control_lb", "control_ub")
    kinds = [("state", e["sym_x"]), ("control", e["sym_u"]), ("auxvar (theta)", e["sym_th"]), ("time", e["tv"])]
    out = []
    for nm, part in zip(names, bounds):
        row = []
        for i, v in enumerate(part):
            if is_symbolic(v):
                for kind, syms in kinds:
                    bad = v.free_symbols & set(syms)
                    if bad:
                        raise ValueError("%s[%d] = %s depends on the %s variable(s) %s: a bound may use only the problem variables "
                                         "(setProblemVariable) and constants" % (nm, i, v, kind, sorted(map(str, bad))))
                extra = v.free_symbols - set(e["sym_pd"])
                if extra:
                    raise ValueError("%s[%d] = %s has free symbols %s that are not problem variables (setProblemVariable)"
                                     % (nm, i, v, sorted(map(str, extra))))
                v = v.subs(dict(zip(e["sym_pd"], e["ps"])))
            row.append(v)
        out.append(row)
    return out


def _bounds_block(bounds, n, m, e=None):
    """Model members of the box bounds on the states and controls; empty text when no bound is finite, so that an unbounded
    model's header does not change.  Bounds with expressions of the per-problem constants (``e``: _model_exprs) give BOUNDS_PD
    and bound functions of pd."""
    if bounds is None:
        return ""
    if bounds_symbolic(bounds):
        return _bounds_block_pd(bounds, n, m, e)
    xlb, xub, ulb, uub = bounds
    if all(v <= -1e19 for v in list(xlb) + list(ulb)) and all(v >= 1e19 for v in list(xub) + list(uub)):
        return ""
    xlb, xub = normalize_bounds(xlb, xub, n)
    ulb, uub = normalize_bounds(ulb, uub, m)
    lines = ["    static constexpr int HAS_BOUNDS = 1;      // box bounds (+-1e20: none), read by the kernels' barrier method"]
    for nm, v in (("XLB", xlb), ("XUB", xub), ("ULB", ulb), ("UUB", uub)):
        # a chain of selects, not a table: a table indexed by a lane-dependent i would live in local memory
        expr = repr(v[-1])
        for i in range(len(v) - 2, -1, -1):
            expr = "i == %d ? %r : %s" % (i, v[i], expr)
        lines.append("    CPDP_HD static constexpr double %s(int i) { return %s; }" % (nm, expr))
    return "\n".join(lines) + "\n"


def _bounds_block_pd(bounds, n, m, e):
    xlb, xub, ulb, uub = bounds
    xlb, xub = normalize_bounds(xlb, xub, n)
    ulb, uub = normalize_bounds(ulb, uub, m)
    xlb, xub, ulb, uub = _bound_exprs((xlb, xub, ulb, uub), e)
    lines = ["    static constexpr int HAS_BOUNDS = 1;      // box bounds (+-1e20: none), read by the kernels' barrier method",
             "    static constexpr int BOUNDS_PD = 1;       // some bound is an expression of the per-problem constants pd"]
    val = lambda v: "(%s)" % _pr.doprint(v) if is_symbolic(v) else repr(v)
    for nm, v in (("XLB", xlb), ("XUB", xub), ("ULB", ulb), ("UUB", uub)):
        # a chain of selects, as for constant bounds; pd: the problem's constants (never the time slot)
        expr = val(v[-1])
        for i in range(len(v) - 2, -1, -1):
            expr = "i == %d ? %s : %s" % (i, val(v[i]), expr)
        lines.append("    CPDP_HD static double %s(int i, const double* __restrict__ pd) { (void)pd; return %s; }" % (nm, expr))
    return "\n".join(lines) + "\n"


def _model_exprs(state, control, auxvar, dyn, path_cost, final_cost, pdata, time):
    """The model's expressions in the array names of the generated C (x[i], u[i], th[i], pd[i], mu[i], w, dx[i], du[i]) and the
    derivatives that every generated function shares."""
    x, u, th = _vec(state), _vec(control), _vec(auxvar)
    pdv = _vec(pdata) if pdata is not None else []
    n, m, r = len(x), len(u), len(th)
    nq = len(pdv)
    tv = _vec(time) if time is not None else []
    assert len(tv) <= 1, "the time variable is a scalar"
    pdv = pdv + tv                                   # nq stays the number of USER constants; t rides behind them
    # sx.SX.sym is backed by sympy symbols, which are identified by NAME (CasADi's are distinct objects): a name reused across
    # state / control / auxvar / problem constants would silently alias two variables
    allsyms = x + u + th + pdv
    assert len(set(allsyms)) == len(allsyms), "state, control, auxvar and problem variables must have distinct symbol names"
    nz = n + m
    f = sp.Matrix(_vec(dyn))
    c = _to_matrix(path_cost)[0, 0]
    h = _to_matrix(final_cost)[0, 0]
    assert f.shape[0] == n
    extra = (f.free_symbols | c.free_symbols | h.free_symbols) - set(x) - set(u) - set(th) - set(pdv)
    assert not extra, "free symbols that are neither state, control nor auxvar: %s" % extra
    assert not (h.free_symbols & set(u)), "final cost must not depend on the control"

    # rename to array accesses
    xs = [sp.Symbol("x[%d]" % i, real=True) for i in range(n)]
    us = [sp.Symbol("u[%d]" % i, real=True) for i in range(m)]
    ts = [sp.Symbol("th[%d]" % i, real=True) for i in range(r)]
    ps = [sp.Symbol("pd[%d]" % i, real=True) for i in range(len(pdv))]
    sub = dict(zip(x + u + th + pdv, xs + us + ts + ps))
    f = f.subs(sub); c = c.subs(sub); h = h.subs(sub)
    z = xs + us
    mus = [sp.Symbol("mu[%d]" % i, real=True) for i in range(n)]
    w = sp.Symbol("w", real=True)
    dxs = [sp.Symbol("dx[%d]" % i, real=True) for i in range(n)]
    dus = [sp.Symbol("du[%d]" % i, real=True) for i in range(m)]

    fz = f.jacobian(z)
    Ham = w * c + sum(mus[i] * f[i] for i in range(n))
    Hz = sp.Matrix([Ham]).jacobian(z)
    Hzz = Hz.jacobian(z)
    dz = sp.Matrix(dxs + dus)

    return dict(n=n, m=m, r=r, nq=nq, nz=nz, tv=tv, f=f, c=c, h=h, xs=xs, us=us, ts=ts, ps=ps, z=z, mus=mus, w=w,
                fz=fz, Hz=Hz, Hzz=Hzz, dz=dz, sym_x=x, sym_u=u, sym_th=th, sym_pd=pdv[:nq])


def generate_model_header(name, state, control, auxvar, dyn, path_cost, final_cost, pdata=None, time=None, bounds=None):
    """Returns (header_text, info dict).  All arguments are SX / sympy matrices / scalars.
    ``pdata``: optional per-problem constants (e.g. a goal position) that are not learnable.
    ``time``: the explicit time variable of a COCSys_TimeVarying model (CPDP.py:434); the generated functions read it as
    one more constant, pd[nq], which the kernels fill in (the node time t_k in the RK4 map, the true t in the sweeps).
    ``bounds``: optional (state_lb, state_ub, control_lb, control_ub); the header gets HAS_BOUNDS and the four bound tables
    only when some bound is finite.  An entry may be an expression of the per-problem constants (DESIGN.md §3.12): then the
    header gets BOUNDS_PD and bound functions XLB(i, pd) ..."""
    e = _model_exprs(state, control, auxvar, dyn, path_cost, final_cost, pdata, time)
    n, m, r, nq, nz, tv = e["n"], e["m"], e["r"], e["nq"], e["nz"], e["tv"]
    f, c, h, xs, us, ts, z, mus, w = (e[k] for k in ("f", "c", "h", "xs", "us", "ts", "z", "mus", "w"))
    fz, Hz, Hzz, dz = e["fz"], e["Hz"], e["Hzz"], e["dz"]

    info = {}
    parts = []
    body, info["ops_fc"] = _emit_body([("f[%d]" % i, f[i]) for i in range(n)] + [("c", c)])
    parts.append("    CPDP_HD static void fc(const double* __restrict__ x, const double* __restrict__ u, "
                 "const double* __restrict__ th, const double* __restrict__ pd, double* __restrict__ f, double& c) {\n%s\n    }" % body)

    body, info["ops_hgrad"] = _emit_body([("gx[%d]" % i, Hz[i]) for i in range(n)] +
                                         [("gu[%d]" % i, Hz[n + i]) for i in range(m)])
    parts.append("    CPDP_HD static void hgrad(const double* __restrict__ x, const double* __restrict__ u, "
                 "const double* __restrict__ th, const double* __restrict__ pd, const double* __restrict__ mu, const double w, "
                 "double* __restrict__ gx, double* __restrict__ gu) {\n%s\n    }" % body)

    df = fz * dz
    hz = Hzz * dz
    body, info["ops_dir"] = _emit_body([("df[%d]" % i, df[i]) for i in range(n)] +
                                       [("hz[%d]" % i, hz[i]) for i in range(nz)])
    parts.append("    CPDP_HD static void dir(const double* __restrict__ x, const double* __restrict__ u, "
                 "const double* __restrict__ th, const double* __restrict__ pd, const double* __restrict__ mu, const double w, "
                 "const double* __restrict__ dx, const double* __restrict__ du, "
                 "double* __restrict__ df, double* __restrict__ hz) {\n%s\n    }" % body)

    # the same directional derivatives with a parameter tangent dth (forward theta-sensitivities of the RK4 stages and the
    # mixed z-theta Hessian of the interval Lagrangian, used by the discrete auxiliary mode)
    dths = [sp.Symbol("dth[%d]" % i, real=True) for i in range(r)]
    dth = sp.Matrix(dths)
    df_th = fz * dz + f.jacobian(ts) * dth
    hz_th = Hzz * dz + Hz.T.jacobian(ts) * dth
    body, info["ops_dir_th"] = _emit_body([("df[%d]" % i, df_th[i]) for i in range(n)] +
                                          [("hz[%d]" % i, hz_th[i]) for i in range(nz)])
    part_dir_th = ("    CPDP_HD static void dir_th(const double* __restrict__ x, const double* __restrict__ u, "
                   "const double* __restrict__ th, const double* __restrict__ pd, const double* __restrict__ mu, const double w, "
                   "const double* __restrict__ dx, const double* __restrict__ du, const double* __restrict__ dth, "
                   "double* __restrict__ df, double* __restrict__ hz) {\n%s\n    }" % body)

    # PMP set, H = c + lam' f  (lam takes the role of mu, w = 1)
    Hp = c + sum(mus[i] * f[i] for i in range(n))
    Hx = sp.Matrix([Hp]).jacobian(xs)
    Hu = sp.Matrix([Hp]).jacobian(us)
    mats = [("FX", f.jacobian(xs)), ("FU", f.jacobian(us)), ("FE", f.jacobian(ts)),
            ("HXX", Hx.jacobian(xs)), ("HXU", Hx.jacobian(us)), ("HXE", Hx.jacobian(ts)),
            ("HUU", Hu.jacobian(us)), ("HUE", Hu.jacobian(ts))]
    offs, off = [], 0
    assigns = []
    for nm, M in mats:
        offs.append("    static constexpr int PMP_%s = %d;" % (nm, off))
        for i in range(M.shape[0]):
            for j in range(M.shape[1]):
                if M[i, j] != 0:
                    assigns.append(("M[%d]" % (off + i * M.shape[1] + j), M[i, j]))
        off += M.shape[0] * M.shape[1]
    offs.append("    static constexpr int PMP_SIZE = %d;" % off)
    huu = mats[6][1]
    offs.append("    static constexpr bool HUU_DIAG = %s;      // structurally diagonal Huu: its inverse is NU reciprocals"
                % ("true" if all(huu[i, j] == 0 for i in range(m) for j in range(m) if i != j) else "false"))
    body, info["ops_pmp"] = _emit_body(assigns)
    body = body.replace("mu[", "lam[")
    parts.append("    CPDP_HD static void pmp(const double* __restrict__ x, const double* __restrict__ u, "
                 "const double* __restrict__ lam, const double* __restrict__ th, const double* __restrict__ pd, double* __restrict__ M) {\n%s\n    }" % body)
    info["pmp_nnz"] = len(assigns)

    # compact set for the forward auxiliary sweep (CPDP.py:295-297 needs fx, fu, fe and, through the aux control, Hxu, Hue, Huu;
    # not Hxx / Hxe): fx and fu as value lists in the row-major order of the FX_/FU_ COO tables, the rest dense
    fassign = []
    for tag, M in (("fxc", mats[0][1]), ("fuc", mats[1][1])):
        pidx = 0
        for i in range(M.shape[0]):
            for j in range(M.shape[1]):
                if M[i, j] != 0:
                    fassign.append(("%s[%d]" % (tag, pidx), M[i, j]))
                    pidx += 1
    for tag, M in (("fe", mats[2][1]), ("hxu", mats[4][1]), ("hue", mats[7][1]), ("huu", mats[6][1])):
        for i in range(M.shape[0]):
            for j in range(M.shape[1]):
                if M[i, j] != 0:
                    fassign.append(("%s[%d]" % (tag, i * M.shape[1] + j), M[i, j]))
    body, info["ops_pmp_fwd"] = _emit_body(fassign)
    body = body.replace("mu[", "lam[")
    parts.append("    CPDP_HD static void pmp_fwd(const double* __restrict__ x, const double* __restrict__ u, "
                 "const double* __restrict__ lam, const double* __restrict__ th, const double* __restrict__ pd, "
                 "double* __restrict__ fxc, double* __restrict__ fuc, double* __restrict__ fe, double* __restrict__ hxu, "
                 "double* __restrict__ hue, double* __restrict__ huu) {\n%s\n    }" % body)

    hx = sp.Matrix([h]).jacobian(xs)
    body, info["ops_term"] = _emit_body([("h", h)] + [("hx[%d]" % i, hx[i]) for i in range(n)])
    parts.append("    CPDP_HD static void term(const double* __restrict__ x, const double* __restrict__ th, const double* __restrict__ pd, "
                 "double& h, double* __restrict__ hx) {\n%s\n    }" % body)
    hxx = hx.jacobian(xs)
    hxe = hx.jacobian(ts)
    body, info["ops_term2"] = _emit_body([("hxx[%d]" % (i * n + j), hxx[i, j]) for i in range(n) for j in range(n)] +
                                         [("hxe[%d]" % (i * r + j), hxe[i, j]) for i in range(n) for j in range(r)])
    parts.append("    CPDP_HD static void term2(const double* __restrict__ x, const double* __restrict__ th, const double* __restrict__ pd, "
                 "double* __restrict__ hxx, double* __restrict__ hxe) {\n%s\n    }" % body)
    parts.append(part_dir_th)

    tables = "\n".join([_sparse_tables("FX", mats[0][1]), _sparse_tables("FU", mats[1][1]),
                        _sparse_tables("FE", mats[2][1])])
    info.update(n=n, m=m, r=r, nq=nq, nnz_fx=sum(1 for e in mats[0][1] if e != 0),
                nnz_fu=sum(1 for e in mats[1][1] if e != 0))

    text = """// GENERATED by lfsd_b200/codegen.py -- do not edit.  model: {name}
// n={n} m={m} r={r}; op counts after CSE: fc={ops_fc} hgrad={ops_hgrad} dir={ops_dir} pmp={ops_pmp} ({pmp_nnz} nnz)
#pragma once
#include "cpdp_port.h"
struct Model {{
    static constexpr int NX = {n};
    static constexpr int NU = {m};
    static constexpr int NP = {r};
    static constexpr int NQ = {nq};
    static constexpr int HAS_TIME = {has_time};
    static constexpr int NZ = {nz};
{bounds}{offs}
{tables}
{parts}
}};
""".format(name=name, nz=nz, has_time=len(tv), bounds=_bounds_block(bounds, n, m, e), offs="\n".join(offs), tables=tables,
           parts="\n\n".join(parts), **info)
    info["hash"] = hashlib.sha1(text.encode()).hexdigest()[:16]
    return text, info


def generate_pdata_header(name, state, control, auxvar, dyn, path_cost, final_cost, pdata=None, time=None, bounds=None):
    """Companion header ``model_<name>_pd.cuh``: ``struct ModelPd`` with the derivatives with respect to the NQ per-problem
    constants that the pdata adjoint (cpdp_aux_adjoint_pd, DESIGN.md §3.11) needs.  A separate file, so that the model header and
    its hash do not change.  Only the user constants pd[0..NQ-1] are differentiated; the time of a time-varying model, pd[NQ], is
    not a pdata column.  Returns (header_text, info dict).
      dir_pd(x,u,th,pd,mu,w,dx,du,dpd, df[n], hz[nz])   df = fz dz + f_pd dpd ; hz = Hess_z(Ham) dz + Hess_zpd(Ham) dpd
      term2_pd(x,th,pd, hxp[n*nq])                     d(grad_x h)/dpd, row-major
      dbounds(pd, dlb[nz*nq], dub[nz*nq])              d(bounds)/dpd, row-major, when some bound is an expression of pd
                                                       (BOUNDS_PD = 1; ``bounds`` as for generate_model_header)
    For NQ = 0 the struct holds NQ only."""
    e = _model_exprs(state, control, auxvar, dyn, path_cost, final_cost, pdata, time)
    n, nq, nz = e["n"], e["nq"], e["nz"]
    info = dict(nq=nq)
    parts = []
    if nq > 0:
        pq = e["ps"][:nq]
        dpd = sp.Matrix([sp.Symbol("dpd[%d]" % i, real=True) for i in range(nq)])
        df = e["fz"] * e["dz"] + e["f"].jacobian(pq) * dpd
        hz = e["Hzz"] * e["dz"] + e["Hz"].T.jacobian(pq) * dpd
        body, info["ops_dir_pd"] = _emit_body([("df[%d]" % i, df[i]) for i in range(n)] +
                                              [("hz[%d]" % i, hz[i]) for i in range(nz)])
        parts.append("    CPDP_HD static void dir_pd(const double* __restrict__ x, const double* __restrict__ u, "
                     "const double* __restrict__ th, const double* __restrict__ pd, const double* __restrict__ mu, const double w, "
                     "const double* __restrict__ dx, const double* __restrict__ du, const double* __restrict__ dpd, "
                     "double* __restrict__ df, double* __restrict__ hz) {\n%s\n    }" % body)
        hxp = sp.Matrix([e["h"]]).jacobian(e["xs"]).jacobian(pq)
        body, info["ops_term2_pd"] = _emit_body([("hxp[%d]" % (i * nq + j), hxp[i, j]) for i in range(n) for j in range(nq)])
        parts.append("    CPDP_HD static void term2_pd(const double* __restrict__ x, const double* __restrict__ th, "
                     "const double* __restrict__ pd, double* __restrict__ hxp) {\n%s\n    }" % body)
    if nq > 0 and bounds_symbolic(bounds):
        xlb, xub = normalize_bounds(bounds[0], bounds[1], e["n"])
        ulb, uub = normalize_bounds(bounds[2], bounds[3], e["m"])
        xlb, xub, ulb, uub = _bound_exprs((xlb, xub, ulb, uub), e)
        pq = e["ps"][:nq]
        assigns = []
        for tag, v in (("dlb", xlb + ulb), ("dub", xub + uub)):
            for j in range(nz):
                for q in range(nq):
                    assigns.append(("%s[%d]" % (tag, j * nq + q), sp.diff(v[j], pq[q]) if is_symbolic(v[j]) else sp.Integer(0)))
        body, info["ops_dbounds"] = _emit_body(assigns)
        parts.insert(0, "    static constexpr int BOUNDS_PD = 1;       // the bounds depend on pd: dbounds gives their Jacobians")
        parts.append("    CPDP_HD static void dbounds(const double* __restrict__ pd, double* __restrict__ dlb, double* __restrict__ dub) {"
                     "\n    (void)pd;\n%s\n    }" % body)
    text = """// GENERATED by lfsd_b200/codegen.py -- do not edit.  model: {name}, derivatives with respect to the per-problem constants
#pragma once
#include "cpdp_port.h"
struct ModelPd {{
    static constexpr int NQ = {nq};
{parts}
}};
""".format(name=name, nq=nq, parts="\n\n".join(parts))
    info["hash"] = hashlib.sha1(text.encode()).hexdigest()[:16]
    return text, info
