"""CPU restatement of the joint position limits (cfs_set_joint_limits, include/cfs_b200.h).  TEST INFRASTRUCTURE.

The C part (tests/limits_oracle.c) is compiled as the tail of a copy of oracle/cfs_oracle.c whose orc_cfs_solve appends the 2n
constant limit rows after the bound rows when limits are given (m = mcon + bounds + 2n); the copy is made here, in the system's
temporary directory (keyed by the sources' contents), so neither the oracle nor the repository tree is written.  With no limits
the copy runs the oracle's exact code.  twin=True builds the same sources with FMA contraction allowed (the oracle's FMA twin,
DESIGN.md section 2).
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_HERE = os.path.dirname(os.path.abspath(__file__))
_ORC = os.path.join(_ROOT, "oracle", "cfs_oracle.c")
_SRC = [os.path.join(_HERE, "limits_oracle.c"), os.path.join(_ROOT, "oracle", "cfs_oracle.h")]
# (line of the oracle, its replacement): the row count of orc_cfs_solve, and the limit rows filled once before the outer loop
_PATCHES = [
    ("  const int m = mcon + (use_bounds ? 2 * n : 0);\n",
     "  const int m = mcon + (use_bounds ? 2 * n : 0) + (orc_qlim ? 2 * n : 0);\n"),
    ("  if (c->solver == 0) { /* unconstrained minimiser -QQ^{-1} ff = -J0 J0' ff, constant over the outer loop */\n",
     "  if (orc_qlim) orc_limit_rows(nj, H, r->dt, x0, orc_qlim, Cmat + (size_t)(m - 2 * n) * n, dvec + (m - 2 * n));\n"
     "  if (c->solver == 0) { /* unconstrained minimiser -QQ^{-1} ff = -J0 J0' ff, constant over the outer loop */\n"),
]
_DECL = ("static _Thread_local const double *orc_qlim;\n"
         "static void orc_limit_rows(int nj, int H, double dt, const double *x0, const double *qlim, double *A, double *b);\n")
_libs = {}


def lib(twin=False):
    if twin not in _libs:
        src = open(_ORC).read()
        if any(src.count(a) != 1 for a, _ in _PATCHES) or src.count("int orc_get_con(") != 1:
            raise RuntimeError("oracle/cfs_oracle.c: a line the limits oracle patches changed; update tests/limits_oracle.py")
        for a, b in _PATCHES:
            src = src.replace(a, b)
        src = src.replace("int orc_get_con(", _DECL + "int orc_get_con(", 1)
        src += '\n#include "%s"\n' % os.path.join(_HERE, "limits_oracle.c")
        h = hashlib.sha256(src.encode())
        for f in _SRC:
            with open(f, "rb") as fh:
                h.update(fh.read())
        key = h.hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "cfs_limits_oracle%s_%d_%s.so" % ("_fma" if twin else "", os.getuid(), key))
        if not os.path.exists(so):
            d = tempfile.mkdtemp(prefix="cfs_limits_oracle_")
            cfile = os.path.join(d, "cfs_oracle_lim.c")
            with open(cfile, "w") as fh:
                fh.write(src)
            tmp = so + ".%d.tmp" % os.getpid()
            fp = ["-ffp-contract=fast", "-mfma"] if twin else ["-ffp-contract=off"]
            subprocess.check_call(["gcc", "-O2"] + fp + ["-fopenmp", "-fPIC", "-std=c11", "-shared", "-I",
                                   os.path.join(_ROOT, "oracle"), "-o", tmp, cfile, "-lm"])
            os.replace(tmp, so)
        _libs[twin] = C.CDLL(so)
    return _libs[twin]


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _qlim(qmin, qmax):
    if qmin is None:
        return None
    return _f64(np.concatenate([np.asarray(qmin, dtype=np.float64).reshape(-1), np.asarray(qmax, dtype=np.float64).reshape(-1)]))


def solve_batch_lim(P, x0, ff, caug, xref, qmin=None, qmax=None, noise=None, nthreads=0, twin=False):
    """oracle.Problem.solve_batch with joint limits qmin / qmax (nj,) or None"""
    x0, ff, caug, xref = _f64(x0), _f64(ff), _f64(caug), _f64(xref)
    B, n, K = x0.shape[0], P.n, P.cfg.max_outer
    q = _qlim(qmin, qmax)
    nz = None if noise is None else _f64(noise)
    out = dict(u=np.zeros((B, n)), x=np.zeros((B, 2 * n)), cost_hist=np.zeros((B, K)), e_u_hist=np.zeros((B, K)),
               iters=np.zeros(B, dtype=np.int32), status=np.zeros(B, dtype=np.int32))
    qp = np.zeros((B, 2), dtype=np.int32)
    lib(twin).orc_cfs_solve_batch_lim(C.byref(P.r), C.byref(P.cfg), C.c_int(B), C.c_int(nthreads), _p(x0), _p(ff), _p(caug),
                                      _p(xref), _p(nz), _p(q), _p(out["u"]), _p(out["x"]), _p(out["cost_hist"]),
                                      _p(out["e_u_hist"]), _p(out["iters"]), _p(out["status"]), _p(qp))
    out["qp_iters"], out["qp_max_active"] = qp[:, 0], qp[:, 1]
    return out


def get_con_lim(P, x0, xcur, u, qmin=None, qmax=None):
    """oracle.Problem.get_con rows followed by the limit rows (upper, then lower, [waypoint][joint] order): (A, b)"""
    rows = P.cfg.nobs * P.H * ((1 + 2 * P.nj) if P.lim is not None else 1) + (2 * P.n if qmin is not None else 0)
    A = np.zeros((rows, P.n))
    b = np.zeros(rows)
    m = lib().orc_get_con_lim(C.byref(P.r), C.byref(P.cfg), _p(_f64(x0)), _p(_f64(xcur)), _p(_f64(u)), _p(_qlim(qmin, qmax)),
                              _p(A), _p(b))
    assert m == rows
    return A, b


def waypoint_theta(x, nj):
    """theta at waypoints 1..H of trajectories x (B, 2 nj H): (B, H, nj)"""
    x = np.asarray(x)
    return x.reshape(x.shape[0], -1, 2 * nj)[:, :, :nj]
