"""CPU restatement of the checked solve (cfs_solve_batch_margins / cfs_solve_checked, include/cfs_b200.h).  TEST INFRASTRUCTURE.

The C part (tests/repair_oracle.c) is compiled as the tail of a copy of oracle/cfs_oracle.c whose obstacle row reads
dist - (margin + offset) when offsets are given; the copy is made here, in the system's temporary directory (keyed by the
sources' contents), so neither the oracle nor the repository tree is written.  tests/check_oracle.c is linked in for the
continuous check.  The round loop of cfs_solve_checked is restated in Python (checked_solve).  twin=True builds the same sources
with FMA contraction allowed (the oracle's FMA twin, DESIGN.md section 2): a second faithful evaluation whose roundings differ.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import oracle as O
from tests import check_oracle as CO

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_HERE = os.path.dirname(os.path.abspath(__file__))
_ORC = os.path.join(_ROOT, "oracle", "cfs_oracle.c")
_SRC = [os.path.join(_HERE, "repair_oracle.c"), os.path.join(_HERE, "check_oracle.c"), os.path.join(_ROOT, "oracle", "cfs_oracle.h")]
_LINE = "      const double I = distance - c->margin[j];                             /* :117 */\n"
_NEW = "      const double I = distance - (orc_moff ? c->margin[j] + orc_moff[j * H + (i - 1)] : c->margin[j]); /* :117 */\n"
_libs = {}


def lib(twin=False):
    if twin not in _libs:
        src = open(_ORC).read()
        if src.count(_LINE) != 1 or src.count("int orc_get_con(") != 1:
            raise RuntimeError("oracle/cfs_oracle.c: the obstacle-row line of orc_get_con changed; update tests/repair_oracle.py")
        src = src.replace(_LINE, _NEW).replace("int orc_get_con(", "static _Thread_local const double *orc_moff;\nint orc_get_con(", 1)
        src += '\n#include "%s"\n' % os.path.join(_HERE, "repair_oracle.c")
        h = hashlib.sha256(src.encode())
        for f in _SRC:
            with open(f, "rb") as fh:
                h.update(fh.read())
        key = h.hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "cfs_repair_oracle%s_%d_%s.so" % ("_fma" if twin else "", os.getuid(), key))
        if not os.path.exists(so):
            d = tempfile.mkdtemp(prefix="cfs_repair_oracle_")
            cfile = os.path.join(d, "cfs_oracle_off.c")
            with open(cfile, "w") as fh:
                fh.write(src)
            tmp = so + ".%d.tmp" % os.getpid()
            fp = ["-ffp-contract=fast", "-mfma"] if twin else ["-ffp-contract=off"]
            subprocess.check_call(["gcc", "-O2"] + fp + ["-fopenmp", "-fPIC", "-std=c11", "-shared", "-I",
                                   os.path.join(_ROOT, "oracle"), "-o", tmp, cfile, os.path.join(_HERE, "check_oracle.c"), "-lm"])
            os.replace(tmp, so)
        _libs[twin] = C.CDLL(so)
    return _libs[twin]


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def solve_batch_off(P, x0, ff, caug, xref, moff=None, noise=None, nthreads=0, twin=False):
    """oracle.Problem.solve_batch with per-waypoint margin offsets moff (B, nobs, H) or None"""
    x0, ff, caug, xref = _f64(x0), _f64(ff), _f64(caug), _f64(xref)
    B, n, K = x0.shape[0], P.n, P.cfg.max_outer
    mo = None if moff is None else _f64(moff)
    nz = None if noise is None else _f64(noise)
    out = dict(u=np.zeros((B, n)), x=np.zeros((B, 2 * n)), cost_hist=np.zeros((B, K)), e_u_hist=np.zeros((B, K)),
               iters=np.zeros(B, dtype=np.int32), status=np.zeros(B, dtype=np.int32))
    lib(twin).orc_cfs_solve_batch_off(C.byref(P.r), C.byref(P.cfg), C.c_int(B), C.c_int(nthreads), _p(x0), _p(ff), _p(caug), _p(xref),
                                  _p(nz), _p(mo), _p(out["u"]), _p(out["x"]), _p(out["cost_hist"]), _p(out["e_u_hist"]),
                                  _p(out["iters"]), _p(out["status"]))
    return out


def repair_increments(scene, x0, x, u, seg_verdict, seg_s_hit, eta, gain, off):
    """adds the increments of B trajectories (per-segment verdict / s_hit (B, H)) to off (B, nobs, H) in place"""
    x0, x, u = _f64(np.atleast_2d(x0)), _f64(np.atleast_2d(x)), _f64(np.atleast_2d(u))
    B, H = x0.shape[0], u.shape[1] // scene.nj
    sv = np.ascontiguousarray(seg_verdict, dtype=np.int32)
    ss = _f64(seg_s_hit)
    assert off.flags["C_CONTIGUOUS"] and off.dtype == np.float64 and off.shape == (B, scene.nobs, H)
    lib().orc_repair_increments(C.byref(scene.r), C.c_int(scene.nobs), _p(scene.obs), _p(scene.margin), C.c_int(B), C.c_int(H),
                                _p(x0), _p(x), _p(u), _p(sv), _p(ss), C.c_double(eta), C.c_double(gain), _p(off))


def segment_check(scene, x0, x, u, eta, max_evals=4096):
    """per-segment verdict / s_hit / cmin (B, H) of B trajectories: every segment checked as a one-step trajectory (its t_hit is
    the segment's s_hit exactly, and for a HIT segment cmin is the clearance at the witness)"""
    nj = scene.nj
    B, H = x0.shape[0], u.shape[1] // nj
    X = np.concatenate([x0[:, None, :], x.reshape(B, H, 2 * nj)], axis=1)
    ck = scene.check_trajectories(X[:, :-1].reshape(B * H, 2 * nj), X[:, 1:].reshape(B * H, 2 * nj), u.reshape(B * H, nj),
                                  eta=eta, max_evals=max_evals)
    return ck["verdict"].reshape(B, H), ck["t_hit"].reshape(B, H), ck["cmin"].reshape(B, H)


def checked_solve(P, scene, x0, ff, caug, xref, eta=1e-3, rounds=4, gain=2.0, max_evals=4096, nthreads=0, twin=False):
    """The round loop of cfs_solve_checked on the CPU restatement (semantics in include/cfs_b200.h).  Also returns near (B,): the
    smallest distance to the -eta/2 threshold of any checked trajectory's cmin or any repair witness of the problem."""
    B, H, O_ = x0.shape[0], P.cfg.H, scene.nobs
    sol = solve_batch_off(P, x0, ff, caug, xref, None, nthreads=nthreads, twin=twin)
    ck = scene.check_trajectories(x0, sol["x"], sol["u"], eta=eta, max_evals=max_evals)
    near = np.abs(ck["cmin"] + 0.5 * eta)
    sol["near"] = near
    for k in ("verdict", "t_hit", "cmin"):
        sol[k] = ck[k].copy()
    sol["rounds_used"] = np.zeros(B, dtype=np.int32)
    off = np.zeros((B, O_, H))
    sol["margin_off"] = np.zeros((B, O_, H))  # the offsets of the returned solution
    if rounds == 0 or O_ == 0:
        return sol
    idx = np.nonzero((sol["verdict"] == CO.HIT) & ((sol["status"] & 0xFF) < 2))[0]
    cx0, cx, cu = x0[idx], sol["x"][idx], sol["u"][idx]
    for r in range(1, rounds + 1):
        if len(idx):
            sv, ss, scm = segment_check(scene, cx0, cx, cu, eta, max_evals)
            near[idx] = np.minimum(near[idx], np.where(sv == CO.HIT, np.abs(scm + 0.5 * eta), np.inf).min(axis=1))
            sub = np.ascontiguousarray(off[idx])
            repair_increments(scene, cx0, cx, cu, sv, ss, eta, gain, sub)
            off[idx] = sub
        else:
            break
        cand = solve_batch_off(P, x0[idx], ff[idx], caug[idx], xref[idx], off[idx], nthreads=nthreads, twin=twin)
        acc = (cand["status"] & 0xFF) < 2
        cck = scene.check_trajectories(x0[idx], cand["x"], cand["u"], eta=eta, max_evals=max_evals)
        near[idx] = np.minimum(near[idx], np.abs(cck["cmin"] + 0.5 * eta))
        a = idx[acc]
        for k in ("u", "x", "cost_hist", "e_u_hist", "iters", "status"):
            sol[k][a] = cand[k][acc]
        for k in ("verdict", "t_hit", "cmin"):
            sol[k][a] = cck[k][acc]
        sol["rounds_used"][a] = r
        sol["margin_off"][a] = off[a]
        keep = acc & (cck["verdict"] == CO.HIT)
        idx, cx0, cx, cu = idx[keep], x0[idx][keep], cand["x"][keep], cand["u"][keep]
    return sol
