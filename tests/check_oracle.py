"""ctypes binding of the CPU restatement of the continuous collision checks (tests/check_oracle.c).  TEST INFRASTRUCTURE ONLY.

The library is oracle/cfs_oracle.c and tests/check_oracle.c compiled together with the oracle's flags; it is built on first use
into the system's temporary directory (keyed by the sources' contents), so the repository tree is never written.
Array layouts are the C ABI's, as numpy rows: theta (N, nj), x0 (B, 2nj), x (B, 2njH), u (B, njH).
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import oracle as O

CLEAR, HIT, UNDECIDED = 0, 1, 2
_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_SRC = [os.path.join(_ROOT, "oracle", "cfs_oracle.c"), os.path.join(os.path.dirname(os.path.abspath(__file__)), "check_oracle.c")]
_HDR = os.path.join(_ROOT, "oracle", "cfs_oracle.h")
_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for f in _SRC + [_HDR]:
            with open(f, "rb") as fh:
                h.update(fh.read())
        so = os.path.join(tempfile.gettempdir(), "cfs_check_oracle_%d_%s.so" % (os.getuid(), h.hexdigest()[:16]))
        if not os.path.exists(so):
            tmp = so + ".%d.tmp" % os.getpid()
            subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fopenmp", "-fPIC", "-std=c11", "-shared",
                                   "-I", os.path.join(_ROOT, "oracle"), "-o", tmp] + _SRC + ["-lm"])
            os.replace(tmp, so)
        _lib = C.CDLL(so)
        _lib.orc_clearance.restype = C.c_double
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def motion_bound(r):
    R = np.zeros(O.MAXL)
    lib().orc_motion_bound(C.byref(r), _p(R))
    return R[:r.nj]


class Scene:
    """Robot + obstacles + margins (obs{j}.D if margin_is_D else obs{j}.epsilon), as the library's context holds them."""

    def __init__(self, robot_name, obs, margin_is_D=True):
        self.r = O.robot(robot_name)
        self.nj = self.r.nj
        self.obs = _f64(np.concatenate([O.obs6(o) for o in obs]))
        self.margin = _f64([o["D"] if margin_is_D else o["epsilon"] for o in obs])
        self.nobs = len(obs)

    def check_args(self, eta, max_evals):
        if not (eta > 0 and np.isfinite(eta)):
            raise ValueError("eta must be positive and finite")
        if max_evals < 1:
            raise ValueError("max_evals must be >= 1")
        if self.nobs and not (self.margin.min() - eta >= 1e-4):
            raise ValueError("margin - eta is below 1e-4")

    def clearance(self, theta):
        """c(theta) for theta (N, nj)"""
        th = _f64(np.atleast_2d(theta))
        c = np.zeros(th.shape[0])
        lib().orc_clearance_batch(C.byref(self.r), C.c_int(self.nobs), _p(self.obs), _p(self.margin), C.c_int(th.shape[0]),
                                  _p(th), _p(c))
        return c

    def check_edges(self, theta_a, theta_b, eta=1e-3, max_evals=4096):
        self.check_args(eta, max_evals)
        ta, tb = _f64(np.atleast_2d(theta_a)), _f64(np.atleast_2d(theta_b))
        N = ta.shape[0]
        out = dict(verdict=np.zeros(N, dtype=np.int32), s_hit=np.zeros(N), cmin=np.zeros(N), evals=np.zeros(N, dtype=np.int32))
        lib().orc_check_edges_batch(C.byref(self.r), C.c_int(self.nobs), _p(self.obs), _p(self.margin), C.c_int(N), _p(ta), _p(tb),
                                    C.c_double(eta), C.c_int(max_evals), _p(out["verdict"]), _p(out["s_hit"]), _p(out["cmin"]),
                                    _p(out["evals"]))
        return out

    def check_trajectories(self, x0, x, u, eta=1e-3, max_evals=4096):
        self.check_args(eta, max_evals)
        x0, x, u = _f64(np.atleast_2d(x0)), _f64(np.atleast_2d(x)), _f64(np.atleast_2d(u))
        B, H = x0.shape[0], u.shape[1] // self.nj
        out = dict(verdict=np.zeros(B, dtype=np.int32), t_hit=np.zeros(B), cmin=np.zeros(B), evals=np.zeros(B, dtype=np.int32))
        lib().orc_check_trajectories_batch(C.byref(self.r), C.c_int(self.nobs), _p(self.obs), _p(self.margin), C.c_int(B),
                                           C.c_int(H), _p(x0), _p(x), _p(u), C.c_double(eta), C.c_int(max_evals),
                                           _p(out["verdict"]), _p(out["t_hit"]), _p(out["cmin"]), _p(out["evals"]))
        return out


def segment_points(x0, x, u, nj, dt, k, tau):
    """theta(tau) on segment k of one trajectory (tau an array), the double integrator of include/cfs_b200.h"""
    xs = x0 if k == 0 else x[(k - 1) * 2 * nj:k * 2 * nj]
    th, om, uk = xs[:nj], xs[nj:2 * nj], u[k * nj:(k + 1) * nj]
    tau = np.asarray(tau, dtype=np.float64)[:, None]
    return (th + om * tau) + ((0.5 * tau) * tau) * uk
