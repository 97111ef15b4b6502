"""-m gpu : the gateway's 'solve' command with sys_info.qlim (matlab/cfs_mex.cpp, compiled against tests/mex_stub/) returns bit for
bit what Context.solve_batch returns with the same joint limits, and the following calls without qlim ('solve', 'routes') on the
gateway's cached context are the plain solves."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np
import pytest

import motionplanning_5d_m_b200 as M
from tests import common
from motionplanning_5d_m_b200 import problem
from tests.test_limits import inside_box, limit_box
from tests.test_mex_gateway import call_mex_routes

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
KEYS = ("u", "x", "cost_hist", "e_u_hist", "iters", "status")


@pytest.fixture(scope="module")
def harness():
    """tests/mex_stub/limits_harness.cpp + matlab/cfs_mex.cpp, built into the temporary directory (keyed by the sources)"""
    src = [os.path.join(HERE, "mex_stub", "limits_harness.cpp"), os.path.join(ROOT, "matlab", "cfs_mex.cpp")]
    deps = src + [os.path.join(HERE, "mex_stub", f) for f in ("harness.cpp", "mex.h")] + [os.path.join(ROOT, "include", "cfs_b200.h")]
    h = hashlib.sha256()
    for f in deps:
        with open(f, "rb") as fh:
            h.update(fh.read())
    libdir = os.path.join(ROOT, "motionplanning_5d_m_b200")
    so = os.path.join(tempfile.gettempdir(), "cfs_mex_limits_%d_%s.so" % (os.getuid(), h.hexdigest()[:16]))
    if not os.path.exists(so):
        tmp = so + ".%d.tmp" % os.getpid()
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-I", os.path.join(HERE, "mex_stub"), "-I",
                               os.path.join(ROOT, "include"), "-o", tmp] + src + ["-L", libdir, "-lcfs_b200", "-Wl,-rpath," + libdir])
        os.replace(tmp, so)
    lib = C.CDLL(so)
    lib.mexh_last_error.restype = C.c_char_p
    yield lib
    lib.mexh_shutdown()


def _dp(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def call_mex(h, robot, obs, s, x0, ff, caug, xref, qlim=None):
    nj, H = int(s["njoint"]), int(s["H"])
    n, B, K = nj * H, x0.shape[0], int(s["MAX_O_ITER"])
    f = lambda a: np.ascontiguousarray(a, dtype=np.float64)
    DH = np.asfortranarray(robot["DH"], dtype=np.float64)
    cap = np.asfortranarray(np.stack([np.asarray(robot["cap"][i]["p"], dtype=np.float64)[:, :2] for i in range(nj)], axis=2))
    seg = np.asfortranarray(np.stack([np.asarray(o["l"], dtype=np.float64) for o in obs], axis=2))
    keep = dict(D=f([o["D"] for o in obs]), eps=f([o["epsilon"] for o in obs]), base=f(np.asarray(robot["base"]).reshape(-1)),
                QQ=f(s["QQ"].T), lim=f(s["lim"]), mi=f(s["MAX_input"]), x0=f(x0), ff=f(ff), caug=f(caug), xref=f(xref),
                q=None if qlim is None else np.asfortranarray(qlim, dtype=np.float64))
    out = dict(u=np.zeros((B, n)), x=np.zeros((B, 2 * n)), cost_hist=np.zeros((B, K)), e_u_hist=np.zeros((B, K)),
               iters=np.zeros(B, dtype=np.int32), status=np.zeros(B, dtype=np.int32))
    rc = h.mexh_solve_qlim(b"M16iB", C.c_int(nj), C.c_int(H), C.c_int(B), C.c_int(DH.shape[0]), _dp(DH), _dp(keep["base"]), _dp(cap),
                           C.c_double(robot["delta_t"]), C.c_int(len(obs)), _dp(seg), _dp(keep["D"]), _dp(keep["eps"]), _dp(keep["QQ"]),
                           _dp(keep["lim"]), _dp(keep["mi"]), _dp(keep["q"]), _dp(keep["x0"]), _dp(keep["ff"]), _dp(keep["caug"]),
                           _dp(keep["xref"]), C.c_double(s["epsilon_O"]), C.c_int(K), *(_dp(out[k]) for k in KEYS))
    if rc:
        raise RuntimeError(h.mexh_last_error().decode())
    return out


def test_solve_qlim_through_the_gateway(harness, oracle):
    cfg = common.batch_m16ib(oracle, 2048)
    idx = inside_box(cfg)[:128]
    s, obs = cfg["sys_info"], cfg["obs"]
    args = tuple(np.ascontiguousarray(cfg[k][idx]) for k in ("x0", "ff", "caug", "xref"))
    lo, hi = limit_box()
    ctx = M.Context(0)
    try:
        ctx.set_robot(dict(cfg["robot"], name="M16iB"), 5)
        ctx.set_obstacles(obs)
        ctx.set_cost(s["H"], s["QQ"], s["lim"], s["MAX_input"])
        plain = ctx.solve_batch(*args, s["epsilon_O"], s["MAX_O_ITER"])
        ctx.set_joint_limits(lo, hi)
        limited = ctx.solve_batch(*args, s["epsilon_O"], s["MAX_O_ITER"])
    finally:
        ctx.close()
    th0, thg = cfg["theta0"][idx], cfg["thetag"][idx]
    routes = np.ascontiguousarray(np.stack([th0, 0.5 * (th0 + thg), thg], axis=1))
    rl = np.full(len(idx), 3.0)
    mi = np.asarray(s["MAX_input"]).reshape(-1)
    rargs = ("M16iB", cfg["robot"], obs, s["H"], routes, rl, problem.Q_MAIN_FANUC, problem.R_MAIN_FANUC, 50.0, s["lim"], mi)
    rt_clean = call_mex_routes(harness, *rargs, eps_outer=s["epsilon_O"], max_outer=s["MAX_O_ITER"])
    out = call_mex(harness, cfg["robot"], obs, s, *args, qlim=np.stack([lo, hi], axis=1))
    for k in KEYS:
        assert np.array_equal(out[k], limited[k], equal_nan=True), k
    rt = call_mex_routes(harness, *rargs, eps_outer=s["epsilon_O"], max_outer=s["MAX_O_ITER"])  # must not keep the limits
    for k in KEYS:
        assert np.array_equal(rt[k], rt_clean[k], equal_nan=True), k
    call_mex(harness, cfg["robot"], obs, s, *args, qlim=np.stack([lo, hi], axis=1))
    again = call_mex(harness, cfg["robot"], obs, s, *args)  # the cached context must not keep the limits
    for k in KEYS:
        assert np.array_equal(again[k], plain[k], equal_nan=True), k
    with pytest.raises(RuntimeError, match="cfs_set_joint_limits"):
        call_mex(harness, cfg["robot"], obs, s, *args, qlim=np.stack([hi, lo], axis=1))
