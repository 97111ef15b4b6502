"""-m gpu : the 'check' command of the MEX gateway (matlab/cfs_mex.cpp, compiled against tests/mex_stub/) returns bit for bit
what the ctypes path returns, for edges and for solved trajectories."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np
import pytest

import motionplanning_5d_m_b200 as M
from motionplanning_5d_m_b200 import synthetic
from tests import common
from tests.test_edge_check import random_edges

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


@pytest.fixture(scope="module")
def harness():
    """tests/mex_stub/check_harness.cpp + matlab/cfs_mex.cpp, built into the temporary directory (keyed by the sources)"""
    src = [os.path.join(HERE, "mex_stub", "check_harness.cpp"), os.path.join(ROOT, "matlab", "cfs_mex.cpp")]
    deps = src + [os.path.join(HERE, "mex_stub", f) for f in ("harness.cpp", "mex.h")] + [os.path.join(ROOT, "include", "cfs_b200.h")]
    h = hashlib.sha256()
    for f in deps:
        with open(f, "rb") as fh:
            h.update(fh.read())
    libdir = os.path.join(ROOT, "motionplanning_5d_m_b200")
    so = os.path.join(tempfile.gettempdir(), "cfs_mex_check_%d_%s.so" % (os.getuid(), h.hexdigest()[:16]))
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


def call_mex_check(h, ROBOT, robot, obs, nj, what, a, b, c=None, H=0, eta=1e-3, margin_is_D=True):
    """cfs_mex('check', ROBOT, obs, sys_info, what, ...): a, b, c as (N, rows) arrays (row i = MATLAB column i)"""
    f = lambda v: np.ascontiguousarray(v, dtype=np.float64)
    DH = np.asfortranarray(robot["DH"], dtype=np.float64)
    cap = np.asfortranarray(np.stack([np.asarray(robot["cap"][i]["p"], dtype=np.float64)[:, :2] for i in range(nj)], axis=2))
    seg = np.asfortranarray(np.stack([np.asarray(o["l"], dtype=np.float64) for o in obs], axis=2))
    D, eps, base = f([o["D"] for o in obs]), f([o["epsilon"] for o in obs]), f(np.asarray(robot["base"]).reshape(-1))
    a, b = f(a), f(b)
    c = None if c is None else f(c)
    N = a.shape[0]
    out = dict(verdict=np.zeros(N, dtype=np.int32), where=np.zeros(N), cmin=np.zeros(N), evals=np.zeros(N, dtype=np.int32))
    h.mexh_check.restype = C.c_int
    rc = h.mexh_check(ROBOT.encode(), C.c_int(nj), C.c_int(DH.shape[0]), _dp(DH), _dp(base), _dp(cap), None,
                      C.c_double(robot["delta_t"]), C.c_int(len(obs)), _dp(seg), _dp(D), _dp(eps), what.encode(), C.c_int(N),
                      C.c_int(H), _dp(a), _dp(b), _dp(c), C.c_double(eta), C.c_int(1 if margin_is_D else 0),
                      _dp(out["verdict"]), _dp(out["where"]), _dp(out["cmin"]), _dp(out["evals"]))
    if rc:
        raise RuntimeError(h.mexh_last_error().decode())
    return out


def test_check_through_the_gateway(harness, ctx, oracle):
    robot = M.robotproperty2("M16iB")
    obs = [synthetic.OBS_M16IB]
    r = dict(robot, name="M16iB")
    ctx.set_robot(r, 5)
    ctx.set_obstacles(obs)
    a, b = random_edges(np.random.default_rng(2), 3000, synthetic.SAMPLE_OFF, synthetic.REGION_S)
    ref = ctx.check_edges(a, b)
    out = call_mex_check(harness, "M16iB", robot, obs, 5, "edges", a, b)
    assert np.array_equal(out["verdict"], ref["verdict"]) and np.array_equal(out["where"], ref["s_hit"])
    assert np.array_equal(out["cmin"], ref["cmin"]) and np.array_equal(out["evals"], ref["evals"])

    cfg = common.batch_m16ib(oracle, 64, horizon=30)
    s = cfg["sys_info"]
    ctx.set_cost(s["H"], s["QQ"], s["lim"], s["MAX_input"])
    sol = ctx.solve_batch(cfg["x0"], cfg["ff"], cfg["caug"], cfg["xref"], s["epsilon_O"], s["MAX_O_ITER"])
    ref = ctx.check_trajectories(cfg["x0"], sol["x"], sol["u"], eta=2e-3)
    out = call_mex_check(harness, "M16iB", robot, obs, 5, "trajectory", cfg["x0"], sol["x"], sol["u"], H=s["H"], eta=2e-3)
    assert np.array_equal(out["verdict"], ref["verdict"]) and np.array_equal(out["where"], ref["t_hit"])
    assert np.array_equal(out["cmin"], ref["cmin"]) and np.array_equal(out["evals"], ref["evals"])
    with pytest.raises(RuntimeError, match="cfs_check_edges failed"):
        call_mex_check(harness, "M16iB", robot, obs, 5, "edges", a[:2], b[:2], eta=0.0)
