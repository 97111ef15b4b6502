"""-m gpu : the 'solve_checked' command of the MEX gateway (matlab/cfs_mex.cpp, compiled against tests/mex_stub/) returns bit for
bit what Context.solve_checked returns."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np
import pytest

from tests import common

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


@pytest.fixture(scope="module")
def harness():
    """tests/mex_stub/checked_harness.cpp + matlab/cfs_mex.cpp, built into the temporary directory (keyed by the sources)"""
    src = [os.path.join(HERE, "mex_stub", "checked_harness.cpp"), os.path.join(ROOT, "matlab", "cfs_mex.cpp")]
    deps = src + [os.path.join(HERE, "mex_stub", f) for f in ("harness.cpp", "mex.h")] + [os.path.join(ROOT, "include", "cfs_b200.h")]
    h = hashlib.sha256()
    for f in deps:
        with open(f, "rb") as fh:
            h.update(fh.read())
    libdir = os.path.join(ROOT, "motionplanning_5d_m_b200")
    so = os.path.join(tempfile.gettempdir(), "cfs_mex_checked_%d_%s.so" % (os.getuid(), h.hexdigest()[:16]))
    if not os.path.exists(so):
        tmp = so + ".%d.tmp" % os.getpid()
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-I", os.path.join(HERE, "mex_stub"), "-I",
                               os.path.join(ROOT, "include"), "-o", tmp] + src + ["-L", libdir, "-lcfs_b200", "-Wl,-rpath," + libdir])
        os.replace(tmp, so)
    lib = C.CDLL(so)
    lib.mexh_last_error.restype = C.c_char_p
    lib.mexh_solve_checked.restype = C.c_int
    yield lib
    lib.mexh_shutdown()


def _dp(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def call_mex_checked(h, ROBOT, robot, obs, s, x0, ff, caug, xref, eta=1e-3, rounds=4, gain=2.0):
    nj, H = int(s["njoint"]), int(s["H"])
    n, B, K = nj * H, x0.shape[0], int(s["MAX_O_ITER"])
    f = lambda a: np.ascontiguousarray(a, dtype=np.float64)
    DH = np.asfortranarray(robot["DH"], dtype=np.float64)
    cap = np.asfortranarray(np.stack([np.asarray(robot["cap"][i]["p"], dtype=np.float64)[:, :2] for i in range(nj)], axis=2))
    seg = np.asfortranarray(np.stack([np.asarray(o["l"], dtype=np.float64) for o in obs], axis=2))
    keep = dict(D=f([o["D"] for o in obs]), eps=f([o["epsilon"] for o in obs]), base=f(np.asarray(robot["base"]).reshape(-1)),
                QQ=f(s["QQ"].T), lim=f(s["lim"]), mi=f(s["MAX_input"]), x0=f(x0), ff=f(ff), caug=f(caug), xref=f(xref))
    out = dict(u=np.zeros((B, n)), x=np.zeros((B, 2 * n)), cost_hist=np.zeros((B, K)), e_u_hist=np.zeros((B, K)),
               iters=np.zeros(B, dtype=np.int32), status=np.zeros(B, dtype=np.int32), verdict=np.zeros(B, dtype=np.int32),
               t_hit=np.zeros(B), cmin=np.zeros(B), rounds_used=np.zeros(B, dtype=np.int32), margin_off=np.zeros((B, len(obs), H)))
    rc = h.mexh_solve_checked(b"CFS", b"num_jac", ROBOT.encode(), C.c_int(nj), C.c_int(H), C.c_int(B), C.c_int(DH.shape[0]), _dp(DH),
                              _dp(keep["base"]), _dp(cap), None, C.c_double(robot["delta_t"]), C.c_int(len(obs)), _dp(seg),
                              _dp(keep["D"]), _dp(keep["eps"]), _dp(keep["QQ"]), _dp(keep["lim"]), _dp(keep["mi"]), _dp(keep["x0"]),
                              _dp(keep["ff"]), _dp(keep["caug"]), _dp(keep["xref"]), C.c_double(s["epsilon_O"]), C.c_int(K),
                              C.c_double(eta), C.c_int(rounds), C.c_double(gain), *(_dp(out[k]) for k in (
                                  "u", "x", "cost_hist", "e_u_hist", "iters", "status", "verdict", "t_hit", "cmin", "rounds_used",
                                  "margin_off")))
    if rc:
        raise RuntimeError(h.mexh_last_error().decode())
    return out


def test_solve_checked_through_the_gateway(harness, ctx, oracle):
    cfg = common.batch_m16ib(oracle, 256)
    s, obs = cfg["sys_info"], cfg["obs"]
    r = dict(cfg["robot"], name="M16iB")
    ctx.set_robot(r, 5)
    ctx.set_obstacles(obs)
    ctx.set_cost(s["H"], s["QQ"], s["lim"], s["MAX_input"])
    args = (cfg["x0"], cfg["ff"], cfg["caug"], cfg["xref"])
    ref = ctx.solve_checked(*args, s["epsilon_O"], s["MAX_O_ITER"], eta=1e-3, rounds=3, gain=2.0)
    out = call_mex_checked(harness, "M16iB", cfg["robot"], obs, s, *args, eta=1e-3, rounds=3, gain=2.0)
    for k in ref:
        assert np.array_equal(out[k], ref[k], equal_nan=True), k
    assert (ref["rounds_used"] > 0).any()
    with pytest.raises(RuntimeError, match="cfs_solve_checked failed"):
        call_mex_checked(harness, "M16iB", cfg["robot"], obs, s, *args, gain=0.0)
