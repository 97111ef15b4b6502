"""GPU tests of the joint position limits (cfs_set_joint_limits): wide limits change nothing bit for bit, active limits match
the limits oracle (tests/limits_oracle.c) under the parity rules of DESIGN.md section 2, and every returned trajectory with
status < 2 holds the limits at its waypoints."""
import numpy as np
import pytest

import motionplanning_5d_m_b200 as M
from motionplanning_5d_m_b200 import _lib, problem
from tests import common
from tests import limits_oracle as L
from tests.test_gpu_parity import BULK_DEFAULT, BULK_MODES, _set
from tests.test_limits import assert_binding, assert_within_limits, inside_box, limit_box
from tests.test_oracle import _golden_cases

pytestmark = pytest.mark.gpu
KEYS = ("u", "x", "cost_hist", "e_u_hist", "iters", "status")
LAUNCHES = {"lockstep": 44, "lockstep_warp": 64, "cta": 6, "warp_noscreen": 6, "warp_screen1": 8, "warp_screen3": 12}
WIDE = (np.full(5, -1e3), np.full(5, 1e3))


def _same(a, b, keys=KEYS):
    for k in keys:
        assert np.array_equal(a[k], b[k], equal_nan=True), k


@pytest.fixture(scope="module")
def lctx():
    """a context of its own: the session context never carries limits"""
    c = M.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def active(oracle):
    """the headline batch's problems with start and goal inside the limit box, and the limits oracle's solve with that box
    (and its FMA twin's)"""
    cfg = common.batch_m16ib(oracle, 4096)
    idx = inside_box(cfg)
    s, obs = cfg["sys_info"], cfg["obs"]
    args = tuple(np.ascontiguousarray(cfg[k][idx]) for k in ("x0", "ff", "caug", "xref"))
    P = common.oracle_problem(oracle, "M16iB", obs, s)
    lo, hi = limit_box()
    ref = L.solve_batch_lim(P, *args, lo, hi, nthreads=16)
    twin = L.solve_batch_lim(P, *args, lo, hi, nthreads=16, twin=True)
    return dict(cfg=cfg, idx=idx, args=args, ref=ref, twin=twin, P=P)


def _compare_limits(out, ref, twin, tol=1e-6):
    """status, iterations and touch flag equal; 1e-6 on u / x / cost elsewhere, except where the oracle and its FMA twin
    disagree by more than 1e-8 (DESIGN.md section 2)"""
    assert (out["status"] == ref["status"]).all(), np.nonzero(out["status"] != ref["status"])[0][:10]
    assert (out["iters"] == ref["iters"]).all()
    ok = (ref["status"] & 0xFF) < 2
    cond = np.maximum(np.abs(ref["x"] - twin["x"]).max(axis=1), np.abs(ref["u"] - twin["u"]).max(axis=1)) <= 1e-8
    sel = ok & cond
    dx = np.abs(out["x"] - ref["x"]).max(axis=1)
    du = np.abs(out["u"] - ref["u"]).max(axis=1)
    assert (dx[sel] < tol).all() and (du[sel] < tol).all(), (dx[sel].max(), du[sel].max())
    for b in np.nonzero(sel)[0]:
        it = ref["iters"][b]
        assert np.all(np.abs(out["cost_hist"][b, :it] - ref["cost_hist"][b, :it]) <= tol * np.abs(ref["cost_hist"][b, :it]))
    return sel.sum(), ok.sum()


@pytest.mark.parametrize("mode", list(BULK_MODES))
def test_wide_limits_bitwise(lctx, oracle, mode):
    """limits at +-1e3 rad: cfs_solve_batch bit for bit, with the plain solve's launch count"""
    cfg = common.batch_m16ib(oracle, 192)
    s, obs = cfg["sys_info"], cfg["obs"]
    args = (cfg["x0"], cfg["ff"], cfg["caug"], cfg["xref"], s["epsilon_O"], s["MAX_O_ITER"])
    for k, v in BULK_MODES[mode].items():
        lctx.set_option(k, v)
    try:
        _set(lctx, "M16iB", cfg["robot"], obs, s)
        ref = lctx.solve_batch(*args)
        lctx.set_joint_limits(*WIDE)
        out = lctx.solve_batch(*args)
        launches = lctx.stats()["launches"]
        inf = (np.full(5, -np.inf), np.full(5, np.inf))
        lctx.set_joint_limits(*inf)
        out_inf = lctx.solve_batch(*args)
    finally:
        lctx.set_joint_limits(None, None)
        for k, v in BULK_DEFAULT.items():
            lctx.set_option(k, v)
    _same(out, ref)
    _same(out_inf, ref)
    assert launches == LAUNCHES.get(mode, 10)


@pytest.mark.parametrize("name", ["main_fanuc_psgcfs", "m16ib_script_derivest", "main_2l_cfs"])
def test_wide_limits_psgcfs_derivest(lctx, oracle, name):
    ROBOT, obs, s, solver, grad, noise = _golden_cases(oracle)[name]
    nj = 2 if ROBOT == "2L" else 5
    _set(lctx, ROBOT, s["robot"], obs)
    lctx.set_cost(s["H"], s["QQ"], s.get("lim"), s["MAX_input"] if solver == 0 else None)
    args = (s["xR"][:, 0][None], s["ff"][None], np.array([s["caug"]]), s["x_"][None], s["epsilon_O"], s["MAX_O_ITER"])
    kw = dict(solver=solver, grad=grad, noise=noise, alpha=s.get("alpha", 0.0))
    ref = lctx.solve_batch(*args, **kw)
    lctx.set_joint_limits(np.full(nj, -1e3), np.full(nj, 1e3))
    out = lctx.solve_batch(*args, **kw)
    lctx.set_joint_limits(None, None)
    _same(out, ref)


def test_wide_limits_psgcfs_batch(lctx, oracle):
    """PSGCFS on a seeded batch (H = 30, 8 noisy projection steps): wide limits are bit for bit the plain solve"""
    B, H, K = 96, 30, 8
    cfg = common.batch_m16ib(oracle, B, horizon=H)
    s = dict(cfg["sys_info"])
    s["alpha"] = 1.0 / np.linalg.svd(s["QQ"], compute_uv=False).max()
    noise = np.random.default_rng(5).normal(0.0, 0.1, size=(B, K, H * 5))
    _set(lctx, "M16iB", cfg["robot"], cfg["obs"], s, bounds=False)
    args = (cfg["x0"], cfg["ff"], cfg["caug"], cfg["xref"], s["epsilon_O"], K)
    kw = dict(solver=_lib.SOLVER_PSGCFS, noise=noise, alpha=s["alpha"])
    ref = lctx.solve_batch(*args, **kw)
    lctx.set_joint_limits(*WIDE)
    out = lctx.solve_batch(*args, **kw)
    lctx.set_joint_limits(None, None)
    _same(out, ref)


@pytest.mark.parametrize("mode", list(BULK_MODES))
def test_active_limits_vs_oracle(lctx, active, mode):
    """the limit box on >= 256 headline problems: parity with the limits oracle, and the limits hold at every waypoint"""
    cfg, a = active["cfg"], active
    s = cfg["sys_info"]
    assert len(a["idx"]) >= 256
    lo, hi = limit_box()
    for k, v in BULK_MODES[mode].items():
        lctx.set_option(k, v)
    try:
        _set(lctx, "M16iB", cfg["robot"], cfg["obs"], s)
        lctx.set_joint_limits(lo, hi)
        out = lctx.solve_batch(*a["args"], s["epsilon_O"], s["MAX_O_ITER"])
    finally:
        lctx.set_joint_limits(None, None)
        for k, v in BULK_DEFAULT.items():
            lctx.set_option(k, v)
    n_cmp, n_ok = _compare_limits(out, a["ref"], a["twin"])
    assert n_cmp >= 0.9 * n_ok, (n_cmp, n_ok)
    assert_within_limits(out["x"], out["status"], 5, lo, hi)
    assert_binding(out["x"], out["status"], 5, lo, hi)  # upper and lower rows bind in this tier


def test_active_limits_derivest_psgcfs(lctx, oracle, active):
    """DERIVEST gradients and one PSGCFS projection step with the limit box against the limits oracle"""
    cfg, a = active["cfg"], active
    s = dict(cfg["sys_info"])
    lo, hi = limit_box()
    args = tuple(x[:128] for x in a["args"])
    _set(lctx, "M16iB", cfg["robot"], cfg["obs"], s)
    lctx.set_joint_limits(lo, hi)
    P = common.oracle_problem(oracle, "M16iB", cfg["obs"], s, grad=1)
    ref = L.solve_batch_lim(P, *args, lo, hi, nthreads=16)
    twin = L.solve_batch_lim(P, *args, lo, hi, nthreads=16, twin=True)
    out = lctx.solve_batch(*args, s["epsilon_O"], s["MAX_O_ITER"], grad=_lib.GRAD_DERIVEST)
    _compare_limits(out, ref, twin)
    assert_within_limits(out["x"], out["status"], 5, lo, hi)
    assert_binding(out["x"], out["status"], 5, lo, hi)
    # PSGCFS: one projection step from identical inputs
    s["alpha"] = 1.0 / np.linalg.svd(s["QQ"], compute_uv=False).max()
    s["MAX_O_ITER"] = 1
    noise = np.random.default_rng(5).normal(0.0, 0.1, size=(128, 1, s["H"] * 5))
    _set(lctx, "M16iB", cfg["robot"], cfg["obs"], s, bounds=False)
    lctx.set_joint_limits(lo, hi)
    P = common.oracle_problem(oracle, "M16iB", cfg["obs"], s, solver=1)
    ref = L.solve_batch_lim(P, *args, lo, hi, noise=noise, nthreads=16)
    twin = L.solve_batch_lim(P, *args, lo, hi, noise=noise, nthreads=16, twin=True)
    out = lctx.solve_batch(*args, s["epsilon_O"], 1, solver=_lib.SOLVER_PSGCFS, noise=noise, alpha=s["alpha"])
    lctx.set_joint_limits(None, None)
    _compare_limits(out, ref, twin)
    assert_within_limits(out["x"], out["status"], 5, lo, hi)


def test_entry_points_and_state(lctx, oracle, active):
    """device / async forms equal the host form bit for bit; get_con rows; clearing the limits gives a fresh context's solve bit for bit; determinism and permutation invariance"""
    import torch
    cfg, a = active["cfg"], active
    s = cfg["sys_info"]
    lo, hi = limit_box()
    args = tuple(x[:256] for x in a["args"])
    _set(lctx, "M16iB", cfg["robot"], cfg["obs"], s)
    lctx.set_joint_limits(lo, hi)
    out = lctx.solve_batch(*args, s["epsilon_O"], s["MAX_O_ITER"])
    again = lctx.solve_batch(*args, s["epsilon_O"], s["MAX_O_ITER"])
    _same(again, out)
    perm = np.random.default_rng(2).permutation(256)
    pout = lctx.solve_batch(*(x[perm] for x in args), s["epsilon_O"], s["MAX_O_ITER"])
    _same({k: pout[k] for k in KEYS}, {k: out[k][perm] for k in KEYS})
    # device pointers
    dev = torch.device("cuda:0")
    hin = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in zip(("x0", "ff", "caug", "xref"), args)}
    B, n, K = 256, lctx.n, s["MAX_O_ITER"]
    o = dict(u=torch.zeros(B, n, dtype=torch.float64, device=dev), x=torch.zeros(B, 2 * n, dtype=torch.float64, device=dev),
             cost=torch.zeros(B, K, dtype=torch.float64, device=dev), eu=torch.zeros(B, K, dtype=torch.float64, device=dev),
             iters=torch.zeros(B, dtype=torch.int32, device=dev), status=torch.zeros(B, dtype=torch.int32, device=dev))
    lctx.solve_batch_ptr(B, hin["x0"].data_ptr(), hin["ff"].data_ptr(), hin["caug"].data_ptr(), hin["xref"].data_ptr(),
                         s["epsilon_O"], K, o["u"].data_ptr(), o["x"].data_ptr(), o["cost"].data_ptr(), o["eu"].data_ptr(),
                         o["iters"].data_ptr(), o["status"].data_ptr(), device=True, sync=True)
    got = dict(u=o["u"].cpu().numpy(), x=o["x"].cpu().numpy(), cost_hist=o["cost"].cpu().numpy(),
               e_u_hist=o["eu"].cpu().numpy(), iters=o["iters"].cpu().numpy(), status=o["status"].cpu().numpy())
    _same(got, out)
    # get_con rows against the limits oracle
    P = a["P"]
    b = 3
    Ag, bg = lctx.get_con(args[0][b], out["x"][b], out["u"][b])
    Ao, bo = L.get_con_lim(P, args[0][b], out["x"][b], out["u"][b], lo, hi)
    m = Ao.shape[0] - 2 * P.n
    assert Ag.shape == Ao.shape
    assert np.array_equal(Ag[m:], Ao[m:]) and np.array_equal(bg[m:], bo[m:])
    np.testing.assert_allclose(Ag[:m], Ao[:m], rtol=1e-6, atol=1e-9)
    # asynchronous host-pointer form
    ho = {k: np.zeros_like(out[k]) for k in KEYS}
    hargs = [np.ascontiguousarray(x) for x in args]
    lctx.solve_batch_ptr(B, *(x.ctypes.data for x in hargs), s["epsilon_O"], K, *(ho[k].ctypes.data for k in KEYS), sync=False)
    lctx.wait()
    _same(ho, out)
    # clearing: a fresh context's solve bit for bit; set_robot clears too
    _set(lctx, "M16iB", cfg["robot"], cfg["obs"], s)
    lctx.set_joint_limits(lo, hi)
    lctx.set_joint_limits(None, None)
    cleared = lctx.solve_batch(*args, s["epsilon_O"], s["MAX_O_ITER"])
    fresh = M.Context(0)
    try:
        _set(fresh, "M16iB", cfg["robot"], cfg["obs"], s)
        ref = fresh.solve_batch(*args, s["epsilon_O"], s["MAX_O_ITER"])
    finally:
        fresh.close()
    _same(cleared, ref)
    lctx.set_joint_limits(lo, hi)
    _set(lctx, "M16iB", cfg["robot"], cfg["obs"], s)
    _same(lctx.solve_batch(*args, s["epsilon_O"], s["MAX_O_ITER"]), ref)


def test_errors(oracle):
    """CFS_E_STATE without a robot; CFS_E_ARG for one NULL pointer, a NaN entry, qmin > qmax, qmin = +inf or qmax = -inf"""
    cfg = common.batch_m16ib(oracle, 4)
    c = M.Context(0)
    try:
        with pytest.raises(M.CfsError, match="cfs_set_robot first"):
            c.set_joint_limits(None, None)
        _set(c, "M16iB", cfg["robot"], cfg["obs"])
        z = np.ascontiguousarray(np.zeros(5))
        for lo, hi in [(z, None), (None, z)]:
            rc = c._lib.cfs_set_joint_limits(c._h, _lib._dp(lo), _lib._dp(hi))
            assert rc == -1, rc
        for lo, hi in [(np.full(5, np.nan), np.zeros(5)), (np.zeros(5), np.full(5, np.nan)), (np.ones(5), np.zeros(5)),
                       (np.full(5, np.inf), np.full(5, np.inf)), (np.full(5, -np.inf), np.full(5, -np.inf))]:
            with pytest.raises(M.CfsError, match="cfs_set_joint_limits"):
                c.set_joint_limits(lo, hi)
        c.set_joint_limits(np.full(5, -np.inf), np.zeros(5))  # one-sided limits are accepted
        c.set_joint_limits(None, None)
    finally:
        c.close()


def test_checked_solve_with_limits(lctx, active):
    """every returned solution with status < 2 holds the limits; CLEAR verdicts carry their guarantee (checked on a dense sample
    by the checked solve's own tests; here: the verdict comes from the continuous check of the returned trajectory)"""
    cfg, a = active["cfg"], active
    s = cfg["sys_info"]
    lo, hi = limit_box()
    _set(lctx, "M16iB", cfg["robot"], cfg["obs"], s)
    lctx.set_joint_limits(lo, hi)
    out = lctx.solve_checked(*a["args"], s["epsilon_O"], s["MAX_O_ITER"], eta=1e-3, rounds=4, gain=2.0)
    ck = lctx.check_trajectories(a["args"][0], out["x"], out["u"], eta=1e-3, margin_is_D=False)
    lctx.set_joint_limits(None, None)
    assert_within_limits(out["x"], out["status"], 5, lo, hi)
    assert np.array_equal(ck["verdict"], out["verdict"])


def test_start_goal_routes_async_with_limits(lctx, oracle, active):
    """cfs_solve_start_goal[_async] and cfs_solve_routes[_var][_async] with limits.  No entry returns the inputs these entries
    build on the device, so: wide limits reproduce each entry's plain solve bit for bit; the async forms equal the synchronous
    ones bit for bit; routes and routes_var (full lengths) agree bit for bit; active limits hold and bind; start_goal agrees with
    solve_batch on the host-built problem (1e-6: the device-built QQ differs in the last bits)."""
    cfg, a = active["cfg"], active
    s = cfg["sys_info"]
    lo, hi = limit_box()
    idx = a["idx"][:256]
    B, K, n = len(idx), s["MAX_O_ITER"], s["H"] * 5
    th0, thg = np.ascontiguousarray(cfg["theta0"][idx]), np.ascontiguousarray(cfg["thetag"][idx])
    _set(lctx, "M16iB", cfg["robot"], cfg["obs"])
    lctx.set_cost_blocks(s["H"], problem.Q_MAIN_FANUC, problem.R_MAIN_FANUC, 50.0, s["lim"], s["MAX_input"])
    routes = np.ascontiguousarray(np.stack([th0, 0.5 * (th0 + thg), thg], axis=1))  # (B, 3, nj) straight polylines
    rl = np.full(B, 3, dtype=np.int32)
    ek = (s["epsilon_O"], K)

    def outs():
        return dict(u=np.zeros((B, n)), x=np.zeros((B, 2 * n)), cost_hist=np.full((B, K), np.nan),
                    e_u_hist=np.full((B, K), np.nan), iters=np.zeros(B, dtype=np.int32), status=np.zeros(B, dtype=np.int32))

    def ptrs(o):
        return [o[k].ctypes.data for k in KEYS]

    try:
        sg0, rt0 = lctx.solve_start_goal(th0, thg, *ek), lctx.solve_routes(routes, *ek)
        lctx.set_joint_limits(*WIDE)
        _same(lctx.solve_start_goal(th0, thg, *ek), sg0)
        _same(lctx.solve_routes(routes, *ek), rt0)
        lctx.set_joint_limits(lo, hi)
        sg = lctx.solve_start_goal(th0, thg, *ek)
        o = outs()
        lctx.solve_start_goal_ptr(B, th0.ctypes.data, thg.ctypes.data, *ek, *ptrs(o), sync=False)
        lctx.wait()
        _same(o, sg)
        rt = lctx.solve_routes(routes, *ek)
        _same(lctx.solve_routes_var(routes, rl, *ek), rt)
        o = outs()
        lctx.solve_routes_var_ptr(B, 3, rl.ctypes.data, routes.ctypes.data, *ek, *ptrs(o), sync=False)
        lctx.wait()
        _same(o, rt)
        lctx.set_cost(s["H"], s["QQ"], s["lim"], s["MAX_input"])
        ref = lctx.solve_batch(*(x[:B] for x in a["args"]), *ek)
    finally:
        lctx.set_joint_limits(None, None)
    for r in (sg, rt):
        assert_within_limits(r["x"], r["status"], 5, lo, hi)
        assert_binding(r["x"], r["status"], 5, lo, hi)
    assert (sg["status"] == ref["status"]).all() and (sg["iters"] == ref["iters"]).all()
    ok = (ref["status"] & 0xFF) < 2
    assert np.abs(sg["x"][ok] - ref["x"][ok]).max() < 1e-6 and np.abs(sg["u"][ok] - ref["u"][ok]).max() < 1e-6
