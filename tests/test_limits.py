"""CPU tests of the joint position limits' restatement (tests/limits_oracle.c on a copy of oracle/cfs_oracle.c): wide limits
change nothing, active limits bind and hold at every waypoint, and the limit rows of get_con are the roll-out's positions."""
import numpy as np
import pytest

from motionplanning_5d_m_b200 import synthetic
from tests import common
from tests import limits_oracle as L
from tests.test_oracle import _golden_cases

BOX = 0.5  # active limits: SAMPLE_OFF +- BOX * REGION_S on the LIMITED joints
LIMITED = [2, 4]
MIN_SHARE = 0.3  # least share of the status < 2 problems with an upper, and with a lower, row binding (measured: 0.48 / 0.40)


def _same(a, b):
    for k in ("u", "x", "cost_hist", "e_u_hist", "iters", "status"):
        assert np.array_equal(a[k], b[k], equal_nan=True), k


@pytest.mark.parametrize("name", ["main_fanuc_cfs", "main_fanuc_psgcfs", "main_2l_cfs", "m16ib_script_derivest",
                                  "m16ib_script_alt_numjac", "rrtstar_cfs"])
def test_wide_limits_equal_oracle(oracle, name):
    """limits at +-1e3 rad, and infinite ones, reproduce the oracle bit for bit on the golden cases"""
    ROBOT, obs, s, solver, grad, noise = _golden_cases(oracle)[name]
    P = common.oracle_problem(oracle, ROBOT, obs, s, solver=solver, grad=grad)
    args = (s["xR"][:, 0][None], s["ff"][None], np.array([s["caug"]]), s["x_"][None])
    ref = P.solve_batch(*args, noise=noise)
    nj = P.nj
    _same(L.solve_batch_lim(P, *args, None, None, noise=noise), ref)
    _same(L.solve_batch_lim(P, *args, np.full(nj, -1e3), np.full(nj, 1e3), noise=noise), ref)
    _same(L.solve_batch_lim(P, *args, np.full(nj, -np.inf), np.full(nj, np.inf), noise=noise), ref)


def limit_box():
    """the active limits: joints 3 and 5 (where the headline solutions swing furthest) limited to SAMPLE_OFF +- 0.5 REGION_S,
    the other joints unlimited (infinite bounds: rows that can never be violated)"""
    lo, hi = np.full(5, -np.inf), np.full(5, np.inf)
    lo[LIMITED] = (synthetic.SAMPLE_OFF - BOX * synthetic.REGION_S)[LIMITED]
    hi[LIMITED] = (synthetic.SAMPLE_OFF + BOX * synthetic.REGION_S)[LIMITED]
    return lo, hi


def inside_box(cfg):
    """problems of a headline batch whose start lies inside the limits.  Their goal may lie outside: the cost then pulls the
    trajectory onto the limit, so upper and lower rows bind in a large share of them."""
    lo, hi = limit_box()
    return np.nonzero(((cfg["theta0"] >= lo) & (cfg["theta0"] <= hi)).all(axis=1))[0]


def binding_shares(x, status, nj, lo, hi, tol=1e-9):
    """fractions of the problems with status < 2 that end with a joint on its upper / on its lower limit (within tol) at some
    waypoint: an upper / a lower position row active in the final QP"""
    th = L.waypoint_theta(x, nj)
    good = (status & 0xFF) < 2
    up = (np.abs(th - hi) <= tol).any(axis=(1, 2))
    dn = (np.abs(th - lo) <= tol).any(axis=(1, 2))
    return up[good].mean(), dn[good].mean()


def assert_within_limits(x, status, nj, lo, hi, tol=1e-9):
    th = L.waypoint_theta(x, nj)
    good = (status & 0xFF) < 2
    assert (th[good] <= hi + tol).all() and (th[good] >= lo - tol).all(), \
        (np.max(th[good] - hi), np.max(lo - th[good]))


def assert_binding(x, status, nj, lo, hi, share=MIN_SHARE):
    up, dn = binding_shares(x, status, nj, lo, hi)
    assert up >= share and dn >= share, (up, dn)


def test_active_limits_headline(oracle):
    """The headline batch with the active limits, problems whose start lies inside them: every solution with status < 2 holds
    the limits at waypoints 1..H within 1e-9, and upper rows as well as lower rows bind in a large share of them.  Measured on
    1024 drawn problems: 248 qualify, 197 end with status < 2; 48 % of those end on an upper limit, 40 % on a lower one.
    Without limits, the same solutions leave the limits."""
    cfg = common.batch_m16ib(oracle, 1024)
    s, obs = cfg["sys_info"], cfg["obs"]
    idx = inside_box(cfg)
    P = common.oracle_problem(oracle, "M16iB", obs, s)
    args = (cfg["x0"][idx], cfg["ff"][idx], cfg["caug"][idx], cfg["xref"][idx])
    lo, hi = limit_box()
    out = L.solve_batch_lim(P, *args, lo, hi)
    assert len(idx) >= 200 and ((out["status"] & 0xFF) < 2).sum() >= 150
    assert_within_limits(out["x"], out["status"], 5, lo, hi)
    assert_binding(out["x"], out["status"], 5, lo, hi)
    free = P.solve_batch(*args)
    th = L.waypoint_theta(free["x"], 5)
    outside = ((th > hi + 1e-6) | (th < lo - 1e-6)).any(axis=(1, 2))[(free["status"] & 0xFF) < 2].mean()
    assert outside >= 2 * MIN_SHARE, outside


def test_get_con_limit_rows(oracle):
    """the appended rows: A_up u - b_up = theta - qmax and A_dn u - b_dn = qmin - theta at the roll-out of u"""
    cfg = common.batch_m16ib(oracle, 4)
    s, obs = cfg["sys_info"], cfg["obs"]
    P = common.oracle_problem(oracle, "M16iB", obs, s)
    lo, hi = limit_box()
    rng = np.random.default_rng(3)
    u = rng.normal(0, 0.3, P.n)
    x0 = cfg["x0"][1]
    # roll-out as the oracle does it (CFS_FANUC.m:90-94)
    dt, nj = s["robot"]["delta_t"], 5
    th, om, x = x0[:nj].copy(), x0[nj:].copy(), []
    for i in range(s["H"]):
        uk = u[i * nj:(i + 1) * nj]
        th, om = (th + dt * om) + (0.5 * dt * dt) * uk, om + dt * uk
        x.append(np.concatenate([th, om]))
    x = np.concatenate(x)
    A0, b0 = P.get_con(x0, x, u)[:2]
    A, b = L.get_con_lim(P, x0, x, u, lo, hi)
    m, n = A0.shape[0], P.n
    assert A.shape == (m + 2 * n, n) and np.array_equal(A[:m], A0) and np.array_equal(b[:m], b0)
    theta = L.waypoint_theta(x[None], nj)[0].reshape(-1)
    np.testing.assert_allclose(A[m:m + n] @ u - b[m:m + n], theta - np.tile(hi, s["H"]), atol=1e-12)
    np.testing.assert_allclose(A[m + n:] @ u - b[m + n:], np.tile(lo, s["H"]) - theta, atol=1e-12)


def _np_get_con_with_limits(orig, lo, hi):
    """tests/np_restatement.get_con followed by the limit rows of the finite bounds, built from its own Baug / Aaug: theta rows
    of Baug for waypoints 1..H, right-hand sides qmax - Aaug_theta x0 and Aaug_theta x0 - qmin"""
    def get_con(x_, u, x0, robot, obs_list, kind, Aaug, Baug, lim, H, nj, margin_key):
        A, b = orig(x_, u, x0, robot, obs_list, kind, Aaug, Baug, lim, H, nj, margin_key)
        ns = 2 * nj
        Bt = np.vstack([Baug[ns * i:ns * i + nj] for i in range(H)])
        fm = np.concatenate([Aaug[ns * i:ns * i + nj] @ x0 for i in range(H)])
        Al, bl = np.vstack([Bt, -Bt]), np.concatenate([np.tile(hi, H) - fm, fm - np.tile(lo, H)])
        fin = np.isfinite(bl)  # an infinite bound has no row
        return np.vstack([A, Al[fin]]), np.concatenate([b, bl[fin]])
    return get_con


def test_limits_oracle_against_numpy_restatement(oracle, monkeypatch):
    """the limits oracle and the numpy restatement (interior-point QP on dense rows: an independent solver family) agree to
    1e-7 on u and x_ with identical iteration counts, on two headline problems whose limited solution ends on an upper
    limit, two on a lower limit and one on neither"""
    from tests import np_restatement as NP
    cfg = common.batch_m16ib(oracle, 1024)
    s, obs = cfg["sys_info"], cfg["obs"]
    idx = inside_box(cfg)
    P = common.oracle_problem(oracle, "M16iB", obs, s)
    lo, hi = limit_box()
    args = (cfg["x0"][idx], cfg["ff"][idx], cfg["caug"][idx], cfg["xref"][idx])
    out = L.solve_batch_lim(P, *args, lo, hi)
    th = L.waypoint_theta(out["x"], 5)
    good = (out["status"] & 0xFF) < 2
    up = (np.abs(th - hi) <= 1e-9).any(axis=(1, 2)) & good
    dn = (np.abs(th - lo) <= 1e-9).any(axis=(1, 2)) & good
    free = good & ~up & ~dn
    pick = list(np.nonzero(up & ~dn)[0][:2]) + list(np.nonzero(dn & ~up)[0][:2]) + list(np.nonzero(free)[0][:1])
    assert len(pick) == 5
    monkeypatch.setattr(NP, "get_con", _np_get_con_with_limits(NP.get_con, lo, hi))
    rb = dict(cfg["robot"])
    rb["cap"] = [{"p": np.asarray(c["p"], dtype=np.float64)[:, :2]} for c in cfg["robot"]["cap"]]
    for k in pick:
        b = idx[k]
        sk = dict(s, xR=cfg["x0"][b][:, None], ff=cfg["ff"][b], caug=float(cfg["caug"][b]), x_=cfg["xref"][b])
        u, x_, cost_all, iters = NP.cfs_optimizer(sk, rb, obs, "M16iB")
        assert iters == out["iters"][k], (k, iters, out["iters"][k])
        assert np.abs(u - out["u"][k]).max() < 1e-7 and np.abs(x_ - out["x"][k]).max() < 1e-7, k
