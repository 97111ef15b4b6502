"""-m "not gpu": pins the CPU oracle against the reference's own known answers and an independent numpy restatement."""
import numpy as np
import pytest

import motionplanning_5d_m_b200 as M
from tests import common, np_restatement as NP


def test_distlinseg_doc_example(oracle):
    # Lib/functions/distLinSeg.m:15-18
    d, pts = oracle.dist_lin_seg([0, 0], [1, 1], [1, 0], [2, 0])
    assert abs(d - 0.7071) < 5e-5 and abs(d - np.sqrt(0.5)) < 1e-15
    assert np.allclose(pts, [[0.5, 0.5], [1, 0]], atol=0)


def test_distlinseg_branches(oracle):
    rng = np.random.default_rng(0)
    cases = []
    for _ in range(300):
        a, b, c, d = rng.normal(size=(4, 3))
        cases.append((a, b, c, d))
        cases.append((a, a, c, d))            # first segment is a point (distLinSeg.m:45-50)
        cases.append((a, b, c, c))            # second is a point (:39-44)
        cases.append((a, a, c, c))            # both points (:51-53)
        cases.append((a, b, c, c + 2.0 * (b - a)))  # parallel (:55-66)
    for a, b, c, d in cases:
        do, po = oracle.dist_lin_seg(a, b, c, d)
        dn, pn = NP.dist_lin_seg(a, b, c, d)
        assert abs(do - dn) < 1e-14
        assert np.abs(po.reshape(-1) - pn).max() < 1e-13


def test_derivest_known_answers(oracle):
    # derivest.m:163-174 : derivest(@exp,1) = 2.71828182845904 (15 digits shown)
    d, e, _ = oracle.derivest_named(0, 1.0)
    assert abs(d - 2.71828182845904) < 5e-14 and e < 1e-12
    # demo/derivest_demo.m:13 exp at 0 -> 1 ; :71 sinh central at 0 -> 1, err 1.0412e-15 ; :82 log at 1e-3 -> 1000
    assert abs(oracle.derivest_named(0, 0.0)[0] - 1.0) < 1e-13
    d, e, _ = oracle.derivest_named(2, 0.0)
    assert abs(d - 1.0) < 1e-14 and abs(e - 1.0412e-15) < 1e-19
    assert abs(oracle.derivest_named(3, 1e-3)[0] - 1000.0) < 1e-6
    # demo/derivest_demo.m:31 : sin at linspace(0,2*pi,13) -> cos
    for x in np.linspace(0, 2 * np.pi, 13):
        assert abs(oracle.derivest_named(1, x)[0] - np.cos(x)) < 1e-12


def test_derivest_vs_numpy_restatement(oracle):
    funs = {0: np.exp, 1: np.sin, 2: np.sinh}  # (log leaves the real line for x0-h*delta<0: MATLAB goes complex)
    rng = np.random.default_rng(1)
    for which, f in funs.items():
        for x in rng.uniform(0.05, 3.0, size=20):
            do, eo, fo = oracle.derivest_named(which, x)
            dn, en, fn = NP.derivest(lambda t: float(f(t)), x)
            # the error estimates are rounding noise, so the two implementations may select neighbouring steps:
            # the derivative itself agrees to ~1e-13 relative
            assert abs(do - dn) <= 1e-11 * max(1, abs(dn))


@pytest.mark.parametrize("ROBOT", ["M16iB", "M200i"])
def test_fk_dist_numjac_vs_numpy_restatement(oracle, ROBOT):
    rng = np.random.default_rng(2)
    robot = M.robotproperty2(ROBOT)
    r = oracle.robot(ROBOT)
    obs = np.array([[3.906, 3.906], [8.313, 8.313], [0.001, 1.938]])
    o6 = oracle.obs6(obs)
    for th in common.sampling_box(rng, 200):
        DH = robot["DH"][:5].copy()
        DH[:, 0] = th
        if ROBOT == "M200i":
            DH[1, 0] -= np.pi / 2
        pn = NP.cap_pos(robot["base"], DH, [c["p"] for c in robot["cap"]])
        po = oracle.cap_pos(r, th)
        for i in range(5):
            assert np.abs(po[i].T - pn[i]).max() < 1e-14
        dn, ln = NP.dist_arm(th, robot, obs, ROBOT)
        do, lo, _ = oracle.dist_arm(r, th, o6)
        assert abs(do - dn) < 1e-14 and lo == ln
        gn = NP.num_jac(lambda t: NP.dist_arm(t, robot, obs, ROBOT)[0], th)
        go = oracle.num_jac(r, th, o6)
        assert np.abs(go - gn).max() < 1e-9


def test_derivest_gradient_vs_numpy_restatement(oracle):
    rng = np.random.default_rng(3)
    robot = M.robotproperty2("M16iB")
    r = oracle.robot("M16iB")
    obs = np.array([[3.906, 3.906], [8.313, 8.313], [0.001, 1.938]])
    o6 = oracle.obs6(obs)

    def dist_link(th, lid):
        DH = robot["DH"][:5].copy()
        DH[:, 0] = th
        pos = NP.cap_pos(robot["base"], DH, [c["p"] for c in robot["cap"]])
        dis, pts = NP.dist_lin_seg(pos[lid - 1][:, 0], pos[lid - 1][:, 1], obs[:, 0], obs[:, 1])
        return dis if abs(dis) >= 1e-4 else -np.linalg.norm(pts[:3] - pos[lid - 1][:, 1])

    for th in common.sampling_box(rng, 12):
        _, lid, _ = oracle.dist_arm(r, th, o6)
        go = oracle.derivest_grad(r, th, o6, lid)
        for s in range(5):
            f = lambda x: dist_link(np.concatenate([th[:s], [x], th[s + 1:]]), lid)
            gn = NP.derivest(f, th[s])[0]
            assert abs(go[s] - gn) < 1e-9 * max(1.0, abs(gn)), (s, go[s], gn)


def test_qp_kkt_random(oracle):
    rng = np.random.default_rng(4)
    for trial in range(25):
        n, m = int(rng.integers(3, 30)), int(rng.integers(1, 60))
        Mx = rng.normal(size=(n, n))
        G = Mx @ Mx.T + 0.1 * np.eye(n)
        a = rng.normal(size=n) * 3
        Cm = rng.normal(size=(m, n))
        xf = rng.normal(size=n)
        d = Cm @ xf + rng.uniform(0.0, 1.0, size=m)  # xf strictly feasible
        x, lam, rc, it, kkt = oracle.qp_gi(G, a, Cm, d)
        assert rc == 0 and kkt < 1e-8 * (1 + np.abs(a).max()), (trial, rc, kkt)


def test_qp_infeasible_detected(oracle):
    G = np.eye(3)
    a = np.zeros(3)
    Cm = np.array([[1.0, 0, 0], [-1.0, 0, 0]])
    d = np.array([-1.0, -1.0])  # x1 <= -1 and x1 >= 1
    assert oracle.qp_gi(G, a, Cm, d)[2] == 2


def test_main_fanuc_oracle_golden(oracle):
    """Frozen oracle golden for main_FANUC.m's configuration (SURVEY.md section 6 scratch: 10 iterations, cost
    1.22532e5, clearance = epsilon) and the sanity pin against the reference's own logged RRT*-CFS costs."""
    ROBOT, robot, obs, s = common.main_fanuc_config()
    P = common.oracle_problem(oracle, ROBOT, obs, s)
    ref = P.solve_batch(s["xR"][:, 0][None], s["ff"][None], np.array([s["caug"]]), s["x_"][None])
    it = int(ref["iters"][0])
    assert it == 10 and (ref["status"][0] & 0xFF) == 0
    assert abs(ref["cost_hist"][0, it - 1] - 122532.0927) < 1e-3
    r = oracle.robot(ROBOT)
    x = ref["x"][0].reshape(30, 10)
    dmin = min(oracle.dist_arm(r, x[i, :5], oracle.obs6(obs[0]["l"]))[0] for i in range(30))
    assert abs(dmin - 0.25) < 1e-4
    # re-linearised at the converged trajectory the constraints hold up to the clearance error seen above
    A, b, *_ = P.get_con(s["xR"][:, 0], x.reshape(-1), ref["u"][0])
    assert (A @ ref["u"][0] - b).max() < 1e-4


# ---- golden fixtures (tests/golden/, frozen by tests/golden/make_golden.py) ------------------------------------------
def _golden_cases(O):
    """name -> (ROBOT, obs, sys_info, solver, grad, noise): the reference's shipped configurations rebuilt from the
    committed input fixtures, with the solver inputs the goldens were computed from (common.frozen_inputs)."""
    inp = common.golden("inputs.npz")
    cases = {}
    ROBOT, robot, obs, s = common.main_fanuc_config()
    s = common.frozen_inputs("main_fanuc", s)
    cases["main_fanuc_cfs"] = (ROBOT, obs, s, 0, 0, None)
    noise = np.random.default_rng(123).normal(0.0, 0.1, size=(1, s["MAX_O_ITER"], s["H"] * 5))
    cases["main_fanuc_psgcfs"] = (ROBOT, obs, s, 1, 0, noise)
    ROBOT, robot, obs, s = common.main_2l_config()
    cases["main_2l_cfs"] = (ROBOT, obs, common.frozen_inputs("main_2l", s), 0, 0, None)
    ROBOT, robot, obs, s = common.main_cfs_m16ib_config(inp["xuori"])
    s = common.frozen_inputs("m16ib_script", s)
    cases["m16ib_script_derivest"] = (ROBOT, obs, s, 0, 1, None)
    obs2 = [dict(obs[0], l=np.array(common.OBS_M16_SCRIPT_ALT))]
    cases["m16ib_script_alt_derivest"] = (ROBOT, obs2, s, 0, 1, None)
    cases["m16ib_script_alt_numjac"] = (ROBOT, obs2, s, 0, 0, None)
    ROBOT, robot, obs, s = common.rrtstar_route_config(inp["route_wp"])
    cases["rrtstar_cfs"] = (ROBOT, obs, common.frozen_inputs("rrtstar", s), 0, 0, None)
    return cases


def check_against_golden(name, out, gold, tol_x=1e-6, tol_c=1e-6):
    """out: dict of per-problem arrays (first axis = problem) ; gold: tests/golden/cases.npz"""
    g = {k: gold["%s.%s" % (name, k)] for k in ("u", "x", "cost_hist", "iters", "status")}
    assert int(out["status"][0]) == int(g["status"]) and int(out["iters"][0]) == int(g["iters"]), name
    it = int(g["iters"])
    if (int(g["status"]) & 0xFF) < 2:
        assert np.abs(out["x"][0] - g["x"]).max() < tol_x and np.abs(out["u"][0] - g["u"]).max() < tol_x, name
    if it:
        assert np.all(np.abs(out["cost_hist"][0][:it] - g["cost_hist"][:it]) <= tol_c * np.abs(g["cost_hist"][:it])), name


@pytest.mark.parametrize("name", ["main_fanuc_cfs", "main_fanuc_psgcfs", "main_2l_cfs", "m16ib_script_derivest",
                                  "m16ib_script_alt_derivest", "m16ib_script_alt_numjac", "rrtstar_cfs"])
def test_oracle_reproduces_golden_cases(oracle, name):
    gold = common.golden("cases.npz")
    ROBOT, obs, s, solver, grad, noise = _golden_cases(oracle)[name]
    P = common.oracle_problem(oracle, ROBOT, obs, s, solver=solver, grad=grad)
    out = P.solve_batch(s["xR"][:, 0][None], s["ff"][None], np.array([s["caug"]]), s["x_"][None], noise=noise)
    check_against_golden(name, out, gold, tol_x=1e-9, tol_c=1e-12)


def test_golden_kat_file_matches_oracle(oracle):
    import json, os
    kat = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "kat.json")))
    k = kat["distLinSeg"]
    d, pts = oracle.dist_lin_seg(k["p1"], k["p2"], k["p3"], k["p4"])
    assert abs(d - k["dist"]) < 0.5 * 10 ** -k["digits"] and np.allclose(pts, k["points"], atol=1e-15)
    which = {"exp": 0, "sin": 1, "sinh": 2, "log": 3}
    for e in kat["derivest"]:
        der, err, _ = oracle.derivest_named(which[e["fun"]], e["x0"])
        assert abs(der - e["der"]) <= 0.5 * 10 ** -e["digits"] * max(1.0, abs(e["der"])), e
        if "errest" in e:
            assert abs(err - e["errest"]) < 1e-19


def test_golden_batch_inputs_regenerate(oracle):
    gold = common.golden("cases.npz")
    cfg = common.batch_m16ib(oracle, 32)
    assert np.array_equal(cfg["theta0"], gold["batch_m16ib_32.theta0"])
    assert np.array_equal(cfg["thetag"], gold["batch_m16ib_32.thetag"])


def test_cubicpolytraj_restatement():
    """RRTstar_CFS.m:96-100: zero-velocity cubic blend through the waypoints (toolbox defaults)."""
    from motionplanning_5d_m_b200 import problem
    wp = np.array([[0.0, 1.0, 3.0], [1.0, 1.0, -1.0]])
    t = np.array([0.0, 0.5, 1.0])
    q = problem.cubicpolytraj(wp, t, np.array([0.0, 0.25, 0.5, 0.75, 1.0]))
    assert np.allclose(q[:, [0, 2, 4]], wp)
    assert np.allclose(q[:, 1], (wp[:, 0] + wp[:, 1]) / 2) and np.allclose(q[:, 3], (wp[:, 1] + wp[:, 2]) / 2)
    eps = 1e-6  # zero velocity at interior waypoints
    qa = problem.cubicpolytraj(wp, t, np.array([0.5 - eps, 0.5 + eps]))
    assert np.abs(qa[:, 1] - qa[:, 0]).max() < 1e-10


def test_rrt_find_route_restatement_properties(oracle):
    """orc_rrt_find_route (RRT_FANUC.m:63-207): structural properties of the tree the reference grows -- every edge is a 0.1 rad
    step from its (original) parent towards a sample (:129), every node passes RRT_FANUC.feasible (:146-181), the route walks
    the parents from the root to the last node (:86-91), the goal box holds unless the search failed (:193-207), RRT and RRT*
    grow the same nodes, and RRT* never lengthens a path to a node (:134-142)."""
    O = oracle
    ROBOT, robot, obs, s = common.rrtstar_cfs_config(np.zeros((5, 41)))
    r = O.robot(ROBOT)
    x0 = np.array([0.421, 0, -0.0092, -0.0010, -1.5786])
    goal = np.array([-1.4090, 0.8873, 0.4008, 0.0, 0.4430])
    region_g = np.array([np.pi / 20, np.pi / 20, np.pi / 10, np.pi / 2, np.pi / 2])
    region_s = np.array([np.pi / 2, np.pi / 2, np.pi / 2, np.pi / 1.5, np.pi / 1.5])
    ratial, off = np.array([1, 1, 0.5, 0.1, 0.1]), np.zeros(5)
    seg, D = [o["l"] for o in obs], [o["D"] for o in obs]
    found = 0
    for seed in range(8):
        rnd = np.random.default_rng(seed).random(12000)
        a = O.rrt_find_route(r, seg, D, x0, goal, region_g, region_s, off, goal, ratial, rnd, star=False)
        b = O.rrt_find_route(r, seg, D, x0, goal, region_g, region_s, off, goal, ratial, rnd, star=True)
        assert a is not None and b is not None
        assert np.array_equal(a["nodes"], b["nodes"]) and a["rnd_used"] == b["rnd_used"] and a["fail"] == b["fail"]
        assert (b["total_dis"] <= a["total_dis"] + 1e-12).all()
        n = a["n_nodes"]
        assert a["parent"][0] == -1 and ((a["parent"][1:] >= 1) & (a["parent"][1:] <= np.arange(1, n))).all()
        step = np.linalg.norm(a["nodes"][1:] - a["nodes"][a["parent"][1:] - 1], axis=1)
        assert np.abs(step - 0.1).max() < 1e-12
        assert all(O.rrt_feasible(r, th, seg, D)[0] for th in a["nodes"][1:])
        assert np.array_equal(a["route"][0], x0) and np.array_equal(a["route"][-1], a["nodes"][-1])
        if not a["fail"]:
            found += 1
            last = a["route"][-1]
            assert ((goal - region_g < last) & (last < goal + region_g)).all() and n <= 400
        else:
            assert n == 401
    assert found >= 3
    assert O.rrt_find_route(r, seg, D, x0, goal, region_g, region_s, off, goal, ratial, np.full(10, 0.3)) is None   # stream too short
    one = O.rrt_find_route(r, seg, D, goal, goal, region_g, region_s, off, goal, ratial, np.zeros(1))              # starts in the goal box
    assert len(one["route"]) == 1 and one["rnd_used"] == 0 and not one["fail"]


@pytest.mark.parametrize("case", ["main_fanuc_cfs", "rrtstar_cfs", "main_fanuc_psgcfs"])
def test_solver_loop_against_an_independent_restatement(oracle, case):
    """SURVEY section 7.1: the frozen oracle goldens of the shipped configurations against tests/np_restatement.py's own
    get_con (duplicated velocity rows), CFS / PSGCFS loop (iteration-1 u = 0 quirk, EVAL stop rule, x_old = ones) and its own
    QP (interior point + active-set polish) -- a second implementation that shares no code with oracle/cfs_oracle.c."""
    g = common.golden("cases.npz")
    if case == "rrtstar_cfs":
        ROBOT, robot, obs, s = common.rrtstar_route_config(common.golden("inputs.npz")["route_wp"])
    else:
        ROBOT, robot, obs, s = common.main_fanuc_config()
    psg = case.endswith("psgcfs")
    noise = np.random.default_rng(123).normal(0.0, 0.1, size=(1, s["MAX_O_ITER"], s["H"] * 5))[0] if psg else None
    rb = dict(robot)
    rb["cap"] = [{"p": np.asarray(c["p"], dtype=np.float64)[:, :2]} for c in robot["cap"]]
    u, x_, cost_all, iters = NP.cfs_optimizer(s, rb, obs, ROBOT, psg=psg, noise=noise)
    assert iters == int(g[case + ".iters"])
    assert np.abs(x_ - g[case + ".x"]).max() < 1e-7 and np.abs(u - g[case + ".u"]).max() < 1e-7
    ref = g[case + ".cost_hist"][:iters]
    assert np.all(np.abs(cost_all - ref) <= 1e-7 * np.abs(ref))


def test_oracle_infeasibility_verdicts_against_an_lp(oracle):
    """The oracle's "QP infeasible" verdicts on the PSGCFS bench batch (M200i, H = 30, 2048 problems), checked by a phase-1 LP
    (scipy / HiGHS) on the oracle's dense rows: min t s.t. A u - t <= b.  Includes the 8 problems on which the CUDA projection
    used to return a point (DESIGN.md section 2, "a parity bug this rule exposed"): the LP confirms the oracle on all of them."""
    scipy_opt = pytest.importorskip("scipy.optimize")
    import bench
    from motionplanning_5d_m_b200 import synthetic
    O = oracle
    B, H = 2048, 30
    c0 = synthetic.batch_config_m200i_psgcfs(B, bench.oracle_feasible(O, "M200i", [synthetic.OBS_M200I]), horizon=H, seed=synthetic.SEED)
    s = c0["sys_info"]
    n = H * 5
    P = bench.make_oracle_problem(O, c0, 0, solver=1)
    ref = P.solve_batch(c0["x0"], c0["ff"], c0["caug"], c0["xref"], noise=c0["noise"])
    st = ref["status"] & 0xFF
    first_infeasible = np.where((st == 2) & (ref["iters"] == 0))[0]
    assert len(first_infeasible) > 100
    disputed = [646, 652, 1325, 1376, 1521, 1651, 1706, 2021]
    assert all(b in first_infeasible for b in disputed)
    feasible = np.where(st == 1)[0][:6]
    for b in list(disputed) + list(first_infeasible[:6]) + list(feasible):
        A_, b_, _, _, _, _ = P.get_con(c0["x0"][b], c0["xref"][b], np.zeros(n))
        m = A_.shape[0]
        cvec = np.zeros(n + 1)
        cvec[-1] = 1.0
        res = scipy_opt.linprog(cvec, A_ub=np.hstack([A_, -np.ones((m, 1))]), b_ub=b_, bounds=[(None, None)] * n + [(-1.0, None)],
                                method="highs")
        assert res.status == 0
        if st[b] == 2:
            assert res.fun > 1e-6, (b, res.fun)      # no u satisfies every row: the smallest maximal violation is positive
        else:
            assert res.fun < -1e-6, (b, res.fun)


@pytest.mark.parametrize("star", [False, True])
def test_rrt_find_route_against_an_independent_restatement(oracle, star):
    """orc_rrt_find_route against tests/np_restatement.py's own RRT_FANUC.find_route (own FK / distLinSeg / feasibility, python
    lists for the tree) on the scene of RRTstar_CFS.m, same uniform stream: same parents, node counts, numbers consumed and
    failure flags; nodes, accumulated distances and the route to 1e-12."""
    from motionplanning_5d_m_b200 import rrt
    O = oracle
    sc = rrt.SCENE_RRTSTAR
    robot = M.robotproperty2("M200i")
    rb = dict(robot)
    rb["cap"] = [{"p": np.asarray(c["p"], dtype=np.float64)[:, :2]} for c in robot["cap"]]
    r = O.robot("M200i")
    found = 0
    for seed, max_iter in ((1, 400), (0, 120), (2, 120), (3, 120)):   # seed 1 reaches the goal box after 186 nodes, the others hit MAX_ITER
        rnd = np.random.default_rng(900 + seed).random(4096)
        a = O.rrt_find_route(r, sc["obs"], [o["D"] for o in sc["obs"]], sc["x0"], sc["goal"], sc["region_g"], sc["region_s"],
                             sc["sample_off"], sc["goal"], sc["ratial"], rnd, max_iter=max_iter, star=star)
        route, nodes, tot, fail, used = NP.rrt_find_route(rb, "M200i", sc["obs"], sc["x0"], sc["goal"], sc["goal"], sc["region_g"],
                                                          sc["region_s"], sc["sample_off"], sc["ratial"], rnd, max_iter=max_iter,
                                                          star=star)
        assert a is not None
        assert a["n_nodes"] == nodes.shape[1] and a["fail"] == fail and a["rnd_used"] == used
        assert np.array_equal(a["parent"], nodes[0].astype(np.int32))
        assert np.abs(a["nodes"] - nodes[1:].T).max() < 1e-12 and np.abs(a["total_dis"] - tot).max() < 1e-12
        assert a["route"].shape == route.T.shape and np.abs(a["route"] - route.T).max() < 1e-12
        found += 0 if fail else 1
    assert found >= 1 and found < 4   # both exits of find_route are exercised: goal box reached, MAX_ITER
