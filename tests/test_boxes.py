"""Box obstacles (SURVEY.md section 8f N3; an extension: the reference's own mesh path is dead code, Lib/functions/
dist_arm_surface.m:44).  CPU: known answers of the oracle's segment-to-box distance (degenerate, inside, edge-parallel, corner
cases), an independent brute-force cross-check, the STL -> box tool on a synthetic mesh, and the frozen golden built from the
reference's map/assembly line_Assem1.STL.  GPU (-m gpu): K1 / K1d / K6 / the fused solver against the oracle on those boxes."""
import struct

import numpy as np
import pytest

import motionplanning_5d_m_b200 as M
from motionplanning_5d_m_b200 import _lib, stl_boxes, synthetic
from tests import common


def _boxes():
    g = common.golden("stl_boxes.npz")
    obs = [{"shape": "box", "l": g["box_l"][:, :, j], "D": float(g["box_D"][j]), "epsilon": float(g["box_epsilon"][j])}
           for j in range(g["box_l"].shape[2])]
    return g, obs


def test_segment_box_distance_known_answers(oracle):
    O = oracle
    lo, hi = np.array([0.0, 0.0, 0.0]), np.array([1.0, 2.0, 3.0])
    kat = [  # (ps, pe, distance, closest point of the segment)
        ([2, 1, 1], [2, 1, 2], 1.0, [2, 1, 1]),                       # parallel to a face: distance 1, first minimiser t = 0
        ([-1, -1, -1], [-1, -1, -1], np.sqrt(3.0), [-1, -1, -1]),      # degenerate segment (a point) off the min corner
        ([0.5, 1, 1], [0.5, 1, 2], 0.0, [0.5, 1, 1]),                 # inside the box
        ([-1, 1, 1], [3, 1, 1], 0.0, [0, 1, 1]),                      # passes through: distance 0 at the entry point
        ([2, 3, 4], [3, 4, 5], np.sqrt(3.0), [2, 3, 4]),              # pointing away from the max corner
        ([2, 0.5, 5], [0.5, 0.5, 3.5], 0.5, [0.5, 0.5, 3.5]),         # ends above the top face
        ([2, -1, 1.5], [-1, 2 + 1e-300, 1.5], 0.0, None),             # diagonal cut through the x-y cross-section
        ([3, 0, 4], [0, 3 * 0 + 0, 7], None, None),                   # skew, checked by brute force below
        ([1.5, -1, 3.5], [1.5, 3, 3.5], np.sqrt(0.5), [1.5, 0, 3.5]),  # parallel to an EDGE (x = 1, z = 3): first minimiser
    ]
    for ps, pe, d_ref, pt_ref in kat:
        d, pt = O.dist_seg_box(ps, pe, lo, hi)
        ts = np.linspace(0, 1, 20001)
        x = np.asarray(ps, float)[None] + ts[:, None] * (np.asarray(pe, float) - np.asarray(ps, float))[None]
        brute = np.sqrt((np.maximum(np.maximum(lo - x, x - hi), 0.0) ** 2).sum(1)).min()
        assert abs(d - brute) < 2e-4 and d <= brute + 1e-12
        if d_ref is not None:
            assert abs(d - d_ref) < 1e-14, (ps, pe, d, d_ref)
        if pt_ref is not None:
            assert np.abs(pt - np.array(pt_ref, float)).max() < 1e-14, (ps, pe, pt)


def test_segment_box_distance_against_scalar_minimisation(oracle):
    from scipy.optimize import minimize_scalar
    rng = np.random.default_rng(5)
    for _ in range(400):
        lo = rng.uniform(-1, 0, 3)
        hi = lo + rng.uniform(0.05, 2, 3)
        ps, pe = rng.uniform(-3, 3, 3), rng.uniform(-3, 3, 3)
        if rng.random() < 0.2:
            pe[rng.integers(3)] = ps[rng.integers(3)]          # axis-parallel components
        f = lambda t: np.sqrt((np.maximum(np.maximum(lo - (ps + t * (pe - ps)), (ps + t * (pe - ps)) - hi), 0.0) ** 2).sum())
        ref = min(minimize_scalar(f, bounds=(0, 1), method="bounded", options={"xatol": 1e-14}).fun, f(0.0), f(1.0))
        d, pt = oracle.dist_seg_box(ps, pe, lo, hi)
        assert abs(d - ref) < 1e-7 and d <= ref + 1e-12
        assert abs(f(np.dot(pt - ps, pe - ps) / max(np.dot(pe - ps, pe - ps), 1e-300)) - d) < 1e-9


def test_stl_to_boxes_tool(tmp_path):
    """a synthetic binary STL (two separate cubes, millimetres) through MapFromSTL.m's transform and the k-d cover"""
    def cube(lo, hi):
        x0, y0, z0 = lo
        x1, y1, z1 = hi
        v = np.array([[x0, y0, z0], [x1, y0, z0], [x1, y1, z0], [x0, y1, z0], [x0, y0, z1], [x1, y0, z1], [x1, y1, z1], [x0, y1, z1]], float)
        f = [(0, 1, 2), (0, 2, 3), (4, 5, 6), (4, 6, 7), (0, 1, 5), (0, 5, 4), (2, 3, 7), (2, 7, 6), (1, 2, 6), (1, 6, 5), (0, 3, 7), (0, 7, 4)]
        return np.array([[v[a], v[b], v[c]] for a, b, c in f])
    tri = np.concatenate([cube((0, 100, 0), (1000, 1100, 500)), cube((4000, 100, 0), (4500, 600, 2000))])
    p = tmp_path / "two_cubes.stl"
    with open(p, "wb") as fh:
        fh.write(b"\0" * 80 + struct.pack("<I", len(tri)))
        for t in tri:
            fh.write(struct.pack("<12fH", 0, 0, 0, *t.reshape(-1), 0))
    assert np.array_equal(stl_boxes.read_stl(str(p)), tri)
    obs = stl_boxes.boxes_from_stl(str(p), max_boxes=2, D=0.1, epsilon=0.2)
    assert len(obs) == 2 and all(o["shape"] == "box" and o["D"] == 0.1 and o["epsilon"] == 0.2 for o in obs)
    got = sorted([tuple(np.round(o["l"].T.reshape(-1), 9)) for o in obs])
    # MapFromSTL.m:6-11: minimum to 0, second coordinate - 100 mm, (x, y, z) <- (z, x, y); then metres
    want = sorted([(0.0, 0.0, -0.1, 0.5, 1.0, 0.9), (0.0, 4.0, -0.1, 2.0, 4.5, 0.4)])
    assert np.allclose(got, want, atol=1e-9), (got, want)


def test_box_golden_matches_the_oracle(oracle):
    """the frozen STL-box golden (tests/golden/make_box_golden.py) against the current oracle build"""
    g, obs = _boxes()
    r = oracle.robot("M16iB")
    for j, o in enumerate(obs):
        o7 = oracle.obs6(o)
        for i in range(0, 256, 8):
            d, lid = oracle.dist_arm(r, g["theta"][i], o7)[:2]
            assert d == g["dist"][i, j] and lid == g["linkid"][i, j]
    robot = M.robotproperty2("M16iB")
    s = common.frozen_inputs("box_solve1", M.make_sys_info(robot, 5, 30, g["solve1.theta0"], g["solve1.thetag"]))
    P = common.oracle_problem(oracle, "M16iB", obs, s)
    res = P.solve_batch(s["xR"][:, 0][None], s["ff"][None], np.array([s["caug"]]), s["x_"][None])
    assert int(res["iters"][0]) == int(g["solve1.iters"]) and np.array_equal(res["x"][0], g["solve1.x"])


@pytest.mark.gpu
def test_box_distance_gradient_and_feasibility_parity(ctx, oracle):
    """K1 (num_jac), K1d (DERIVEST) and K6 (RRT feasibility) on a MIXED obstacle list: the STL-derived boxes + a capsule."""
    O = oracle
    g, boxes = _boxes()
    obs = boxes + [dict(synthetic.OBS_M16IB)]
    robot = dict(M.robotproperty2("M16iB"))
    robot["name"] = "M16iB"
    ctx.set_robot(robot, 5)
    ctx.set_obstacles(obs)
    th = g["theta"]
    dist, lid, grad, flags = ctx.dist_grad(th)
    nb = len(boxes)
    assert np.abs(dist[:, :nb] - g["dist"]).max() < 1e-12 and (np.sign(dist[:, :nb]) == np.sign(g["dist"])).all()
    assert np.array_equal(lid[:, :nb], g["linkid"])
    smooth = np.abs(g["grad"]).max(axis=2) < 50                        # away from the touch discontinuity
    assert smooth.mean() > 0.95 and np.abs(grad[:, :nb] - g["grad"])[smooth].max() < 1e-8
    r = O.robot("M16iB")
    o7 = O.obs6(obs[nb])
    assert np.abs(dist[:, nb] - np.array([O.dist_arm(r, t, o7)[0] for t in th])).max() < 1e-12   # the capsule is unaffected
    # DERIVEST on dist_link(linkid) against the boxes
    dd, ld, gd, _ = ctx.dist_grad(th[:64], grad=_lib.GRAD_DERIVEST)
    for i in range(0, 64, 4):
        for j in range(nb):
            ref = O.derivest_grad(r, th[i], O.obs6(boxes[j]), int(g["linkid"][i, j]))
            sel = np.abs(ref) < 50
            assert np.abs(gd[i, j] - ref)[sel].max() <= 1e-7 * max(1.0, np.abs(ref[sel]).max())
    # K6: infeasible iff some link is closer than obs.D to some obstacle (RRT_FANUC.m:172)
    feas, dmin = ctx.nodes_feasible(th)
    D = [o["D"] for o in obs]
    for i in range(0, 256, 2):
        f_ref, d_ref = O.rrt_feasible(r, th[i], obs, D)
        assert bool(feas[i]) == f_ref and abs(dmin[i] - d_ref) < 1e-12
    assert feas.any() and not feas.all()


@pytest.mark.gpu
def test_box_solve_parity(ctx, oracle):
    """CFS against the STL-derived boxes: the three golden start/goal pairs (one takes the touch branch) through the fused
    solver and the launch-per-iteration path, plus a seeded batch against boxes + capsule with infeasible problems."""
    O = oracle
    g, boxes = _boxes()
    robot = M.robotproperty2("M16iB")
    rb = dict(robot)
    rb["name"] = "M16iB"
    ctx.set_robot(rb, 5)
    ctx.set_obstacles(boxes)
    H = 30
    cfgs = [M.make_sys_info(robot, 5, H, g["solve%d.theta0" % k], g["solve%d.thetag" % k]) for k in range(3)]
    s = cfgs[0]
    ctx.set_cost(H, s["QQ"], s["lim"], s["MAX_input"])
    args = tuple(np.stack(v) for v in zip(*[(c["xR"][:, 0], c["ff"], np.float64(c["caug"]), c["x_"]) for c in cfgs]))
    for fused in (1, 0):
        ctx.set_option("fused", fused)
        out = ctx.solve_batch(*args, s["epsilon_O"], s["MAX_O_ITER"])
        ctx.set_option("fused", 1)
        for k in range(3):
            it = int(g["solve%d.iters" % k])
            assert int(out["status"][k]) == int(g["solve%d.status" % k]) and int(out["iters"][k]) == it, (fused, k)
            assert np.abs(out["x"][k] - g["solve%d.x" % k]).max() < 1e-6 and np.abs(out["u"][k] - g["solve%d.u" % k]).max() < 1e-6
            ref = g["solve%d.cost_hist" % k][:it]
            assert np.all(np.abs(out["cost_hist"][k, :it] - ref) <= 1e-6 * np.abs(ref))
    # a batch: random start/goal pairs that are feasible against boxes and capsule; lines through a box are infeasible
    obs = boxes + [dict(synthetic.OBS_M16IB)]
    ctx.set_obstacles(obs)
    cfg = synthetic.batch_config("M16iB", 96, lambda c: ctx.nodes_feasible(c)[0], obs, H, 77, synthetic.SAMPLE_OFF)
    sb = cfg["sys_info"]
    ctx.set_cost(H, sb["QQ"], sb["lim"], sb["MAX_input"])
    bargs = (cfg["x0"], cfg["ff"], cfg["caug"], cfg["xref"])
    out = ctx.solve_batch(*bargs, sb["epsilon_O"], sb["MAX_O_ITER"])
    P = common.oracle_problem(O, "M16iB", obs, sb)
    ref = P.solve_batch(*bargs, nthreads=8)
    twin = P.solve_batch(*bargs, nthreads=8, use_twin=True)
    assert np.array_equal(out["status"], ref["status"]) and np.array_equal(out["iters"], ref["iters"])
    ok = (ref["status"] & 0xFF) < 2
    well = ok & (np.abs(twin["x"] - ref["x"]).max(axis=1) < 1e-8)
    assert ok.sum() > 48 and well.sum() >= ok.sum() - 4
    assert np.abs(out["x"] - ref["x"])[well].max() < 1e-6
