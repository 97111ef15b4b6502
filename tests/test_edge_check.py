"""Continuous collision checks, CPU side: the motion bound, and the soundness of the conservative-advancement restatement
(tests/check_oracle.c) against dense brute force on edges and on solved CFS trajectories.  The GPU kernels are held to this
restatement in tests/test_gpu_edge_check.py."""
import numpy as np
import pytest

from motionplanning_5d_m_b200 import rrt, synthetic
from tests import check_oracle as K
from tests import common

ETA = 1e-3
SCENES = {  # name -> (robot, obstacles, sampling box offset, half widths)
    "headline": ("M16iB", [synthetic.OBS_M16IB], synthetic.SAMPLE_OFF, synthetic.REGION_S),
    "rrtstar": ("M200i", rrt.SCENE_RRTSTAR["obs"], rrt.SCENE_RRTSTAR["sample_off"], rrt.SCENE_RRTSTAR["region_s"]),
    "boxes": ("M16iB", None, synthetic.SAMPLE_OFF, synthetic.REGION_S),
    "2L": ("2L", [{"l": np.array([[0.3, 0.3], [0.3, 0.3], [0.0, 0.0]]), "D": 0.05, "epsilon": 0.05}], np.zeros(2),
           np.array([np.pi, np.pi])),
}


def box_obstacles():
    g = common.golden("stl_boxes.npz")
    return [{"shape": "box", "l": g["box_l"][:, :, j], "D": float(g["box_D"][j]), "epsilon": float(g["box_epsilon"][j])}
            for j in range(g["box_l"].shape[2])]


def scene(name):
    robot, obs, off, half = SCENES[name]
    return K.Scene(robot, box_obstacles() if obs is None else obs), off, half


def random_edges(rng, N, off, half, reach=0.6):
    """edges from a uniform start in the sampling box to a point within +-reach rad per joint (a mix of clear and hitting ones)"""
    a = off + (rng.random((N, off.size)) - 0.5) * 2 * half
    return a, a + rng.uniform(-reach, reach, a.shape)


def brute_edges(sc, a, b, M=2001):
    s = np.linspace(0.0, 1.0, M)
    th = (a[:, None, :] + s[None, :, None] * (b - a)[:, None, :]).reshape(-1, a.shape[1])
    return s, sc.clearance(th).reshape(a.shape[0], M)


@pytest.mark.parametrize("robot", ["M16iB", "M200i", "2L"])
def test_motion_bound_dominates_endpoint_speed(robot):
    import oracle as O
    r = O.robot(robot)
    R = K.motion_bound(r)
    rng = np.random.default_rng(11)
    h = 1e-6
    worst = np.zeros(r.nj)
    for _ in range(20000):
        th = rng.uniform(-np.pi, np.pi, r.nj)
        for j in range(r.nj):
            e = np.zeros(r.nj)
            e[j] = h
            dp = (O.cap_pos(r, th + e) - O.cap_pos(r, th - e)) / (2 * h)   # (link, endpoint, xyz)
            worst[j] = max(worst[j], np.linalg.norm(dp[j:], axis=-1).max() / R[j])
    assert (worst <= 1 + 1e-6).all(), worst


@pytest.mark.parametrize("name", list(SCENES))
def test_edge_verdicts_sound_against_brute_force(name):
    sc, off, half = scene(name)
    eta = ETA
    rng = np.random.default_rng(list(SCENES).index(name) + 17)
    a, b = random_edges(rng, 300, off, half, reach=0.6 if name != "2L" else 1.5)
    out = sc.check_edges(a, b, eta=eta)
    s, bf = brute_edges(sc, a, b)
    v = out["verdict"]
    assert (v != K.UNDECIDED).all()
    assert ((v == K.HIT) | (bf.min(1) >= -eta)).all()                  # brute-force min < -eta => HIT
    assert ((v == K.CLEAR) | (bf.min(1) < -eta / 2)).all()             # brute-force min >= -eta/2 => CLEAR
    assert (v == K.CLEAR).sum() > 10 and (v == K.HIT).sum() > 10, np.bincount(v)
    for i in np.flatnonzero(v == K.HIT):
        sh = out["s_hit"][i]
        assert 0.0 <= sh <= 1.0
        w = sc.clearance(a[i] + sh * (b[i] - a[i]))[0]
        assert w < -eta / 2 and out["cmin"][i] <= w
        assert bf[i, s < sh].min(initial=np.inf) >= -eta
    assert (out["s_hit"][v == K.CLEAR] == -1.0).all()
    assert (out["cmin"][v == K.CLEAR] >= -eta / 2).all()


def test_trajectory_verdicts_sound_on_solved_headline_problems(oracle):
    cfg = common.batch_m16ib(oracle, 128)
    s = cfg["sys_info"]
    P = common.oracle_problem(oracle, "M16iB", cfg["obs"], s)
    sol = P.solve_batch(cfg["x0"], cfg["ff"], cfg["caug"], cfg["xref"], nthreads=8)
    conv = np.flatnonzero((sol["status"] & 0xFF) == 0)
    assert conv.size > 64
    sc = K.Scene("M16iB", cfg["obs"])
    x0, x, u = cfg["x0"][conv], sol["x"][conv], sol["u"][conv]
    out = sc.check_trajectories(x0, x, u, eta=ETA)
    nj, H, dt = 5, s["H"], s["robot"]["delta_t"]
    tau = np.linspace(0.0, dt, 401)
    v = out["verdict"]
    assert (v != K.UNDECIDED).all()
    for i in range(conv.size):
        segs = [sc.clearance(K.segment_points(x0[i], x[i], u[i], nj, dt, k, tau)) for k in range(H)]
        bf = np.concatenate(segs)
        t = np.concatenate([k * dt + tau for k in range(H)])
        assert v[i] == K.HIT or bf.min() >= -ETA, i
        assert v[i] == K.CLEAR or bf.min() < -ETA / 2, i
        if v[i] == K.HIT:
            th = out["t_hit"][i]
            k = min(int(th // dt), H - 1)
            w = sc.clearance(K.segment_points(x0[i], x[i], u[i], nj, dt, k, [th - k * dt]))[0]
            assert w < -ETA / 2
            assert bf[t < th - 1e-12].min(initial=np.inf) >= -ETA
        else:
            assert out["t_hit"][i] == -1.0
    # the waypoints of a converged CFS solution sit on the margin; between them the arm may cut it: that is what the check finds
    assert (v == K.HIT).sum() >= 1


def test_known_cases():
    sc, off, half = scene("headline")
    # an edge whose middle sweeps the arm through the obstacle axis while both ends are clear
    rng = np.random.default_rng(3)
    a, b = random_edges(rng, 4000, off, half, reach=1.2)
    ca, cb = sc.clearance(a), sc.clearance(b)
    s, bf = brute_edges(sc, a, b, M=201)
    cross = np.flatnonzero((ca > 0.05) & (cb > 0.05) & (bf.min(1) < -0.19))[:5]   # -0.19: the axis itself (d < 0.01)
    assert cross.size > 0
    out = sc.check_edges(a[cross], b[cross])
    assert (out["verdict"] == K.HIT).all() and (out["s_hit"] > 0).all()
    # zero-length edges: the RRT node verdict and its dmin - D
    import oracle as O
    th = off + (rng.random((200, 5)) - 0.5) * 2 * half
    out = sc.check_edges(th, th)
    for i in range(200):
        feas, dmin = O.rrt_feasible(sc.r, th[i], [synthetic.OBS_M16IB], [0.2])
        assert out["cmin"][i] == dmin - 0.2
        assert out["evals"][i] == 1
        # the hit threshold is -eta/2: a node closer than D by less than that is CLEAR here and infeasible for the RRT
        assert (out["verdict"][i] == K.HIT) == (dmin - 0.2 < -ETA / 2)
        if abs(dmin - 0.2) > ETA:
            assert (out["verdict"][i] == K.CLEAR) == feas
    # far from every obstacle: the evaluation count the step rule predicts
    R = K.motion_bound(sc.r)
    far = [K.Scene("M16iB", [{"l": np.array([[30.0, 30.0], [8.3, 8.3], [0.0, 1.9]]), "D": 0.2, "epsilon": 0.2}])]
    a, b = np.array([[0.1, 1.2, -0.3, 0.4, 0.2]]), np.array([[0.9, 2.0, 0.5, -0.4, 1.0]])
    o = far[0].check_edges(a, b, eta=ETA)
    vmax = 0.0
    for k in range(5):
        vmax = vmax + R[k] * abs(b[0, k] - a[0, k])
    sv, n = 0.0, 0
    while True:
        c = far[0].clearance(a + sv * (b - a))[0]
        n += 1
        if sv == 1.0:
            break
        sv = min(sv + (c + ETA) / vmax, 1.0)
    assert o["verdict"][0] == K.CLEAR and o["evals"][0] == n and n >= 2
    # max_evals bounds the work: UNDECIDED
    o = sc.check_edges(a, b, eta=ETA, max_evals=1)
    assert o["verdict"][0] in (K.UNDECIDED, K.HIT)
    # rejected arguments
    for eta in (0.0, -1e-3, np.nan, 0.2 - 0.5e-4):
        with pytest.raises(ValueError):
            sc.check_edges(a, b, eta=eta)
