"""-m gpu : the warp tier's mapping of waypoints to lanes at every horizon where it changes shape.

The warp tier (k_warp.cu) evaluates the num_jac rows itself, one waypoint per lane (a second round for waypoints 32..H-1),
and its QP scan (qp_warp.cuh, w_scan) holds two consecutive waypoints per lane in its prefix sums, obstacles two at a time.
The launch-per-iteration path with warp_lockstep=1 runs the same warp QP on rows from the stand-alone gradient kernel (K1),
which evaluates every waypoint in one thread.  Both must give the same solve: status, flags and iteration counts identical,
trajectories within the tolerances of tests/test_gpu_parity.py.  H = 1, 17, 31, 32, 33, 50, 64 cover one partial round,
one full round and a partial second round of both mappings; 1-3 obstacles, boxes among them, cover odd and even obstacle
counts in the scan.  Both paths run the same w_scan, so this module checks the warp tier's gradient phase and lane mapping;
w_scan itself is checked against the CPU oracle by tests/test_gpu_parity.py.
"""
import numpy as np
import pytest

import motionplanning_5d_m_b200 as M
from motionplanning_5d_m_b200 import _lib, problem, synthetic
from tests import common
from tests.test_gpu_parity import _compare_solve, _set

pytestmark = pytest.mark.gpu

HORIZONS = [1, 17, 31, 32, 33, 50, 64]
WARP = dict(fused=1, warp=1, warp_lockstep=0)
K1_ROWS = dict(fused=0, warp_lockstep=1)
DEFAULTS = dict(fused=1, warp=1, warp_cfg=3, warp_zs=0, warp_qcap=15, screen=2, warp_lockstep=0)

CAPSULE2 = {"l": np.array([[3.406, 3.406], [7.813, 7.813], [0.800, 1.538]]), "D": 0.2, "epsilon": 0.2}
BOX = {"shape": "box", "l": np.array([[3.6, 4.1], [8.0, 8.6], [0.2, 1.2]]), "D": 0.1, "epsilon": 0.2}
OBSTACLES = {1: [synthetic.OBS_M16IB], 2: [synthetic.OBS_M16IB, BOX], 3: [synthetic.OBS_M16IB, CAPSULE2, BOX]}


def _solve_both(ctx, ROBOT, robot, obs, s, args):
    _set(ctx, ROBOT, robot, obs, s)
    outs = []
    try:
        for mode in (WARP, K1_ROWS):
            for k, v in mode.items():
                ctx.set_option(k, v)
            outs.append(ctx.solve_batch(*args, s["epsilon_O"], s["MAX_O_ITER"]))
    finally:
        for k, v in DEFAULTS.items():
            ctx.set_option(k, v)
    return outs


@pytest.mark.parametrize("nobs", [1, 2, 3])
@pytest.mark.parametrize("H", HORIZONS)
def test_m16ib_warp_rows_match_k1_rows(ctx, oracle, H, nobs):
    """NJ = 5: a seeded M16iB batch (the headline robot) with capsule and box obstacles."""
    cfg = common.batch_m16ib(oracle, 48, horizon=H)
    s = cfg["sys_info"]
    args = (cfg["x0"], cfg["ff"], cfg["caug"], cfg["xref"])
    warp, ref = _solve_both(ctx, "M16iB", cfg["robot"], OBSTACLES[nobs], s, args)
    _compare_solve(warp, ref)
    assert (warp["status"] == ref["status"]).all()  # the touch flag included


@pytest.mark.parametrize("nobs", [1, 2])
@pytest.mark.parametrize("H", HORIZONS)
def test_2l_warp_rows_match_k1_rows(ctx, H, nobs):
    """NJ = 2: main_2L.m's planar arm towards several goals, the second obstacle a box."""
    ROBOT, robot, obs, _ = common.main_2l_config()
    obs = obs + [{"shape": "box", "l": np.array([[0.5, 0.7], [0.1, 0.4], [-0.1, 0.1]]), "D": 0.05, "epsilon": 0.05}]
    rows = []
    for g in (np.pi / 2, np.pi / 3, 2.0, -1.0):
        s = M.make_sys_info(robot, 2, H, [0.0, 0.0], [g, 0.0], Q=problem.Q_2L, Rblk=problem.R_2L, r_scale=0.1,
                            lim=[0.1, 0.2], max_input=np.tile(np.array([1.0, 1.0]) * 0.5 * robot["delta_t"], H),
                            epsilon_O=1e-6, MAX_O_ITER=30)
        rows.append((s["xR"][:, 0], s["ff"], s["caug"], s["x_"]))
    args = tuple(np.ascontiguousarray(np.stack([r[k] for r in rows])) for k in range(4))
    warp, ref = _solve_both(ctx, ROBOT, robot, obs[:nobs], s, args)
    _compare_solve(warp, ref)
    assert (warp["status"] == ref["status"]).all()


@pytest.mark.parametrize("H,touching", [(10, 5), (55, 32), (60, 35)])
def test_touch_flag_on_first_and_second_round_lanes(ctx, oracle, H, touching):
    """The touch flag is an OR over the warp's lanes.  main_FANUC.m's straight start trajectory passes through the obstacle
    axis at 0.6 of its length, so at these horizons exactly one waypoint touches: index 5 of 10 (lane 5, the only round),
    32 of 55 (lane 0, second round) or 35 of 60 (lane 3, second round).  Both paths must raise the flag."""
    ROBOT, robot, obs, _ = common.main_fanuc_config()
    x0 = [0.7825, 0.0284, 0.2172, 0.1444, -1.1779]
    xg = [-0.7825, 0.0284, 0.2172, 0.1444, -1.1779]
    s = M.make_sys_info(robot, 5, H, x0, xg)
    r, o6 = oracle.robot(ROBOT), oracle.obs6(obs[0]["l"])
    d = np.array([oracle.dist_arm(r, th, o6)[0] for th in s["x_"].reshape(H, 10)[:, :5]])
    assert np.where(d < 0)[0].tolist() == [touching]  # the fixture: one touching waypoint, on the intended lane
    args = (s["xR"][:, 0][None], s["ff"][None], np.array([s["caug"]]), s["x_"][None])
    warp, ref = _solve_both(ctx, ROBOT, robot, obs, s, args)
    assert ref["status"][0] & _lib.FLAG_TOUCH
    assert (warp["status"] == ref["status"]).all()
    _compare_solve(warp, ref)
