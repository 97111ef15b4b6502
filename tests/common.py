"""Shared problem builders for the parity tests (reference configurations, SURVEY.md section 8d)."""
import numpy as np

import motionplanning_5d_m_b200 as M
from motionplanning_5d_m_b200 import problem, synthetic


OBS_M16_SCRIPT_ALT = [[4.506, 4.506], [8.513, 8.513], [1.072, 1.538]]  # M16iB/main_CFS.m:53 (commented alternative)


def golden(name):
    import os
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name))


FROZEN_KEYS = ("QQ", "ff", "caug", "alpha")


def assert_rounding_close(got, ref, what):
    """got equals ref up to the rounding of a matrix product: |got - ref| <= 1e-13 max|ref|"""
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    assert got.shape == ref.shape and np.abs(got - ref).max() <= 1e-13 * np.abs(ref).max(), what


def frozen_inputs(name, s):
    """sys_info `s` of the golden configuration `name` with QQ, ff, caug and alpha as they were when its goldens were computed
    (tests/golden/solver_inputs.npz, written by tests/golden/make_solver_inputs.py).  The config builders compute these with
    BLAS / LAPACK products and SIMD sums whose last bits change with the CPU, the BLAS kernel and its thread count, and some
    golden problems amplify that above the golden tolerances.  The freshly built values must agree with the frozen ones to
    rounding; the solve then starts from the exact numbers the goldens came from."""
    g = golden("solver_inputs.npz")
    out = dict(s)
    for k in FROZEN_KEYS:
        ref = g["%s.%s" % (name, k)]
        assert_rounding_close(s.get(k, 0.0), ref, (name, k))
        out[k] = ref if ref.ndim else float(ref)
    return out


def main_fanuc_config():
    """main_FANUC.m:13-60,106-127 : M200i, H=30, one capsule obstacle."""
    robot = M.robotproperty2("M200i")
    x0 = [0.7825, 0.0284, 0.2172, 0.1444, -1.1779]
    xg = [-0.7825, 0.0284, 0.2172, 0.1444, -1.1779]
    s = M.make_sys_info(robot, 5, 30, x0, xg)
    obs = [{"l": np.array([[3.806, 3.606], [8.413, 8.413], [0.001, 1.038]]), "D": 0.2, "epsilon": 0.25}]
    return "M200i", robot, obs, s


def main_2l_config():
    """main_2L.m:14-121 : two-link planar arm, H=40, point obstacle, stationary reference."""
    robot = M.robotproperty2("2L")
    nj, H = 2, 40
    x0, xg = [0.0, 0.0], [np.pi / 2, 0.0]
    s = M.make_sys_info(robot, nj, H, x0, xg, Q=problem.Q_2L, Rblk=problem.R_2L, r_scale=0.1, lim=[0.1, 0.2],
                        max_input=np.tile(np.array([1.0, 1.0]) * 0.5 * robot["delta_t"], H), epsilon_O=1e-6,
                        MAX_O_ITER=100, x_ref=np.tile(np.array([0.0, 0.0, 0.0, 0.0]), H))
    obs = [{"l": np.array([[0.3, 0.3], [0.3, 0.3], [0.0, 0.0]]), "D": 0.05, "epsilon": 0.05}]
    return "2L", robot, obs, s


def rrtstar_cfs_config(route):
    """RRTstar_CFS.m:40-50,96-187 : M200i, H=40, two obstacles, R*10, Q_v=[100,20,1,1,1]; route = 5 x (H+1) samples."""
    robot = M.robotproperty2("M200i")
    H = 40
    s = M.make_sys_info(robot, 5, H, route[:, 0], route[:, -1], Q=problem.Q_RRTSTAR, r_scale=10.0,
                        x_ref=np.concatenate([np.concatenate([route[:, i], np.zeros(5)]) for i in range(1, H + 1)]))
    obs = [{"l": np.array([[3.606, 3.606], [8.413, 8.413], [0.001, 1.038]]), "D": 0.2, "epsilon": 0.2},
           {"l": np.array([[3.406, 3.406], [7.813, 7.813], [0.800, 1.538]]), "D": 0.2, "epsilon": 0.2}]
    return "M200i", robot, obs, s


def main_cfs_m16ib_config(xuori):
    """M16iB/main_CFS.m:15-113 (the DERIVEST script path): H=24, straight line between the ends of data/good_xori.mat with
    constant-velocity rows (dt=0.05 there, :33-39), QQ = Baug'QaugBaug (R*0, :113), no velocity rows, bounds +-0.2,
    D = 0.2, stop ||xref-oldref|| < 0.01, at most 10 iterations."""
    robot = M.robotproperty2("M16iB")  # robotproperty(3): same DH / capsules / dt, base passed explicitly (:17)
    xuori = np.asarray(xuori, dtype=np.float64).reshape(-1)
    nj, H = 5, 24
    x0, xg = xuori[:10], xuori[-10:]
    th = np.stack([np.linspace(x0[k], xg[k], H + 1) for k in range(nj)])                     # :29-31
    w = np.stack([np.concatenate([np.full(H, (xg[k] - x0[k]) / (0.05 * H)), [0.0]]) for k in range(nj)])  # :33-36
    xref_ = np.concatenate([th, w]).T.reshape(-1)                                           # :37-40
    xori = xref_[10:]
    Aaug, Baug, Qaug, QQ = problem.build_cost_matrices(robot, nj, H, problem.Q_M16_SCRIPT, np.eye(5), 0.0)
    ff = ((Aaug @ x0 - xori) @ Qaug @ Baug)
    caug = float((Aaug @ x0 - xori) @ Qaug @ (Aaug @ x0 - xori))
    s = dict(Aaug=Aaug, Baug=Baug, QQ=QQ, ff=ff, Qaug=QQ, paug=ff, caug=caug, robot=robot, H=H, nstate=10, njoint=nj, nu=nj,
             xR=x0.reshape(-1, 1), x_=xori, alpha=0.0, lim=None, epsilon_O=0.01, MAX_O_ITER=10,
             MAX_input=0.2 * np.ones(H * nj))
    obs = [{"l": np.array([[3.906, 3.906], [8.313, 8.313], [0.001, 1.938]]), "D": 0.2, "epsilon": 0.2}]
    return "M16iB", robot, obs, s


def rrtstar_route_config(route_wp):
    """RRTstar_CFS.m:96-100: resample an RRT route to H+1 = 41 waypoints, then the CFS stage set-up (:106-187)."""
    route_wp = np.asarray(route_wp, dtype=np.float64)
    dt = 0.5
    wp_t = np.arange(route_wp.shape[1]) * dt
    sampled = problem.cubicpolytraj(route_wp, wp_t, np.linspace(0, wp_t[-1], 41))
    return rrtstar_cfs_config(sampled)


def oracle_problem(O, ROBOT, obs, s, solver=0, grad=0, margin=None, max_input="default"):
    if margin is None:
        margin = [o["epsilon"] if solver == 0 else o["D"] for o in obs]
    mi = s["MAX_input"] if max_input == "default" else max_input
    return O.Problem(O.robot(ROBOT), s["H"], list(obs), margin, s["QQ"], s.get("lim"),
                     mi if solver == 0 else None, s["epsilon_O"], s["MAX_O_ITER"], solver=solver, grad=grad,
                     alpha=s.get("alpha", 0.0))


def oracle_feasible_fn(O, ROBOT, obs):
    r = O.robot(ROBOT)
    o6 = [O.obs6(o) for o in obs]

    def fn(cand):
        return np.array([all(O.dist_arm(r, th, o)[0] >= ob["D"] for o, ob in zip(o6, obs)) for th in cand])
    return fn


def batch_m16ib(O, B, horizon=50, seed=synthetic.SEED):
    return synthetic.batch_config_m16ib(B, oracle_feasible_fn(O, "M16iB", [synthetic.OBS_M16IB]), horizon, seed)


def sampling_box(rng, N):
    return synthetic.SAMPLE_OFF + (rng.random((N, 5)) - 0.5) * 2 * synthetic.REGION_S
