"""RRT_FANUC / s_Parallel_rrt / the RRT -> CFS pipeline of RRTstar_CFS.m -- host-side mirrors over libcfs_b200.so.

  RRT_FANUC(obs, sys_info, goal, region_g, region_s, sample_off, ROBOT, SOLVER).find_route()    Lib/RRT_FANUC.m:48-91
  s_Parallel_rrt(...)   num_seed trees at once (the parfor of Lib/functions/s_Parallel_rrt.m:11-28), min(routeL)
  rrtstar_cfs(...)      s_Parallel_rrt -> cubicpolytraj -> CFS_FANUC.optimizer                   RRTstar_CFS.m:76-119,194-195

MATLAB's rand stream is an input of the kernels (consumed in the reference's order: pp = rand; rand(nstate,1) when pp < bi,
RRT_FANUC.m:108,111): these mirrors draw it from a numpy Generator, or take it from the caller for parity runs.
"""
import numpy as np

from . import _lib, problem

SCENE_RRTSTAR = dict(  # RRTstar_CFS.m:29-55
    x0=np.array([0.421, 0, -0.0092, -0.0010, -1.5786]),
    goal=np.array([-1.4090, 0.8873, 0.4008, 0.0, 0.4430]),
    region_g=np.array([np.pi / 20, np.pi / 20, np.pi / 10, np.pi / 2, np.pi / 2]),
    region_s=np.array([np.pi / 2, np.pi / 2, np.pi / 2, np.pi / 1.5, np.pi / 1.5]),
    sample_off=np.zeros(5),
    ratial=np.array([1, 1, 0.5, 0.1, 0.1]),
    obs=[{"l": np.array([[3.606, 3.606], [8.413, 8.413], [0.001, 1.038]]), "D": 0.2, "epsilon": 0.2},
         {"l": np.array([[3.406, 3.406], [7.813, 7.813], [0.800, 1.538]]), "D": 0.2, "epsilon": 0.2}])
NRND_DEFAULT = 4096  # uniform numbers per seed: a 400-node tree consumes ~1 + 5*bi numbers per sample, a few rejected samples each


def _bind(ctx, obs, sys_info, ROBOT):
    robot = dict(sys_info["robot"])
    robot["name"] = ROBOT
    ctx.set_robot(robot, int(sys_info["nstate"]))
    ctx.set_obstacles(obs)


class RRT_FANUC:
    """Lib/RRT_FANUC.m: same constructor arguments and result properties (route, fail, node_num, all_nodes, total_dis)."""

    MAX_ITER = 400  # RRT_FANUC.m:37
    bi = 0.5        # RRT_FANUC.m:38

    def __init__(self, obs, sys_info, goal, region_g, region_s, sample_off, ROBOT="M16iB", SOLVER="RRT*", ctx=None, device=0):
        self.obs, self.sys_info, self.goal = obs, sys_info, np.asarray(goal, dtype=np.float64)
        self.region_g, self.region_s, self.sample_off = (np.asarray(v, dtype=np.float64).reshape(-1) for v in (region_g, region_s, sample_off))
        self.ROBOT, self.SOLVER = ROBOT, SOLVER
        self.route = None
        self.fail = False
        self.node_num = 1
        self.all_nodes = None
        self.total_dis = None
        self.rnd_used = 0
        self._ctx = ctx
        self._device = device

    def find_route(self, rnd=None, rng=None):
        """rnd: the uniform numbers this tree consumes (1-D); default: drawn from rng (numpy Generator)."""
        ctx = self._ctx or _lib.Context(self._device)
        self._ctx = ctx
        _bind(ctx, self.obs, self.sys_info, self.ROBOT)
        if rnd is None:
            rnd = (rng or np.random.default_rng()).random(NRND_DEFAULT * 4)
        s = self.sys_info
        out = ctx.rrt_find_routes(np.asarray(s["x0"], dtype=np.float64).reshape(1, -1), self.goal.reshape(1, -1),
                                  np.asarray(s["goal_th"], dtype=np.float64).reshape(1, -1), self.region_g, self.region_s,
                                  self.sample_off, np.asarray(s["ratial"], dtype=np.float64).reshape(-1),
                                  np.asarray(rnd, dtype=np.float64).reshape(1, -1), bi=self.bi, max_iter=self.MAX_ITER,
                                  star=(self.SOLVER == "RRT*"), want_tree=True)
        if out["route_len"][0] < 0:
            raise _lib.CfsError("RRT_FANUC.find_route: the random stream (%d numbers) ran dry" % np.size(rnd))
        nn = int(out["n_nodes"][0])
        self.route = out["routes"][0].T.copy()                      # nstate x routeL, as self.route
        self.fail = bool(out["fail"][0])
        self.node_num = nn
        self.all_nodes = np.vstack([out["parent"][0, :nn][None, :].astype(np.float64),
                                    out["nodes"][0, :nn].T])         # row 1: parent (1-based, -1 for the root), RRT_FANUC.m:66
        self.total_dis = out["total_dis"][0, :nn].copy()
        self.rnd_used = int(out["rnd_used"][0])
        return self


def s_Parallel_rrt(obs, sys_info, goalxyz, region_g, region_s, sample_off, ROBOT="M200i", SOLVER="RRT", num_seed=6, ctx=None,
                   device=0, rng=None, nrnd=NRND_DEFAULT, max_rounds=20):
    """Lib/functions/s_Parallel_rrt.m:11-28: num_seed trees per round until one finds a path, routeL = size(route,2) of the
    successful ones (1000 otherwise), the shortest wins.  Returns dict(route (nstate x L), path_length, id, iter_rrt, routeL,
    routes, fail, ms)."""
    ctx = ctx or _lib.Context(device)
    _bind(ctx, obs, sys_info, ROBOT)
    rng = rng or np.random.default_rng()
    S = int(num_seed)
    tile = lambda v: np.tile(np.asarray(v, dtype=np.float64).reshape(1, -1), (S, 1))
    iter_rrt, ms = 0, 0.0
    while True:
        out = ctx.rrt_find_routes(tile(sys_info["x0"]), tile(goalxyz), tile(sys_info["goal_th"]), region_g, region_s, sample_off,
                                  np.asarray(sys_info["ratial"], dtype=np.float64).reshape(-1), rng.random((S, nrnd)),
                                  star=(SOLVER == "RRT*"))
        iter_rrt += 1
        ms += out["ms"]
        path_fail = out["fail"] | (out["route_len"] < 0)
        routeL = np.where(path_fail, 1000, out["route_len"])          # s_Parallel_rrt.m:14,21
        if not path_fail.all() or iter_rrt >= max_rounds:
            break
    idx = int(np.argmin(routeL))                                       # [path_length, id] = min(routeL)  (:27)
    return dict(route=out["routes"][idx].T.copy(), path_length=int(routeL[idx]), id=idx, iter_rrt=iter_rrt, routeL=routeL,
                routes=out["routes"], fail=path_fail, ms=ms)


def rrtstar_sys_info(robot, x0, goal_th, ratial, nstate=5):
    """sys_info of RRTstar_CFS.m:57-64 (the RRT stage)."""
    return dict(robot=robot, DH=robot["DH"], nstate=nstate, x0=np.asarray(x0, dtype=np.float64), base=robot["base"],
                ratial=np.asarray(ratial, dtype=np.float64), goal_th=np.asarray(goal_th, dtype=np.float64))


def route_edges(routes, route_len):
    """Routes (S, W, nj), the first route_len[s] waypoints of route s valid, -> the edges of their polylines:
    theta_a, theta_b (E, nj) and the route each edge belongs to (E,), ready for Context.check_edges."""
    routes = np.asarray(routes, dtype=np.float64)
    rl = np.minimum(np.maximum(np.asarray(route_len).reshape(-1), 0), routes.shape[1])
    owner = np.repeat(np.arange(routes.shape[0]), np.maximum(rl - 1, 0))
    k = np.concatenate([np.arange(max(n - 1, 0)) for n in rl]).astype(np.int64) if rl.size else np.zeros(0, dtype=np.int64)
    return (np.ascontiguousarray(routes[owner, k]), np.ascontiguousarray(routes[owner, k + 1]), owner)


def combine_verdicts(verdict, owner, n):
    """Per-group verdict of item verdicts: HIT if any item hits, else UNDECIDED if any is, else CLEAR; -1 for a group without
    items (a seed without a route)."""
    out = np.full(n, -1, dtype=np.int32)
    for code in (_lib.CHECK_CLEAR, _lib.CHECK_UNDECIDED, _lib.CHECK_HIT):
        out[np.unique(owner[verdict == code])] = code
    return out


def rrtstar_cfs(ctx, robot, scene=None, ROBOT="M200i", num_seed=6, horizon=40, rng=None, smooth_all=False, nrnd=NRND_DEFAULT,
                check=False):
    """RRTstar_CFS.m end to end on the device: s_Parallel_rrt (:76) -> cubicpolytraj resampling to horizon+1 points (:96-100)
    -> CFS stage set-up (:106-187: R*10, Q_v = [100 20 1 1 1]) -> CFS_FANUC.optimizer (:194-195).
    smooth_all=False: the reference's flow (the shortest route is smoothed).  smooth_all=True: every seed's route is smoothed in
    one batch and the cheapest trajectory wins (the multi-GPU best-of, multi_gpu.best_of, continues this over ranks).
    check=True (extension, include/cfs_b200.h cfs_check_*): continuous collision checks with the default tolerance against
    obs{j}.D -- route_check = per-seed verdict of the route polyline (-1: no route), traj_check = the check of every smoothed
    trajectory; with smooth_all the winner is the cheapest CLEAR trajectory, or the cheapest one if none is CLEAR, and clear says
    which."""
    sc = scene or SCENE_RRTSTAR
    s = rrtstar_sys_info(robot, sc["x0"], sc["goal"], sc["ratial"])
    par = s_Parallel_rrt(sc["obs"], s, sc["goal"], sc["region_g"], sc["region_s"], sc["sample_off"], ROBOT, "RRT", num_seed, ctx=ctx,
                         rng=rng, nrnd=nrnd)
    lim = np.ones(5)
    max_input = np.tile(np.array([1, 1, np.pi, np.pi, np.pi]) * robot["delta_t"], horizon)
    ctx.set_cost_blocks(horizon, problem.Q_RRTSTAR, problem.R_MAIN_FANUC, 10.0, lim, max_input)
    if smooth_all:
        W = max(int(par["routeL"][~par["fail"]].max()) if (~par["fail"]).any() else 2, 2)
        routes = np.zeros((num_seed, W, 5))
        rl = np.zeros(num_seed, dtype=np.int32)
        for k, (r, f) in enumerate(zip(par["routes"], par["fail"])):
            if not f:
                routes[k, :len(r)] = r
                rl[k] = len(r)
        sol = ctx.solve_routes_var(routes, rl, 0.1, 20)
        ok = (sol["status"] & 0xFF) < 2
        fin = np.where(ok & (sol["iters"] > 0), sol["cost_hist"][np.arange(num_seed), np.maximum(sol["iters"], 1) - 1], np.inf)
        win = int(np.argmin(fin))
        if not check:
            return dict(rrt=par, sol=sol, winner=win, cost=float(fin[win]), x=sol["x"][win], u=sol["u"][win])
        route_check = _check_routes(ctx, routes, rl)
        traj = _check_smoothed(ctx, routes[:, 0], sol)
        clear = (traj["verdict"] == _lib.CHECK_CLEAR) & np.isfinite(fin)
        if clear.any():
            win = int(np.argmin(np.where(clear, fin, np.inf)))
        return dict(rrt=par, sol=sol, winner=win, cost=float(fin[win]), x=sol["x"][win], u=sol["u"][win], route_check=route_check,
                    traj_check=traj, clear=bool(clear[win]))
    sol = ctx.solve_routes(par["route"].T[None], 0.1, 20)
    it = int(sol["iters"][0])
    out = dict(rrt=par, sol=sol, winner=par["id"], cost=float(sol["cost_hist"][0, it - 1]) if it else np.inf, x=sol["x"][0],
               u=sol["u"][0])
    if check:
        rl = np.array([len(r) for r in par["routes"]], dtype=np.int32)
        rl[par["fail"]] = 0
        routes = np.zeros((num_seed, max(int(rl.max()), 2), 5))
        for k, r in enumerate(par["routes"]):
            routes[k, :rl[k]] = r[:rl[k]]
        traj = _check_smoothed(ctx, par["route"].T[:1], sol)
        out.update(route_check=_check_routes(ctx, routes, rl), traj_check=traj,
                   clear=bool(traj["verdict"][0] == _lib.CHECK_CLEAR))
    return out


def _check_routes(ctx, routes, route_len):
    ta, tb, owner = route_edges(routes, route_len)
    ev = ctx.check_edges(ta, tb) if owner.size else dict(verdict=np.zeros(0, dtype=np.int32))
    return combine_verdicts(ev["verdict"], owner, routes.shape[0])


def _check_smoothed(ctx, first, sol):
    """first (B, nj): the first waypoint of every route, which is the first resampled point and so x0 = [first; 0]"""
    x0 = np.concatenate([first, np.zeros_like(first)], axis=1)
    return ctx.check_trajectories(x0, sol["x"], sol["u"])
