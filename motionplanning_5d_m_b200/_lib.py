"""ctypes binding of libcfs_b200.so (include/cfs_b200.h) -- the only compute path of this package.

There is no CPU fallback: importing works without a GPU (so host-side logic can be tested), but creating a
Context raises CfsError unless libcfs_b200.so is built and a B200 (sm_100) device is present.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcfs_b200.so")

ROBOT_KIND = {"M16iB": 0, "M200i": 1, "2L": 2}
SOLVER_CFS, SOLVER_PSGCFS = 0, 1
GRAD_NUMJAC, GRAD_DERIVEST = 0, 1
STATUS_CONVERGED, STATUS_MAX_ITER, STATUS_INFEASIBLE, STATUS_NUMERICAL, STATUS_NO_ROUTE = 0, 1, 2, 3, 5
FLAG_TOUCH = 0x100
CHECK_CLEAR, CHECK_HIT, CHECK_UNDECIDED = 0, 1, 2

# every symbol include/cfs_b200.h declares (tests check that the library exports all of them)
SYMBOLS = ["cfs_create", "cfs_destroy", "cfs_last_error", "cfs_version", "cfs_set_stream", "cfs_set_option", "cfs_set_robot", "cfs_set_obstacles", "cfs_set_obstacles_ex",
           "cfs_set_cost", "cfs_set_cost_blocks", "cfs_solve_start_goal", "cfs_solve_start_goal_async", "cfs_solve_routes", "cfs_solve_routes_async", "cfs_solve_routes_var", "cfs_solve_routes_var_async", "cfs_solve_routes_device", "cfs_resample_routes", "cfs_solve_batch", "cfs_solve_batch_async", "cfs_chomp_batch", "cfs_wait", "cfs_solve_batch_device", "cfs_dist_grad", "cfs_time_dist_grad", "cfs_get_con",
           "cfs_nodes_feasible", "cfs_nearest_steer", "cfs_rrt_find_routes", "cfs_rrt_find_routes_device", "cfs_get_stats", "cfs_set_timing", "cfs_get_iter_times", "cfs_get_problem_steps", "cfs_get_qp_profile", "cfs_get_warp_profile", "cfs_measure_fp64_peak",
           "cfs_check_edges", "cfs_check_trajectories", "cfs_check_edges_device", "cfs_check_trajectories_device",
           "cfs_solve_batch_margins", "cfs_solve_batch_margins_device", "cfs_solve_checked", "cfs_solve_checked_device",
           "cfs_set_joint_limits"]


class CfsError(RuntimeError):
    pass


class Stats(C.Structure):
    _fields_ = [("ms_setup", C.c_double), ("ms_total", C.c_double), ("ms_grad", C.c_double), ("ms_qp", C.c_double),
                ("ms_h2d", C.c_double), ("ms_d2h", C.c_double), ("grad_waypoints", C.c_longlong),
                ("problem_iters", C.c_longlong), ("qp_steps", C.c_longlong), ("launches", C.c_int),
                ("max_active", C.c_int), ("ms_bulk", C.c_double), ("ms_heavy", C.c_double)]


_lib = None


def load():
    """Load libcfs_b200.so; fails loudly when the CUDA extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CfsError("libcfs_b200.so is missing (%s): run `python -c 'import __graft_entry__ as g; g.build()'` "
                       "or `make -C motionplanning_5d_m_b200/csrc`. There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    lib.cfs_last_error.restype = C.c_char_p
    lib.cfs_last_error.argtypes = [C.c_void_p]
    lib.cfs_version.restype = C.c_char_p
    lib.cfs_destroy.restype = None
    lib.cfs_destroy.argtypes = [C.c_void_p]
    _lib = lib
    return lib


def _dp(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _f64(a, order="C"):
    return np.require(a, dtype=np.float64, requirements=["C" if order == "C" else "F", "ALIGNED"])


class Context:
    """One cfs_ctx: bound to one CUDA device and one stream (include/cfs_b200.h)."""

    def __init__(self, device=0):
        self._lib = load()
        h = C.c_void_p()
        rc = self._lib.cfs_create(C.byref(h), C.c_int(device))
        if rc != 0:
            raise CfsError("cfs_create failed (%d): %s" % (rc, self._lib.cfs_last_error(None).decode()))
        self._h = h
        self.device = device
        self.nj = self.H = self.n = self.nobs = 0
        self.has_lim = False
        self.has_qlim = False

    def close(self):
        if getattr(self, "_h", None):
            self._lib.cfs_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise CfsError("%s failed (%d): %s" % (what, rc, self._lib.cfs_last_error(self._h).decode()))

    # ---- problem data -------------------------------------------------------------------------------------------
    def set_robot(self, robot, njoint):
        DH = np.asfortranarray(robot["DH"], dtype=np.float64)
        cap = np.zeros((3, 2, njoint), order="F")
        for i in range(njoint):
            cap[:, :, i] = np.asarray(robot["cap"][i]["p"], dtype=np.float64)[:, :2]
        cap = np.asfortranarray(cap)
        base = _f64(np.asarray(robot["base"], dtype=np.float64).reshape(-1))
        T = robot.get("T")
        T = None if T is None else np.asfortranarray(T, dtype=np.float64)
        rc = self._lib.cfs_set_robot(self._h, C.c_int(ROBOT_KIND[robot["name"]]), _dp(DH), C.c_int(DH.shape[0]), _dp(base),
                                     _dp(cap), C.c_int(njoint), _dp(T), C.c_double(robot["delta_t"]))
        self._check(rc, "cfs_set_robot")
        self.nj = njoint
        self.has_qlim = False  # cfs_set_robot clears the joint limits

    def set_joint_limits(self, qmin, qmax):
        """Joint position limits of every following CFS / PSGCFS solve (cfs_set_joint_limits): qmin, qmax (nj,), +-inf for a side
        without a limit; set_joint_limits(None, None) clears them."""
        lo = None if qmin is None else _f64(np.asarray(qmin, dtype=np.float64).reshape(-1))
        hi = None if qmax is None else _f64(np.asarray(qmax, dtype=np.float64).reshape(-1))
        for v in (lo, hi):
            if v is not None and v.shape[0] != self.nj:
                raise CfsError("set_joint_limits: expected %d entries, got %d" % (self.nj, v.shape[0]))
        rc = self._lib.cfs_set_joint_limits(self._h, _dp(lo), _dp(hi))
        self._check(rc, "cfs_set_joint_limits")
        self.has_qlim = lo is not None

    def set_obstacles(self, obs):
        """obs: list of dicts with l (3x2), D, epsilon (main_FANUC.m:56-60).  shape == 'box' (extension): l = [min corner, max
        corner] of a solid axis-aligned box, e.g. from stl_boxes.boxes_from_stl; anything else is a capsule axis."""
        O = len(obs)
        seg = np.zeros((3, 2, max(O, 1)), order="F")
        D = np.zeros(max(O, 1))
        eps = np.zeros(max(O, 1))
        kind = np.zeros(max(O, 1), dtype=np.int32)
        for j, o in enumerate(obs):
            seg[:, :, j] = np.asarray(o["l"], dtype=np.float64)
            D[j] = o.get("D", 0.0)
            eps[j] = o.get("epsilon", 0.0)
            kind[j] = 1 if o.get("shape") == "box" else 0
        rc = self._lib.cfs_set_obstacles_ex(self._h, _dp(np.asfortranarray(seg)), _dp(kind), _dp(D), _dp(eps), C.c_int(O))
        self._check(rc, "cfs_set_obstacles_ex")
        self.nobs = O

    def set_cost(self, H, QQ, lim, max_input):
        QQ = np.asfortranarray(QQ, dtype=np.float64)
        lim_ = None if lim is None else _f64(np.asarray(lim).reshape(-1))
        mi = None if max_input is None else _f64(np.asarray(max_input).reshape(-1))
        rc = self._lib.cfs_set_cost(self._h, C.c_int(H), _dp(QQ), _dp(lim_), _dp(mi))
        self._check(rc, "cfs_set_cost")
        self.H, self.n = H, H * self.nj
        self.has_lim = lim is not None

    def set_cost_blocks(self, H, Q, Rblk, r_scale, lim, max_input, stage_w=0.1, term_w=10000.0):
        """QQ = Baug'QaugBaug + r_scale (R+R') built on the device from its blocks (main_FANUC.m:64-97)."""
        Q = np.asfortranarray(Q, dtype=np.float64)
        Rb = np.asfortranarray(Rblk, dtype=np.float64)
        lim_ = None if lim is None else _f64(np.asarray(lim).reshape(-1))
        mi = None if max_input is None else _f64(np.asarray(max_input).reshape(-1))
        rc = self._lib.cfs_set_cost_blocks(self._h, C.c_int(H), _dp(Q), _dp(Rb), C.c_double(r_scale), C.c_double(stage_w),
                                           C.c_double(term_w), _dp(lim_), _dp(mi))
        self._check(rc, "cfs_set_cost_blocks")
        self.H, self.n = H, H * self.nj
        self.has_lim = lim is not None

    def solve_start_goal(self, theta0, thetag, eps_outer, max_outer, solver=SOLVER_CFS, grad=GRAD_NUMJAC, noise=None,
                         alpha=0.0, want_x=True):
        """theta0, thetag (B,nj): the mains' problem set-up (straight-line reference, ff, caug) is built on the device."""
        t0, tg = _f64(theta0), _f64(thetag)
        B = t0.shape[0]
        n, N, K = self.n, 2 * self.n, max(int(max_outer), 1)
        out = dict(u=np.zeros((B, n)), x=np.zeros((B, N)) if want_x else None, cost_hist=np.full((B, K), np.nan),
                   e_u_hist=np.full((B, K), np.nan), iters=np.zeros(B, dtype=np.int32), status=np.zeros(B, dtype=np.int32))
        nz = None if noise is None else _f64(noise)
        rc = self._lib.cfs_solve_start_goal(self._h, C.c_int(B), C.c_int(solver), C.c_int(grad), _dp(t0), _dp(tg), _dp(nz),
                                            C.c_double(eps_outer), C.c_int(max_outer), C.c_double(alpha), _dp(out["u"]),
                                            _dp(out["x"]), _dp(out["cost_hist"]), _dp(out["e_u_hist"]), _dp(out["iters"]),
                                            _dp(out["status"]))
        self._check(rc, "cfs_solve_start_goal")
        return out

    def solve_routes(self, routes, eps_outer, max_outer, solver=SOLVER_CFS, grad=GRAD_NUMJAC, noise=None, alpha=0.0):
        """routes (B, W, nj): RRT routes; resampling (cubicpolytraj, RRTstar_CFS.m:96-100) and the CFS stage set-up
        (:106-163) run on the device, then optimizer()."""
        r = _f64(routes)
        B, W = r.shape[0], r.shape[1]
        n, N, K = self.n, 2 * self.n, max(int(max_outer), 1)
        out = dict(u=np.zeros((B, n)), x=np.zeros((B, N)), cost_hist=np.full((B, K), np.nan), e_u_hist=np.full((B, K), np.nan),
                   iters=np.zeros(B, dtype=np.int32), status=np.zeros(B, dtype=np.int32))
        nz = None if noise is None else _f64(noise)
        rc = self._lib.cfs_solve_routes(self._h, C.c_int(B), C.c_int(W), C.c_int(solver), C.c_int(grad), _dp(r), _dp(nz),
                                        C.c_double(eps_outer), C.c_int(max_outer), C.c_double(alpha), _dp(out["u"]),
                                        _dp(out["x"]), _dp(out["cost_hist"]), _dp(out["e_u_hist"]), _dp(out["iters"]),
                                        _dp(out["status"]))
        self._check(rc, "cfs_solve_routes")
        return out

    def solve_routes_var(self, routes, route_len, eps_outer, max_outer, solver=SOLVER_CFS, grad=GRAD_NUMJAC, noise=None, alpha=0.0):
        """routes (B, W, nj) padded, route_len (B,): one RRT route per seed (s_Parallel_rrt.m:16-25), all smoothed in one call;
        route_len < 2 (failed seed) -> status STATUS_NO_ROUTE."""
        r = _f64(routes)
        rl = np.require(route_len, dtype=np.int32, requirements=["C", "ALIGNED"])
        B, W = r.shape[0], r.shape[1]
        n, N, K = self.n, 2 * self.n, max(int(max_outer), 1)
        out = dict(u=np.zeros((B, n)), x=np.zeros((B, N)), cost_hist=np.full((B, K), np.nan), e_u_hist=np.full((B, K), np.nan),
                   iters=np.zeros(B, dtype=np.int32), status=np.zeros(B, dtype=np.int32))
        nz = None if noise is None else _f64(noise)
        rc = self._lib.cfs_solve_routes_var(self._h, C.c_int(B), C.c_int(W), _dp(rl), C.c_int(solver), C.c_int(grad), _dp(r), _dp(nz),
                                            C.c_double(eps_outer), C.c_int(max_outer), C.c_double(alpha), _dp(out["u"]),
                                            _dp(out["x"]), _dp(out["cost_hist"]), _dp(out["e_u_hist"]), _dp(out["iters"]),
                                            _dp(out["status"]))
        self._check(rc, "cfs_solve_routes_var")
        return out

    def solve_routes_var_ptr(self, B, W, route_len, routes, eps_outer, max_outer, u, x, cost_hist, e_u_hist, iters, status,
                             solver=SOLVER_CFS, grad=GRAD_NUMJAC, device=False, sync=True):
        """Raw-pointer entry (ints): host pointers (cfs_solve_routes_var[_async]) or device pointers (cfs_solve_routes_device)."""
        vp = lambda p: C.c_void_p(p) if p else None
        if device:
            rc = self._lib.cfs_solve_routes_device(self._h, C.c_int(B), C.c_int(W), vp(route_len), C.c_int(solver), C.c_int(grad),
                                                   vp(routes), None, C.c_double(eps_outer), C.c_int(max_outer), C.c_double(0.0),
                                                   vp(u), vp(x), vp(cost_hist), vp(e_u_hist), vp(iters), vp(status),
                                                   C.c_int(1 if sync else 0))
            self._check(rc, "cfs_solve_routes_device")
        else:
            fn = self._lib.cfs_solve_routes_var if sync else self._lib.cfs_solve_routes_var_async
            rc = fn(self._h, C.c_int(B), C.c_int(W), vp(route_len), C.c_int(solver), C.c_int(grad), vp(routes), None,
                    C.c_double(eps_outer), C.c_int(max_outer), C.c_double(0.0), vp(u), vp(x), vp(cost_hist), vp(e_u_hist),
                    vp(iters), vp(status))
            self._check(rc, "cfs_solve_routes_var")

    def rrt_find_routes_device_ptr(self, S, star, x0, goal, goal_th, params, bi, max_iter, rnd, nrnd, routes, route_len, n_nodes,
                                   fail, rnd_used, route_len_or_fail=0, sync=False):
        """cfs_rrt_find_routes_device: every argument a device pointer (int)."""
        vp = lambda p: C.c_void_p(p) if p else None
        rc = self._lib.cfs_rrt_find_routes_device(self._h, C.c_int(S), C.c_int(1 if star else 0), vp(x0), vp(goal), vp(goal_th),
                                                  vp(params), C.c_double(bi), C.c_int(max_iter), vp(rnd), C.c_int(nrnd),
                                                  vp(routes), vp(route_len), vp(n_nodes), vp(fail), vp(rnd_used),
                                                  vp(route_len_or_fail), C.c_int(1 if sync else 0))
        self._check(rc, "cfs_rrt_find_routes_device")

    def resample_routes(self, routes, H):
        """routes (B, W, nj) -> (B, H+1, nj): cubicpolytraj(route, (0:W-1)*dt, linspace(0,(W-1)*dt,H+1)) on the device."""
        r = _f64(routes)
        B, W = r.shape[0], r.shape[1]
        out = np.zeros((B, H + 1, self.nj))
        self._check(self._lib.cfs_resample_routes(self._h, C.c_int(B), C.c_int(W), C.c_int(H), _dp(r), _dp(out)),
                    "cfs_resample_routes")
        return out

    def solve_start_goal_ptr(self, B, theta0, thetag, eps_outer, max_outer, u, x, cost_hist, e_u_hist, iters, status,
                             solver=SOLVER_CFS, grad=GRAD_NUMJAC, sync=True):
        vp = lambda p: C.c_void_p(p) if p else None
        fn = self._lib.cfs_solve_start_goal if sync else self._lib.cfs_solve_start_goal_async
        rc = fn(self._h, C.c_int(B), C.c_int(solver), C.c_int(grad), vp(theta0), vp(thetag), None, C.c_double(eps_outer),
                C.c_int(max_outer), C.c_double(0.0), vp(u), vp(x), vp(cost_hist), vp(e_u_hist), vp(iters), vp(status))
        self._check(rc, "cfs_solve_start_goal")

    # ---- hot path ---------------------------------------------------------------------------------------------------
    def solve_batch(self, x0, ff, caug, xref, eps_outer, max_outer, solver=SOLVER_CFS, grad=GRAD_NUMJAC, noise=None,
                    alpha=0.0, out=None):
        """x0 (B,2nj), ff (B,n), caug (B,), xref (B,2njH), noise (B,max_outer,n) -- row b = problem b
        (the C ABI's column-major 'n x B' is exactly this C-contiguous (B,n) array)."""
        x0, ff, caug, xref = _f64(x0), _f64(ff), _f64(caug), _f64(xref)
        B = x0.shape[0]
        if not getattr(self, "n", 0):
            raise CfsError("cost not set (cfs_set_cost)")
        n, N = self.n, 2 * self.n
        assert x0.shape == (B, 2 * self.nj) and ff.shape == (B, n) and xref.shape == (B, N) and caug.shape == (B,)
        nz = None if noise is None else _f64(noise)
        if out is None:
            out = dict(u=np.empty((B, n)), x=np.empty((B, N)), cost_hist=np.empty((B, max_outer)),
                       e_u_hist=np.empty((B, max_outer)), iters=np.empty(B, dtype=np.int32),
                       status=np.empty(B, dtype=np.int32))
        rc = self._lib.cfs_solve_batch(self._h, C.c_int(B), C.c_int(solver), C.c_int(grad), _dp(x0), _dp(ff), _dp(caug),
                                       _dp(xref), _dp(nz), C.c_double(eps_outer), C.c_int(max_outer), C.c_double(alpha),
                                       _dp(out["u"]), _dp(out["x"]), _dp(out["cost_hist"]), _dp(out["e_u_hist"]),
                                       _dp(out["iters"]), _dp(out["status"]))
        self._check(rc, "cfs_solve_batch")
        return out

    def solve_batch_margins(self, x0, ff, caug, xref, margin_off, eps_outer, max_outer, solver=SOLVER_CFS, grad=GRAD_NUMJAC,
                            noise=None, alpha=0.0):
        """solve_batch with per-waypoint margin offsets margin_off (B, nobs, H) or None (cfs_solve_batch_margins): the obstacle
        row of (j, i) uses dist - (margin_j + margin_off[b, j, i - 1])."""
        x0, ff, caug, xref = _f64(x0), _f64(ff), _f64(caug), _f64(xref)
        B = x0.shape[0]
        if not getattr(self, "n", 0):
            raise CfsError("cost not set (cfs_set_cost)")
        n, N = self.n, 2 * self.n
        assert x0.shape == (B, 2 * self.nj) and ff.shape == (B, n) and xref.shape == (B, N) and caug.shape == (B,)
        off = None if margin_off is None else _f64(margin_off).reshape(B, self.nobs * self.H)
        nz = None if noise is None else _f64(noise)
        out = dict(u=np.empty((B, n)), x=np.empty((B, N)), cost_hist=np.empty((B, max_outer)), e_u_hist=np.empty((B, max_outer)),
                   iters=np.empty(B, dtype=np.int32), status=np.empty(B, dtype=np.int32))
        rc = self._lib.cfs_solve_batch_margins(self._h, C.c_int(B), C.c_int(solver), C.c_int(grad), _dp(x0), _dp(ff), _dp(caug),
                                               _dp(xref), _dp(nz), _dp(off), C.c_double(eps_outer), C.c_int(max_outer),
                                               C.c_double(alpha), _dp(out["u"]), _dp(out["x"]), _dp(out["cost_hist"]),
                                               _dp(out["e_u_hist"]), _dp(out["iters"]), _dp(out["status"]))
        self._check(rc, "cfs_solve_batch_margins")
        return out

    def solve_checked(self, x0, ff, caug, xref, eps_outer, max_outer, eta=1e-3, rounds=4, gain=2.0, max_evals=4096,
                      solver=SOLVER_CFS, grad=GRAD_NUMJAC, noise=None, alpha=0.0):
        """Checked solve (cfs_solve_checked): the solve, a continuous check of every trajectory, and up to `rounds` re-solves of
        the HIT ones with raised per-waypoint margins.  Returns the solve's dict plus verdict, t_hit, cmin, rounds_used (B,) and
        margin_off (B, nobs, H)."""
        x0, ff, caug, xref = _f64(x0), _f64(ff), _f64(caug), _f64(xref)
        B = x0.shape[0]
        if not getattr(self, "n", 0):
            raise CfsError("cost not set (cfs_set_cost)")
        n, N = self.n, 2 * self.n
        assert x0.shape == (B, 2 * self.nj) and ff.shape == (B, n) and xref.shape == (B, N) and caug.shape == (B,)
        nz = None if noise is None else _f64(noise)
        out = dict(u=np.empty((B, n)), x=np.empty((B, N)), cost_hist=np.empty((B, max_outer)), e_u_hist=np.empty((B, max_outer)),
                   iters=np.empty(B, dtype=np.int32), status=np.empty(B, dtype=np.int32), verdict=np.empty(B, dtype=np.int32),
                   t_hit=np.empty(B), cmin=np.empty(B), rounds_used=np.empty(B, dtype=np.int32),
                   margin_off=np.zeros((B, self.nobs, self.H)))
        rc = self._lib.cfs_solve_checked(self._h, C.c_int(B), C.c_int(solver), C.c_int(grad), _dp(x0), _dp(ff), _dp(caug), _dp(xref),
                                         _dp(nz), C.c_double(eps_outer), C.c_int(max_outer), C.c_double(alpha), C.c_double(eta),
                                         C.c_int(max_evals), C.c_int(rounds), C.c_double(gain), _dp(out["u"]), _dp(out["x"]),
                                         _dp(out["cost_hist"]), _dp(out["e_u_hist"]), _dp(out["iters"]), _dp(out["status"]),
                                         _dp(out["verdict"]), _dp(out["t_hit"]), _dp(out["cmin"]), _dp(out["rounds_used"]),
                                         _dp(out["margin_off"]))
        self._check(rc, "cfs_solve_checked")
        return out

    def solve_batch_margins_ptr(self, B, x0, ff, caug, xref, margin_off, eps_outer, max_outer, u, x, cost_hist, e_u_hist, iters,
                                status, solver=SOLVER_CFS, grad=GRAD_NUMJAC, noise=0, alpha=0.0, sync=True):
        """cfs_solve_batch_margins_device: every array argument a device pointer (int; margin_off, noise, e_u_hist may be 0)."""
        vp = lambda p: C.c_void_p(p) if p else None
        rc = self._lib.cfs_solve_batch_margins_device(self._h, C.c_int(B), C.c_int(solver), C.c_int(grad), vp(x0), vp(ff), vp(caug),
                                                      vp(xref), vp(noise), vp(margin_off), C.c_double(eps_outer), C.c_int(max_outer),
                                                      C.c_double(alpha), vp(u), vp(x), vp(cost_hist), vp(e_u_hist), vp(iters),
                                                      vp(status), C.c_int(1 if sync else 0))
        self._check(rc, "cfs_solve_batch_margins_device")

    def solve_checked_ptr(self, B, x0, ff, caug, xref, eps_outer, max_outer, u, x, cost_hist, e_u_hist, iters, status, verdict, t_hit,
                          cmin, rounds_used, margin_off=0, eta=1e-3, rounds=4, gain=2.0, max_evals=4096, solver=SOLVER_CFS,
                          grad=GRAD_NUMJAC, noise=0, alpha=0.0, sync=True):
        """cfs_solve_checked_device: every array argument a device pointer (int; margin_off, noise, e_u_hist may be 0)."""
        vp = lambda p: C.c_void_p(p) if p else None
        rc = self._lib.cfs_solve_checked_device(self._h, C.c_int(B), C.c_int(solver), C.c_int(grad), vp(x0), vp(ff), vp(caug),
                                                vp(xref), vp(noise), C.c_double(eps_outer), C.c_int(max_outer), C.c_double(alpha),
                                                C.c_double(eta), C.c_int(max_evals), C.c_int(rounds), C.c_double(gain), vp(u), vp(x),
                                                vp(cost_hist), vp(e_u_hist), vp(iters), vp(status), vp(verdict), vp(t_hit), vp(cmin),
                                                vp(rounds_used), vp(margin_off), C.c_int(1 if sync else 0))
        self._check(rc, "cfs_solve_checked_device")

    def chomp_batch(self, x0, ff, caug, xref, u_init, alpha, max_outer):
        """CHOMP_FANUC.optimizer (Lib/CHOMP_FANUC.m:54-165) for B problems: x0 (B,2nj), ff (B,n), caug (B,), xref (B,2njH),
        u_init (B,n) = the constructor's uu.  Exactly max_outer gradient steps per problem (cfs_chomp_batch)."""
        x0, ff, caug, xref, u_init = _f64(x0), _f64(ff), _f64(caug), _f64(xref), _f64(u_init)
        B = x0.shape[0]
        if not getattr(self, "n", 0):
            raise CfsError("cost not set (cfs_set_cost)")
        n, N = self.n, 2 * self.n
        assert x0.shape == (B, 2 * self.nj) and ff.shape == (B, n) and xref.shape == (B, N) and caug.shape == (B,)
        assert u_init.shape == (B, n)
        out = dict(u=np.empty((B, n)), x=np.empty((B, N)), cost_hist=np.empty((B, max_outer)),
                   e_u_hist=np.empty((B, max_outer)), iters=np.empty(B, dtype=np.int32), status=np.empty(B, dtype=np.int32))
        rc = self._lib.cfs_chomp_batch(self._h, C.c_int(B), _dp(x0), _dp(ff), _dp(caug), _dp(xref), _dp(u_init),
                                       C.c_double(alpha), C.c_int(max_outer), _dp(out["u"]), _dp(out["x"]),
                                       _dp(out["cost_hist"]), _dp(out["e_u_hist"]), _dp(out["iters"]), _dp(out["status"]))
        self._check(rc, "cfs_chomp_batch")
        return out

    def solve_batch_ptr(self, B, x0, ff, caug, xref, eps_outer, max_outer, u, x, cost_hist, e_u_hist, iters, status,
                        solver=SOLVER_CFS, grad=GRAD_NUMJAC, noise=0, alpha=0.0, device=False, sync=True):
        """Raw-pointer entry (ints): host pointers (e.g. pinned) or, with device=True, device pointers."""
        vp = lambda p: C.c_void_p(p) if p else None
        if device:
            rc = self._lib.cfs_solve_batch_device(self._h, C.c_int(B), C.c_int(solver), C.c_int(grad), vp(x0), vp(ff),
                                                  vp(caug), vp(xref), vp(noise), C.c_double(eps_outer),
                                                  C.c_int(max_outer), C.c_double(alpha), vp(u), vp(x), vp(cost_hist),
                                                  vp(e_u_hist), vp(iters), vp(status), C.c_int(1 if sync else 0))
            self._check(rc, "cfs_solve_batch_device")
        else:
            fn = self._lib.cfs_solve_batch if sync else self._lib.cfs_solve_batch_async
            rc = fn(self._h, C.c_int(B), C.c_int(solver), C.c_int(grad), vp(x0), vp(ff), vp(caug), vp(xref), vp(noise),
                    C.c_double(eps_outer), C.c_int(max_outer), C.c_double(alpha), vp(u), vp(x), vp(cost_hist),
                    vp(e_u_hist), vp(iters), vp(status))
            self._check(rc, "cfs_solve_batch" if sync else "cfs_solve_batch_async")

    def wait(self):
        """Block until the batch enqueued with sync=False has finished; collects its statistics."""
        self._check(self._lib.cfs_wait(self._h), "cfs_wait")

    def dist_grad(self, theta, grad=GRAD_NUMJAC):
        """theta (N,nj) -> dist (N,nobs), linkid (N,nobs), grad (N,nobs,nj), flags (N,)"""
        theta = _f64(theta)
        N = theta.shape[0]
        O = max(self.nobs, 1)
        dist = np.zeros((N, O))
        lid = np.zeros((N, O), dtype=np.int32)
        g = np.zeros((N, O, self.nj))
        flags = np.zeros(N, dtype=np.int32)
        rc = self._lib.cfs_dist_grad(self._h, C.c_int(N), C.c_int(grad), _dp(theta), _dp(dist), _dp(lid), _dp(g),
                                     _dp(flags))
        self._check(rc, "cfs_dist_grad")
        return dist, lid, g, flags

    def time_dist_grad(self, theta, grad=GRAD_NUMJAC, reps=10):
        """Average device time (ms) of one stand-alone distance/gradient kernel launch over theta (N,nj) resident in HBM."""
        theta = _f64(theta)
        ms = C.c_double()
        rc = self._lib.cfs_time_dist_grad(self._h, C.c_int(theta.shape[0]), C.c_int(grad), _dp(theta), C.c_int(reps),
                                          C.byref(ms))
        self._check(rc, "cfs_time_dist_grad")
        return ms.value

    def get_con(self, x0, xcur, u, grad=GRAD_NUMJAC, margin_is_D=False):
        m = self.nobs * self.H * ((1 + 2 * self.nj) if self.has_lim else 1) + (2 * self.n if self.has_qlim else 0)
        A = np.zeros((m, self.n), order="F")
        b = np.zeros(m)
        rc = self._lib.cfs_get_con(self._h, C.c_int(grad), C.c_int(1 if margin_is_D else 0), _dp(_f64(x0)),
                                   _dp(_f64(xcur)), _dp(_f64(u)), _dp(A), _dp(b))
        self._check(rc, "cfs_get_con")
        return A, b

    def nodes_feasible(self, theta):
        theta = _f64(theta)
        N = theta.shape[0]
        feas = np.zeros(N, dtype=np.uint8)
        dmin = np.zeros(N)
        rc = self._lib.cfs_nodes_feasible(self._h, C.c_int(N), _dp(theta), _dp(feas), _dp(dmin))
        self._check(rc, "cfs_nodes_feasible")
        return feas.astype(bool), dmin

    def check_edges(self, theta_a, theta_b, eta=1e-3, margin_is_D=True, max_evals=4096):
        """Continuous collision check of the joint-space edges theta_a[i] -> theta_b[i] ((N, nj) each; include/cfs_b200.h).
        Returns dict(verdict (CHECK_CLEAR / CHECK_HIT / CHECK_UNDECIDED), s_hit (-1 if none), cmin, evals), each (N,)."""
        ta, tb = _f64(theta_a), _f64(theta_b)
        N = ta.shape[0]
        assert ta.shape == (N, self.nj) and tb.shape == ta.shape
        out = dict(verdict=np.zeros(N, dtype=np.int32), s_hit=np.zeros(N), cmin=np.zeros(N), evals=np.zeros(N, dtype=np.int32))
        rc = self._lib.cfs_check_edges(self._h, C.c_int(N), _dp(ta), _dp(tb), C.c_double(eta), C.c_int(1 if margin_is_D else 0),
                                       C.c_int(max_evals), _dp(out["verdict"]), _dp(out["s_hit"]), _dp(out["cmin"]),
                                       _dp(out["evals"]))
        self._check(rc, "cfs_check_edges")
        return out

    def check_trajectories(self, x0, x, u, eta=1e-3, margin_is_D=True, max_evals=4096):
        """Continuous collision check of B solved trajectories: x0 (B, 2nj), x (B, 2njH) the roll-out of u (B, njH), as every
        solve returns them.  Returns dict(verdict, t_hit (-1 if none), cmin, evals), each (B,)."""
        x0, x, u = _f64(x0), _f64(x), _f64(u)
        B = x0.shape[0]
        H = u.shape[1] // self.nj
        assert x0.shape == (B, 2 * self.nj) and u.shape == (B, H * self.nj) and x.shape == (B, 2 * H * self.nj)
        out = dict(verdict=np.zeros(B, dtype=np.int32), t_hit=np.zeros(B), cmin=np.zeros(B), evals=np.zeros(B, dtype=np.int32))
        rc = self._lib.cfs_check_trajectories(self._h, C.c_int(B), C.c_int(max(H, 1)), _dp(x0), _dp(x), _dp(u), C.c_double(eta),
                                              C.c_int(1 if margin_is_D else 0), C.c_int(max_evals), _dp(out["verdict"]),
                                              _dp(out["t_hit"]), _dp(out["cmin"]), _dp(out["evals"]))
        self._check(rc, "cfs_check_trajectories")
        return out

    def check_edges_ptr(self, N, theta_a, theta_b, verdict, s_hit, cmin, evals, eta=1e-3, margin_is_D=True, max_evals=4096,
                        sync=True):
        """cfs_check_edges_device: every array argument a device pointer (int; evals may be 0)."""
        vp = lambda p: C.c_void_p(p) if p else None
        rc = self._lib.cfs_check_edges_device(self._h, C.c_int(N), vp(theta_a), vp(theta_b), C.c_double(eta),
                                              C.c_int(1 if margin_is_D else 0), C.c_int(max_evals), vp(verdict), vp(s_hit),
                                              vp(cmin), vp(evals), C.c_int(1 if sync else 0))
        self._check(rc, "cfs_check_edges_device")

    def check_trajectories_ptr(self, B, H, x0, x, u, verdict, t_hit, cmin, evals, eta=1e-3, margin_is_D=True, max_evals=4096,
                               sync=True):
        """cfs_check_trajectories_device: every array argument a device pointer (int; evals may be 0)."""
        vp = lambda p: C.c_void_p(p) if p else None
        rc = self._lib.cfs_check_trajectories_device(self._h, C.c_int(B), C.c_int(H), vp(x0), vp(x), vp(u), C.c_double(eta),
                                                     C.c_int(1 if margin_is_D else 0), C.c_int(max_evals), vp(verdict),
                                                     vp(t_hit), vp(cmin), vp(evals), C.c_int(1 if sync else 0))
        self._check(rc, "cfs_check_trajectories_device")

    def nearest_steer(self, nodes, samples, ratial, step=0.1):
        nodes, samples = _f64(nodes), _f64(samples)
        S = samples.shape[0]
        parent = np.zeros(S, dtype=np.int32)
        new = np.zeros((S, self.nj))
        rc = self._lib.cfs_nearest_steer(self._h, C.c_int(nodes.shape[0]), _dp(nodes), C.c_int(S), _dp(samples),
                                         _dp(_f64(ratial)), C.c_double(step), _dp(parent), _dp(new))
        self._check(rc, "cfs_nearest_steer")
        return parent, new

    def rrt_find_routes(self, x0, goal, goal_th, region_g, region_s, sample_off, ratial, rnd, bi=0.5, max_iter=400, star=True,
                        want_tree=False):
        """RRT_FANUC.find_route for S seeds: x0, goal, goal_th (S,nj); rnd (S,nrnd) uniform numbers consumed in MATLAB's
        order.  Returns dict(routes [list of (len,nj)], route_len, n_nodes, fail, rnd_used, ms [, nodes, parent, total_dis])."""
        x0, goal, goal_th, rnd = _f64(x0), _f64(goal), _f64(goal_th), _f64(rnd)
        S, nj, cap = x0.shape[0], self.nj, max_iter + 2
        routes = np.zeros((S, cap, nj))
        ln, nn, fl, ru = (np.zeros(S, dtype=np.int32) for _ in range(4))
        tn = np.zeros((S, cap, nj)) if want_tree else None
        tp = np.zeros((S, cap), dtype=np.int32) if want_tree else None
        tt = np.zeros((S, cap)) if want_tree else None
        ms = C.c_double(0.0)
        rc = self._lib.cfs_rrt_find_routes(self._h, C.c_int(S), C.c_int(1 if star else 0), _dp(x0), _dp(goal), _dp(goal_th),
                                           _dp(_f64(region_g)), _dp(_f64(region_s)), _dp(_f64(sample_off)), _dp(_f64(ratial)),
                                           C.c_double(bi), C.c_int(max_iter), _dp(rnd), C.c_int(rnd.shape[1]), _dp(routes),
                                           _dp(ln), _dp(nn), _dp(fl), _dp(ru), _dp(tn), _dp(tp), _dp(tt), C.byref(ms))
        self._check(rc, "cfs_rrt_find_routes")
        out = dict(routes=[routes[s, :max(ln[s], 0)].copy() for s in range(S)], route_len=ln, n_nodes=nn, fail=fl.astype(bool),
                   rnd_used=ru, ms=ms.value)
        if want_tree:
            out.update(nodes=tn, parent=tp, total_dis=tt)
        return out

    def stats(self):
        s = Stats()
        self._check(self._lib.cfs_get_stats(self._h, C.byref(s)), "cfs_get_stats")
        return {k: getattr(s, k) for k, _ in Stats._fields_}

    def set_stream(self, cuda_stream):
        """cuda_stream: integer cudaStream_t handle (e.g. torch.cuda.current_stream().cuda_stream) or 0/None."""
        self._check(self._lib.cfs_set_stream(self._h, C.c_void_p(cuda_stream or None)), "cfs_set_stream")

    def set_option(self, name, value):
        self._check(self._lib.cfs_set_option(self._h, C.c_char_p(name.encode()), C.c_int(int(value))), "cfs_set_option")

    def set_timing(self, level):
        self._check(self._lib.cfs_set_timing(self._h, C.c_int(level)), "cfs_set_timing")

    def iter_times(self, cap=256):
        g = np.zeros(cap)
        q = np.zeros(cap)
        cnt = self._lib.cfs_get_iter_times(self._h, _dp(g), _dp(q), C.c_int(cap))
        return g[:max(cnt, 0)], q[:max(cnt, 0)]

    def problem_steps(self, B):
        st = np.zeros(B, dtype=np.int32)
        self._check(self._lib.cfs_get_problem_steps(self._h, _dp(st), C.c_int(B)), "cfs_get_problem_steps")
        return st

    def qp_profile(self):
        o = np.zeros(16, dtype=np.int64)
        self._check(self._lib.cfs_get_qp_profile(self._h, _dp(o)), "cfs_get_qp_profile")
        return o

    def warp_profile(self):
        o = np.zeros(6, dtype=np.int64)
        self._check(self._lib.cfs_get_warp_profile(self._h, _dp(o)), "cfs_get_warp_profile")
        return o

    def measure_fp64_peak(self):
        tf, mhz = C.c_double(), C.c_double()
        self._check(self._lib.cfs_measure_fp64_peak(self._h, C.byref(tf), C.byref(mhz)), "cfs_measure_fp64_peak")
        return tf.value, mhz.value
