"""CFS_FANUC / PSGCFS_FANUC / EVAL -- host-side mirrors of the reference's solver classes.

Same constructor arguments, same method names and the same result properties as Lib/CFS_FANUC.m, Lib/PSGCFS_FANUC.m
and Lib/EVAL.m, but optimizer() is one call into libcfs_b200.so (B=1 case of cfs_solve_batch).  BatchCFS runs many
independent problems that share robot, obstacles, horizon and weights (the B200 use case).
"""
import numpy as np

from . import _lib


class EVAL:
    """Result holder with the fields of Lib/EVAL.m:33-35 (cost_all, e_cost_all, e_u_all)."""

    def __init__(self, sys_info):
        self.sys_info = sys_info
        self.epsilon_O = sys_info["epsilon_O"]
        self.MAX_O_ITER = sys_info["MAX_O_ITER"]
        self.cost_all = np.zeros(0)
        self.e_cost_all = np.zeros(0)
        self.e_u_all = np.zeros(0)
        self.cost_old = 100000.0  # EVAL.m:29
        self.cost_new = 0.0

    def get_cost(self, u):  # EVAL.m:51-53
        s = self.sys_info
        return 0.5 * u @ s["Qaug"] @ u + s["paug"] @ u + s["caug"]


def _apply_qlim(ctx, sys_info):
    """Joint position limits from the optional sys_info["qlim"] (nj x 2, [min max] per joint; +-inf for a side without a
    limit), or none: a context shared between calls never keeps the limits of an earlier one."""
    q = sys_info.get("qlim")
    if q is None:
        ctx.set_joint_limits(None, None)
    else:
        q = np.asarray(q, dtype=np.float64).reshape(-1, 2)
        ctx.set_joint_limits(q[:, 0], q[:, 1])


class _SolverBase:
    SOLVER = _lib.SOLVER_CFS
    GRAD = _lib.GRAD_NUMJAC

    def __init__(self, obs, sys_info, ROBOT="M16iB", ctx=None, device=0):
        self.obs = obs
        self.sys_info = sys_info
        self.ROBOT = ROBOT
        self.nn = sys_info["H"] * sys_info["nu"]
        self.x_ = np.array(sys_info["x_"], dtype=np.float64).reshape(-1)  # CFS_FANUC.m:55
        self.u = np.zeros(self.nn)                                        # CFS_FANUC.m:56
        self.eval = EVAL(sys_info)
        self.iter_O = 1
        self.total_iter = 0
        self.status = None
        self._ctx = ctx
        self._device = device

    def _context(self):
        if self._ctx is None:
            self._ctx = _lib.Context(self._device)
        ctx = self._ctx
        s = self.sys_info
        robot = dict(s["robot"])
        robot["name"] = self.ROBOT
        ctx.set_robot(robot, s["njoint"])
        ctx.set_obstacles(self.obs)
        ctx.set_cost(s["H"], s["QQ"], s.get("lim"), s.get("MAX_input") if self.SOLVER == _lib.SOLVER_CFS else None)
        _apply_qlim(ctx, s)
        return ctx

    def optimizer(self, noise=None, rng=None, check=None):
        """check=None: the reference's optimizer.  check=dict(eta=1e-3, rounds=4, gain=2.0, max_evals=4096) (any subset): the
        checked solve (Context.solve_checked); the result then also carries verdict, t_hit, cmin, rounds_used and margin_off
        (nobs x H) of the returned trajectory."""
        s = self.sys_info
        ctx = self._context()
        K = int(s["MAX_O_ITER"])
        if self.SOLVER == _lib.SOLVER_PSGCFS and noise is None:
            # PSGCFS_FANUC.m:109 draws normrnd(0,0.1,[nn,1]) in every PSG step; a run without noise would be a different,
            # deterministic method.  Drawn here with the reference's distribution, one row per outer iteration (all
            # MAX_O_ITER rows up front: the reference only draws when a step is taken, INTEGRATION.md).
            noise = (rng or np.random.default_rng()).normal(0.0, 0.1, size=(K, self.nn))
        solve = ctx.solve_batch if check is None else lambda *a, **kw: ctx.solve_checked(*a, **kw, **dict(check))
        out = solve(np.asarray(s["xR"], dtype=np.float64)[:, 0][None], np.asarray(s["ff"])[None],
                    np.array([s["caug"]], dtype=np.float64), self.x_[None], float(s["epsilon_O"]), K,
                    solver=self.SOLVER, grad=self.GRAD,
                    noise=None if noise is None else np.asarray(noise, dtype=np.float64)[None],
                    alpha=float(s.get("alpha", 0.0)))
        if check is not None:
            self.verdict, self.t_hit, self.cmin = int(out["verdict"][0]), float(out["t_hit"][0]), float(out["cmin"][0])
            self.rounds_used, self.margin_off = int(out["rounds_used"][0]), out["margin_off"][0].copy()
        it = int(out["iters"][0])
        self.u = out["u"][0].copy()
        self.x_ = out["x"][0].copy()
        self.status = int(out["status"][0])
        self.iter_O = it + 1
        self.eval.cost_all = out["cost_hist"][0, :it].copy()
        self.eval.e_u_all = out["e_u_hist"][0, :it].copy()
        prev = np.concatenate([[self.eval.get_cost(np.zeros(self.nn))], self.eval.cost_all[:-1]]) if it else np.zeros(0)
        self.eval.e_cost_all = np.abs(prev - self.eval.cost_all)  # EVAL.m:57 (CFS: cost_old is the previous cost)
        if it:
            self.eval.cost_new = float(self.eval.cost_all[-1])
        self.total_iter = ctx.stats()["qp_steps"]
        if (self.status & 0xFF) == _lib.STATUS_INFEASIBLE:
            raise _lib.CfsError("QP infeasible at outer iteration %d (the reference's quadprog returns [] here and "
                                "CFS_FANUC.m:92 throws)" % self.iter_O)
        return self


class CFS_FANUC(_SolverBase):
    """Lib/CFS_FANUC.m: self = CFS_FANUC(obs, sys_info, ROBOT); self = self.optimizer()"""
    SOLVER = _lib.SOLVER_CFS


class PSGCFS_FANUC(_SolverBase):
    """Lib/PSGCFS_FANUC.m; pass the normrnd(0,0.1,[nn,1]) draws (PSGCFS_FANUC.m:109) as noise (MAX_O_ITER, nn)."""
    SOLVER = _lib.SOLVER_PSGCFS


class CHOMP_FANUC(_SolverBase):
    """Lib/CHOMP_FANUC.m: self = CHOMP_FANUC(obs, sys_info, uu, ROBOT); self = self.optimizer()  -- the gradient-descent
    baseline planner: exactly MAX_O_ITER steps u <- u - alpha*3*(QQ*u + ff + 2000*dcostObs) (CHOMP_FANUC.m:54-83)."""

    def __init__(self, obs, sys_info, uu, ROBOT="M16iB", ctx=None, device=0):
        super().__init__(obs, sys_info, ROBOT, ctx=ctx, device=device)
        self.u = np.array(uu, dtype=np.float64).reshape(-1)  # CHOMP_FANUC.m:48

    def optimizer(self):
        s = self.sys_info
        ctx = self._context()
        K = int(s["MAX_O_ITER"])
        out = ctx.chomp_batch(np.asarray(s["xR"], dtype=np.float64)[:, 0][None], np.asarray(s["ff"])[None],
                              np.array([s["caug"]], dtype=np.float64), self.x_[None], self.u[None], float(s["alpha"]), K)
        cost0 = self.eval.get_cost(self.u)  # CHOMP_FANUC.m:55
        self.u = out["u"][0].copy()
        self.x_ = out["x"][0].copy()
        self.status = int(out["status"][0])
        self.iter_O = K + 1
        self.eval.cost_all = out["cost_hist"][0].copy()
        self.eval.e_u_all = out["e_u_hist"][0].copy()
        self.eval.e_cost_all = np.abs(np.concatenate([[cost0], self.eval.cost_all[:-1]]) - self.eval.cost_all)  # EVAL.m:57
        if K:
            self.eval.cost_new = float(self.eval.cost_all[-1])
        return self


class BatchCFS:
    """B independent problems sharing robot / obstacles / horizon / weights: the batched form of CFS_FANUC.optimizer."""

    def __init__(self, obs, sys_info, ROBOT="M16iB", ctx=None, device=0, solver=_lib.SOLVER_CFS, grad=_lib.GRAD_NUMJAC):
        self.ctx = ctx or _lib.Context(device)
        self.sys_info = sys_info
        self.solver, self.grad = solver, grad
        robot = dict(sys_info["robot"])
        robot["name"] = ROBOT
        self.ctx.set_robot(robot, sys_info["njoint"])
        self.ctx.set_obstacles(obs)
        self.ctx.set_cost(sys_info["H"], sys_info["QQ"], sys_info.get("lim"),
                          sys_info.get("MAX_input") if solver == _lib.SOLVER_CFS else None)

    def optimizer(self, x0, ff, caug, xref, noise=None, check=None):
        """check=None: the plain batched solve.  check=dict(eta=1e-3, rounds=4, gain=2.0, max_evals=4096) (any subset): the
        checked solve (Context.solve_checked), whose result adds verdict, t_hit, cmin, rounds_used and margin_off.  Joint
        position limits: sys_info["qlim"] (optional), applied to the context on every call."""
        s = self.sys_info
        _apply_qlim(self.ctx, s)
        if check is not None:
            return self.ctx.solve_checked(x0, ff, caug, xref, float(s["epsilon_O"]), int(s["MAX_O_ITER"]), solver=self.solver,
                                          grad=self.grad, noise=noise, alpha=float(s.get("alpha", 0.0)), **dict(check))
        return self.ctx.solve_batch(x0, ff, caug, xref, float(s["epsilon_O"]), int(s["MAX_O_ITER"]), solver=self.solver,
                                    grad=self.grad, noise=noise, alpha=float(s.get("alpha", 0.0)))
