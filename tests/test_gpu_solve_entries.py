"""GPU tests of the solve family of the C ABI as a whole: every entry that solves the same problems returns the same bits and
launches the same kernels, every entry rejects the same invalid calls with the same return codes, and the copy times of
cfs_get_stats belong to the host-pointer forms."""
import ctypes as C

import numpy as np
import pytest

import motionplanning_5d_m_b200 as M
from motionplanning_5d_m_b200 import _lib, problem
from tests import common
from tests.test_limits import limit_box

pytestmark = pytest.mark.gpu
KEYS = ("u", "x", "cost_hist", "e_u_hist", "iters", "status")
CHECKED = dict(eta=1e-3, max_evals=4096, rounds=0, gain=2.0)
OBS2 = {"l": np.array(common.OBS_M16_SCRIPT_ALT), "D": 0.2, "epsilon": 0.2}
E_ARG, E_STATE = -1, -3


@pytest.fixture(scope="module")
def sctx():
    """a context of its own: the joint limits set here never reach the session context"""
    c = M.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def cfg(oracle):
    """a seeded M16iB batch with two obstacles, and routes through its start and goal points (W = 6 waypoints)"""
    c = common.batch_m16ib(oracle, 96)
    c["obs"] = c["obs"] + [OBS2]
    t = np.linspace(0.0, 1.0, 6)[None, :, None]
    bend = np.random.default_rng(17).normal(0.0, 0.05, (96, 1, 5)) * np.sin(np.pi * t)
    c["routes"] = np.ascontiguousarray(c["theta0"][:, None] + t * (c["thetag"] - c["theta0"])[:, None] + bend)
    return c


def _set(c, cfg, blocks=False, limits=False):
    s = cfg["sys_info"]
    c.set_robot(dict(cfg["robot"], name="M16iB"), 5)
    c.set_obstacles(cfg["obs"])
    if blocks:
        c.set_cost_blocks(s["H"], problem.Q_MAIN_FANUC, problem.R_MAIN_FANUC, 50.0, s["lim"], s["MAX_input"])
    else:
        c.set_cost(s["H"], s["QQ"], s["lim"], s["MAX_input"])
    c.set_joint_limits(*(limit_box() if limits else (None, None)))
    return s


def _outs(B, n, K, kind):
    """the six solve outputs: numpy ("pageable"), pinned torch ("pinned") or device torch ("device") arrays"""
    import torch
    shapes = dict(u=(B, n), x=(B, 2 * n), cost_hist=(B, K), e_u_hist=(B, K), iters=(B,), status=(B,))
    if kind == "pageable":
        return {k: np.zeros(sh, dtype=np.int32 if k in ("iters", "status") else np.float64) for k, sh in shapes.items()}
    out = {k: torch.zeros(sh, dtype=torch.int32 if k in ("iters", "status") else torch.float64) for k, sh in shapes.items()}
    return {k: (v.pin_memory() if kind == "pinned" else v.cuda()) for k, v in out.items()}


def _ptr(v):
    return v.ctypes.data if isinstance(v, np.ndarray) else v.data_ptr()


def _numpy(out):
    import torch
    torch.cuda.synchronize()
    return {k: (v if isinstance(v, np.ndarray) else v.cpu().numpy()) for k, v in out.items()}


def _same(got, ref, keys=KEYS):
    for k in keys:
        assert np.array_equal(got[k], ref[k], equal_nan=True), k


@pytest.mark.parametrize("limits", [False, True])
def test_array_entries_same_bits(sctx, cfg, limits):
    """cfs_solve_batch against its asynchronous form (pageable and pinned buffers), the device form, the margins entry with NULL
    offsets (host and device) and the checked solve with rounds = 0 (host and device)"""
    import torch
    s = _set(sctx, cfg, limits=limits)
    try:
        B, n, K, eps = 96, s["H"] * 5, s["MAX_O_ITER"], s["epsilon_O"]
        a = tuple(cfg[k] for k in ("x0", "ff", "caug", "xref"))
        ref = sctx.solve_batch(*a, eps, K)
        launches = sctx.stats()["launches"]
        got = {}
        for kind in ("pageable", "pinned"):
            inp = a if kind == "pageable" else tuple(torch.from_numpy(v).pin_memory() for v in a)
            o = _outs(B, n, K, kind)
            sctx.solve_batch_ptr(B, *(_ptr(v) for v in inp), eps, K, *(_ptr(o[k]) for k in KEYS), device=False, sync=False)
            sctx.wait()
            got[kind + " async"] = (_numpy(o), sctx.stats()["launches"])
        d_in = tuple(torch.from_numpy(v).cuda() for v in a)
        o = _outs(B, n, K, "device")
        sctx.solve_batch_ptr(B, *(_ptr(v) for v in d_in), eps, K, *(_ptr(o[k]) for k in KEYS), device=True)
        got["device"] = (_numpy(o), sctx.stats()["launches"])
        got["margins"] = (sctx.solve_batch_margins(*a, None, eps, K), sctx.stats()["launches"])
        o = _outs(B, n, K, "device")
        sctx.solve_batch_margins_ptr(B, *(_ptr(v) for v in d_in), 0, eps, K, *(_ptr(o[k]) for k in KEYS))
        got["margins device"] = (_numpy(o), sctx.stats()["launches"])
        got["checked"] = (sctx.solve_checked(*a, eps, K, **CHECKED), sctx.stats()["launches"])
        o = _outs(B, n, K, "device")
        ck = {k: torch.zeros(B, dtype=dt, device="cuda") for k, dt in
              (("verdict", torch.int32), ("t_hit", torch.float64), ("cmin", torch.float64), ("rounds_used", torch.int32))}
        sctx.solve_checked_ptr(B, *(_ptr(v) for v in d_in), eps, K, *(_ptr(o[k]) for k in KEYS), *(_ptr(v) for v in ck.values()),
                               **CHECKED)
        got["checked device"] = (_numpy(o), sctx.stats()["launches"])
    finally:
        sctx.set_joint_limits(None, None)
    for name, (out, n_launch) in got.items():
        _same(out, ref)
        assert n_launch == launches, name


@pytest.mark.parametrize("limits", [False, True])
def test_route_entries_same_bits(sctx, cfg, limits):
    """cfs_solve_routes against cfs_solve_routes_var with every length W (synchronous, and asynchronous on pinned buffers) and
    cfs_solve_routes_device with and without route_len; cfs_solve_start_goal against its asynchronous form"""
    import torch
    s = _set(sctx, cfg, blocks=True, limits=limits)
    try:
        routes = cfg["routes"]
        B, W, n, K, eps = routes.shape[0], routes.shape[1], s["H"] * 5, s["MAX_O_ITER"], s["epsilon_O"]
        rl = np.full(B, W, dtype=np.int32)
        ref = sctx.solve_routes(routes, eps, K)
        launches = sctx.stats()["launches"]
        got = {"var": (sctx.solve_routes_var(routes, rl, eps, K), sctx.stats()["launches"])}
        o = _outs(B, n, K, "pinned")
        p_routes, p_rl = torch.from_numpy(routes).pin_memory(), torch.from_numpy(rl).pin_memory()
        sctx.solve_routes_var_ptr(B, W, _ptr(p_rl), _ptr(p_routes), eps, K, *(_ptr(o[k]) for k in KEYS), sync=False)
        sctx.wait()
        got["var async pinned"] = (_numpy(o), sctx.stats()["launches"])
        d_routes, d_rl = torch.from_numpy(routes).cuda(), torch.from_numpy(rl).cuda()
        for name, lp in (("device", _ptr(d_rl)), ("device without route_len", 0)):
            o = _outs(B, n, K, "device")
            sctx.solve_routes_var_ptr(B, W, lp, _ptr(d_routes), eps, K, *(_ptr(o[k]) for k in KEYS), device=True)
            got[name] = (_numpy(o), sctx.stats()["launches"])
        sg = sctx.solve_start_goal(cfg["theta0"], cfg["thetag"], eps, K)
        sg_launches = sctx.stats()["launches"]
        o = _outs(B, n, K, "pageable")
        t0, tg = np.ascontiguousarray(cfg["theta0"]), np.ascontiguousarray(cfg["thetag"])
        sctx.solve_start_goal_ptr(B, _ptr(t0), _ptr(tg), eps, K, *(_ptr(o[k]) for k in KEYS), sync=False)
        sctx.wait()
        sg_async = (_numpy(o), sctx.stats()["launches"])
    finally:
        sctx.set_joint_limits(None, None)
    for name, (out, n_launch) in got.items():
        _same(out, ref)
        assert n_launch == launches, name
    _same(sg_async[0], sg)
    assert sg_async[1] == sg_launches


# ---- the same errors from every entry ------------------------------------------------------------------------------------
OUTS = ["u", "x", "cost_hist", "e_u_hist", "iters", "status"]
SCAL = ["eps", "max_outer", "alpha"]
ARRAYS = ["B", "solver", "grad", "x0", "ff", "caug", "xref", "noise"] + SCAL + OUTS
START_GOAL = ["B", "solver", "grad", "theta0", "thetag", "noise"] + SCAL + OUTS
ROUTES = ["B", "W", "solver", "grad", "routes", "noise"] + SCAL + OUTS
ROUTES_VAR = ["B", "W", "route_len", "solver", "grad", "routes", "noise"] + SCAL + OUTS
MARGINS = ["B", "solver", "grad", "x0", "ff", "caug", "xref", "noise", "margin_off"] + SCAL + OUTS
CHECKED_ARGS = (["B", "solver", "grad", "x0", "ff", "caug", "xref", "noise"] + SCAL + ["eta", "max_evals", "rounds", "gain"] + OUTS +
                ["verdict", "t_hit", "cmin", "rounds_used", "margin_off"])
NEED_ARRAYS = ["x0", "ff", "caug", "xref", "u", "cost_hist", "iters", "status"]
NEED_SG = ["theta0", "thetag", "u", "cost_hist", "iters", "status"]
NEED_ROUTES = ["routes", "u", "cost_hist", "iters", "status"]
NEED_CHECKED = NEED_ARRAYS + ["x", "verdict", "t_hit", "cmin", "rounds_used"]
# entry: (argument list, device pointers, needs cfs_set_cost_blocks, the buffers a call must not pass as NULL), as the library
# has always had them
ENTRIES = {
    "cfs_solve_batch": (ARRAYS, False, False, NEED_ARRAYS),
    "cfs_solve_batch_async": (ARRAYS, False, False, NEED_ARRAYS),
    "cfs_solve_batch_device": (ARRAYS + ["sync"], True, False, NEED_ARRAYS + ["x"]),
    "cfs_solve_start_goal": (START_GOAL, False, True, NEED_SG),
    "cfs_solve_start_goal_async": (START_GOAL, False, True, NEED_SG),
    "cfs_solve_routes": (ROUTES, False, True, NEED_ROUTES),
    "cfs_solve_routes_async": (ROUTES, False, True, NEED_ROUTES),
    "cfs_solve_routes_var": (ROUTES_VAR, False, True, NEED_ROUTES + ["route_len"]),
    "cfs_solve_routes_var_async": (ROUTES_VAR, False, True, NEED_ROUTES + ["route_len"]),
    "cfs_solve_routes_device": (ROUTES_VAR + ["sync"], True, True, NEED_ROUTES + ["x"]),
    "cfs_solve_batch_margins": (MARGINS, False, False, NEED_ARRAYS),
    "cfs_solve_batch_margins_device": (MARGINS + ["sync"], True, False, NEED_ARRAYS + ["x"]),
    "cfs_solve_checked": (CHECKED_ARGS, False, False, NEED_CHECKED),
    "cfs_solve_checked_device": (CHECKED_ARGS + ["sync"], True, False, NEED_CHECKED),
}
INTS = {"B", "W", "solver", "grad", "max_outer", "max_evals", "rounds", "sync"}
DOUBLES = {"eps", "alpha", "eta", "gain"}


def _buffers(cfg, B, device):
    """valid buffers of a B-problem call of every solve entry (host numpy arrays, or device torch tensors)"""
    import torch
    s = cfg["sys_info"]
    n, K, O = s["H"] * 5, s["MAX_O_ITER"], len(cfg["obs"])
    f = lambda *sh: np.zeros(sh)
    i = lambda *sh: np.zeros(sh, dtype=np.int32)
    b = dict(x0=cfg["x0"][:B].copy(), ff=cfg["ff"][:B].copy(), caug=cfg["caug"][:B].copy(), xref=cfg["xref"][:B].copy(),
             theta0=cfg["theta0"][:B].copy(), thetag=cfg["thetag"][:B].copy(), routes=cfg["routes"][:B].copy(),
             route_len=np.full(B, cfg["routes"].shape[1], dtype=np.int32), noise=None, margin_off=f(B, O, s["H"]),
             u=f(B, n), x=f(B, 2 * n), cost_hist=f(B, K), e_u_hist=f(B, K), iters=i(B), status=i(B), verdict=i(B), t_hit=f(B),
             cmin=f(B), rounds_used=i(B))
    if device:
        b = {k: None if v is None else torch.from_numpy(v).cuda() for k, v in b.items()}
    return b


def _call(lib, h, name, bufs, **over):
    """entry `name` on context handle h with valid arguments, `over` replacing some (a buffer name mapped to None: NULL)"""
    s = dict(B=4, W=6, solver=0, grad=0, eps=0.1, max_outer=20, alpha=0.0, eta=1e-3, max_evals=4096, rounds=2, gain=2.0, sync=1)
    s.update(over)
    args = []
    for p in ENTRIES[name][0]:
        v = s[p] if p in s else bufs[p]
        args.append(C.c_int(v) if p in INTS else C.c_double(v) if p in DOUBLES else C.c_void_p(None if v is None else _ptr(v)))
    return getattr(lib, name)(h, *args)


def _invalid_calls(name):
    """(what, overrides, code): the invalid calls of entry `name` and the code each returns"""
    params, _, _, need = ENTRIES[name]
    calls = [("B < 0", dict(B=-1), E_ARG), ("max_outer < 0", dict(max_outer=-1), E_ARG), ("solver 7", dict(solver=7), E_ARG),
             ("grad 7", dict(grad=7), E_ARG)]
    if "W" in params:
        calls.append(("W = 1", dict(W=1), E_ARG))
    return calls + [("NULL " + k, {k: None}, E_ARG) for k in need]


@pytest.mark.parametrize("name", list(ENTRIES))
def test_same_errors(sctx, cfg, name):
    """NULL ctx; no robot, obstacles, cost or cost blocks (CFS_E_STATE); bad scalars, W = 1 and every required buffer NULL
    (CFS_E_ARG): the codes every entry has always returned.  B = 0 returns 0 and enqueues nothing."""
    lib = _lib.load()
    params, device, blocks, _ = ENTRIES[name]
    bufs = _buffers(cfg, 4, device)
    assert _call(lib, None, name, bufs) == E_ARG
    c2 = M.Context(0)
    try:
        assert _call(lib, c2._h, name, bufs) == E_STATE, "no robot"
        c2.set_robot(dict(cfg["robot"], name="M16iB"), 5)
        assert _call(lib, c2._h, name, bufs) == E_STATE, "no obstacles"
        c2.set_obstacles(cfg["obs"])
        assert _call(lib, c2._h, name, bufs) == E_STATE, "no cost"
        if blocks:
            s = cfg["sys_info"]
            c2.set_cost(s["H"], s["QQ"], s["lim"], s["MAX_input"])
            assert _call(lib, c2._h, name, bufs) == E_STATE, "no cost blocks"
    finally:
        c2.close()
    _set(sctx, cfg, blocks=True)
    for what, over, code in _invalid_calls(name):
        assert _call(lib, sctx._h, name, bufs, **over) == code, what
    sctx.solve_batch(*(cfg[k][:4] for k in ("x0", "ff", "caug", "xref")), 0.1, 20)
    before = sctx.stats()
    assert _call(lib, sctx._h, name, bufs, B=0) == 0
    assert sctx.stats() == before


def test_copy_times_belong_to_host_forms(sctx, cfg):
    """cfs_get_stats: ms_h2d and ms_d2h time a host form's own copies, and are 0 after a device form"""
    import torch
    s = _set(sctx, cfg)
    B, n, K, eps = 96, s["H"] * 5, s["MAX_O_ITER"], s["epsilon_O"]
    a = tuple(cfg[k] for k in ("x0", "ff", "caug", "xref"))
    d_in = tuple(torch.from_numpy(v).cuda() for v in a)
    o = _outs(B, n, K, "device")
    ck = [torch.zeros(B, dtype=dt, device="cuda") for dt in (torch.int32, torch.float64, torch.float64, torch.int32)]
    copies = lambda: (sctx.stats()["ms_h2d"], sctx.stats()["ms_d2h"])
    steps = [("solve_batch", True, lambda: sctx.solve_batch(*a, eps, K)),
             ("solve_batch_device", False,
              lambda: sctx.solve_batch_ptr(B, *(_ptr(v) for v in d_in), eps, K, *(_ptr(o[k]) for k in KEYS), device=True)),
             ("solve_batch_margins", True, lambda: sctx.solve_batch_margins(*a, None, eps, K)),
             ("solve_batch_margins_device", False,
              lambda: sctx.solve_batch_margins_ptr(B, *(_ptr(v) for v in d_in), 0, eps, K, *(_ptr(o[k]) for k in KEYS))),
             ("solve_checked", True, lambda: sctx.solve_checked(*a, eps, K, **CHECKED)),
             ("solve_checked_device", False,
              lambda: sctx.solve_checked_ptr(B, *(_ptr(v) for v in d_in), eps, K, *(_ptr(o[k]) for k in KEYS),
                                             *(_ptr(v) for v in ck), **CHECKED))]
    for name, host, run in steps:
        run()
        h2d, d2h = copies()
        assert (h2d > 0 and d2h > 0) if host else (h2d == 0 and d2h == 0), (name, h2d, d2h)
