"""GPU tests of the host-pointer entries of the C ABI beyond the solve family (cfs_resample_routes, cfs_chomp_batch,
cfs_dist_grad, cfs_time_dist_grad, cfs_get_con, cfs_nodes_feasible, cfs_check_edges, cfs_check_trajectories,
cfs_nearest_steer, cfs_rrt_find_routes): a host form returns the bits of its device form, pageable and pinned caller buffers
give the same bits, every entry rejects the same invalid calls with the same codes, and a synchronous entry completes the
batch in flight before it runs."""
import ctypes as C

import numpy as np
import pytest

import motionplanning_5d_m_b200 as M
from motionplanning_5d_m_b200 import _lib, rrt
from tests import common

pytestmark = pytest.mark.gpu
E_ARG, E_STATE = -1, -3
N, HS, MAX_ITER, NRND, K = 64, 40, 150, 1024, 10
OBS2 = {"l": np.array(common.OBS_M16_SCRIPT_ALT), "D": 0.2, "epsilon": 0.2}
SC = rrt.SCENE_RRTSTAR

# entry: (parameters in the order of the C signature, the state it needs ("robot", "obstacles" or "cost"), its invalid scalar
# calls, the buffers a call must not pass as NULL, its count parameter (None: it has none), its outputs), as the library has
# always had them
CHECK = ["eta", "margin_is_D", "max_evals"]
BAD_CHECK = [("eta = 0", dict(eta=0.0)), ("eta = inf", dict(eta=np.inf)), ("margin - eta < 1e-4", dict(eta=0.2)),
             ("max_evals = 0", dict(max_evals=0))]
RRT = ["S", "star", "rx0", "rgoal", "rgoal_th"]
RRT_OUT = ["routes_out", "route_len", "nn", "fail", "rnd_used"]
RRT_BAD = [("S < 0", dict(S=-1)), ("max_iter = 0", dict(max_iter=0)), ("nrnd = 0", dict(nrnd=0))]
ENTRIES = {
    "cfs_resample_routes": (["B", "W", "Hs", "routes", "sampled"], "obstacles",
                            [("B < 0", dict(B=-1)), ("W = 1", dict(W=1)), ("H = 0", dict(Hs=0))], ["routes", "sampled"], "B", ["sampled"]),
    "cfs_chomp_batch": (["B", "x0", "ff", "caug", "xref", "u_init", "alpha", "max_outer", "u", "x", "cost_hist", "e_u_hist", "iters",
                         "status"], "cost", [("B < 0", dict(B=-1)), ("max_outer < 0", dict(max_outer=-1))],
                        ["x0", "ff", "caug", "xref", "u_init", "u", "cost_hist", "iters", "status"], "B",
                        ["u", "x", "cost_hist", "e_u_hist", "iters", "status"]),
    "cfs_dist_grad": (["N", "grad", "theta", "dist", "linkid", "g", "flags"], "obstacles", [("N < 0", dict(N=-1))],
                      ["theta", "dist", "g"], "N", ["dist", "linkid", "g", "flags"]),
    "cfs_time_dist_grad": (["N", "grad", "theta", "reps", "ms"], "obstacles", [("N = 0", dict(N=0)), ("reps = 0", dict(reps=0))],
                           ["theta", "ms"], None, []),
    "cfs_get_con": (["grad", "margin_is_D", "x0_1", "xcur", "u1", "Ainq", "binq"], "cost", [], ["x0_1", "xcur", "u1", "Ainq", "binq"],
                    None, ["Ainq", "binq"]),
    "cfs_nodes_feasible": (["N", "theta", "feasible", "dmin"], "obstacles", [("N < 0", dict(N=-1))], ["theta", "feasible"], "N",
                           ["feasible", "dmin"]),
    "cfs_check_edges": (["N", "theta_a", "theta_b"] + CHECK + ["verdict", "s_hit", "cmin", "evals"], "obstacles",
                        [("N < 0", dict(N=-1))] + BAD_CHECK, ["theta_a", "theta_b", "verdict", "s_hit", "cmin"], "N",
                        ["verdict", "s_hit", "cmin", "evals"]),
    "cfs_check_trajectories": (["B", "H", "x0", "xs", "us"] + CHECK + ["verdict", "t_hit", "cmin", "evals"], "obstacles",
                               [("B < 0", dict(B=-1)), ("H = 0", dict(H=0))] + BAD_CHECK,
                               ["x0", "xs", "us", "verdict", "t_hit", "cmin"], "B", ["verdict", "t_hit", "cmin", "evals"]),
    "cfs_nearest_steer": (["n_nodes", "nodes", "S", "samples", "ratial", "step", "parent", "newnode"], "robot",
                          [("n_nodes = 0", dict(n_nodes=0)), ("S < 0", dict(S=-1))], ["nodes", "samples", "ratial", "parent", "newnode"],
                          "S", ["parent", "newnode"]),
    "cfs_rrt_find_routes": (RRT + ["region_g", "region_s", "sample_off", "ratial", "bi", "max_iter", "rnd", "nrnd"] + RRT_OUT +
                            ["tree_nodes", "tree_parent", "tree_total", "ms_kernel"], "obstacles", RRT_BAD,
                            ["rx0", "rgoal", "rgoal_th", "region_g", "region_s", "sample_off", "ratial", "rnd"] + RRT_OUT, "S",
                            RRT_OUT + ["tree_nodes", "tree_parent", "tree_total"]),
    "cfs_check_edges_device": (["N", "theta_a", "theta_b"] + CHECK + ["verdict", "s_hit", "cmin", "evals", "sync"],
                               "obstacles", [("N < 0", dict(N=-1))] + BAD_CHECK, ["theta_a", "theta_b", "verdict", "s_hit", "cmin"],
                               "N", ["verdict", "s_hit", "cmin", "evals"]),
    "cfs_check_trajectories_device": (["B", "H", "x0", "xs", "us"] + CHECK + ["verdict", "t_hit", "cmin", "evals", "sync"], "obstacles",
                                      [("B < 0", dict(B=-1)), ("H = 0", dict(H=0))] + BAD_CHECK,
                                      ["x0", "xs", "us", "verdict", "t_hit", "cmin"], "B", ["verdict", "t_hit", "cmin", "evals"]),
    "cfs_rrt_find_routes_device": (RRT + ["params", "bi", "max_iter", "rnd", "nrnd"] + RRT_OUT + ["route_len_or_fail", "sync"],
                                   "obstacles", RRT_BAD, ["rx0", "rgoal", "rgoal_th", "params", "rnd"] + RRT_OUT, "S",
                                   RRT_OUT + ["route_len_or_fail"]),
}
HOST = [k for k in ENTRIES if not k.endswith("_device")]
INTS = {"B", "N", "S", "W", "H", "Hs", "grad", "max_outer", "reps", "margin_is_D", "max_evals", "n_nodes", "star", "max_iter", "nrnd",
        "sync"}
DOUBLES = {"alpha", "eta", "step", "bi"}
STATES = ["robot", "obstacles", "cost"]


@pytest.fixture(scope="module")
def hctx():
    c = M.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def cfg(oracle):
    """a seeded M16iB batch with two obstacles, routes through its start and goal points, and its solved trajectories"""
    c = common.batch_m16ib(oracle, N)
    c["obs"] = c["obs"] + [OBS2]
    t = np.linspace(0.0, 1.0, 6)[None, :, None]
    bend = np.random.default_rng(17).normal(0.0, 0.05, (N, 1, 5)) * np.sin(np.pi * t)
    c["routes"] = np.ascontiguousarray(c["theta0"][:, None] + t * (c["thetag"] - c["theta0"])[:, None] + bend)
    ctx = M.Context(0)
    try:
        _set(ctx, c)
        c["solved"] = ctx.solve_batch(c["x0"], c["ff"], c["caug"], c["xref"], c["sys_info"]["epsilon_O"], K)
    finally:
        ctx.close()
    return c


def _set(c, cfg, upto="cost"):
    s = cfg["sys_info"]
    c.set_robot(dict(cfg["robot"], name="M16iB"), 5)
    if upto != "robot":
        c.set_obstacles(cfg["obs"])
    if upto == "cost":
        c.set_cost(s["H"], s["QQ"], s["lim"], s["MAX_input"])
    return s


def _buffers(cfg, kind):
    """valid buffers of every entry: numpy ("pageable"), pinned torch ("pinned") or device torch ("device") arrays; outputs zero"""
    import torch
    s = cfg["sys_info"]
    H, n, O, cap = s["H"], s["H"] * 5, len(cfg["obs"]), MAX_ITER + 2
    f = lambda *sh: np.zeros(sh)
    i = lambda *sh: np.zeros(sh, dtype=np.int32)
    rnd = np.random.default_rng(7).random((N, NRND))
    b = dict(routes=cfg["routes"], sampled=f(N, HS + 1, 5), x0=cfg["x0"], ff=cfg["ff"], caug=cfg["caug"], xref=cfg["xref"],
             u_init=np.random.default_rng(3).normal(0.0, 1e-3, (N, n)), u=f(N, n), x=f(N, 2 * n), cost_hist=f(N, K), e_u_hist=f(N, K),
             iters=i(N), status=i(N), theta=cfg["theta0"], dist=f(N, O), linkid=i(N, O), g=f(N, O, 5), flags=i(N), ms=f(1),
             x0_1=cfg["x0"][0].copy(), xcur=cfg["solved"]["x"][0].copy(), u1=cfg["solved"]["u"][0].copy(),
             Ainq=f(n, O * H * 11), binq=f(O * H * 11), feasible=np.zeros(N, dtype=np.uint8), dmin=f(N), theta_a=cfg["theta0"],
             theta_b=cfg["thetag"], verdict=i(N), s_hit=f(N), cmin=f(N), evals=i(N), xs=cfg["solved"]["x"], us=cfg["solved"]["u"],
             t_hit=f(N), nodes=np.ascontiguousarray(cfg["thetag"][:50]), samples=cfg["theta0"], ratial=SC["ratial"].copy(),
             parent=i(N), newnode=f(N, 5), rx0=cfg["theta0"], rgoal=cfg["thetag"], rgoal_th=cfg["thetag"], region_g=SC["region_g"].copy(),
             region_s=SC["region_s"].copy(), sample_off=SC["sample_off"].copy(), rnd=rnd, routes_out=f(N, cap, 5), route_len=i(N),
             nn=i(N), fail=i(N), rnd_used=i(N), tree_nodes=f(N, cap, 5), tree_parent=i(N, cap), tree_total=f(N, cap), ms_kernel=f(1),
             params=np.concatenate([SC["region_g"], SC["region_s"], SC["sample_off"], SC["ratial"]]), route_len_or_fail=i(N))
    b = {k: np.ascontiguousarray(v) for k, v in b.items()}
    if kind == "pinned":
        b = {k: torch.from_numpy(v).pin_memory() for k, v in b.items()}
    elif kind == "device":
        b = {k: torch.from_numpy(v).cuda() for k, v in b.items()}
    return b


def _ptr(v):
    return v.ctypes.data if isinstance(v, np.ndarray) else v.data_ptr()


def _numpy(v):
    return v if isinstance(v, np.ndarray) else v.cpu().numpy()


def _call(lib, h, name, bufs, cfg, **over):
    """entry `name` on context handle h with valid arguments, `over` replacing some (a buffer name mapped to None: NULL)"""
    s = dict(B=N, N=N, S=N, W=6, H=cfg["sys_info"]["H"], Hs=HS, grad=0, alpha=1e-3, max_outer=K, reps=3, margin_is_D=1, max_evals=4096,
             eta=1e-3, n_nodes=50, step=0.1, star=0, bi=0.5, max_iter=MAX_ITER, nrnd=NRND, sync=1)
    s.update(over)
    args = []
    for p in ENTRIES[name][0]:
        v = s[p] if p in s else bufs[p]
        args.append(C.c_int(v) if p in INTS else C.c_double(v) if p in DOUBLES else C.c_void_p(None if v is None else _ptr(v)))
    return getattr(lib, name)(h, *args)


def _run(ctx, name, cfg, kind):
    """the outputs of one valid call of `name` on fresh buffers of `kind`"""
    import torch
    b = _buffers(cfg, kind)
    assert _call(_lib.load(), ctx._h, name, b, cfg) == 0, name
    torch.cuda.synchronize()
    return {k: _numpy(b[k]) for k in ENTRIES[name][5]}


def _same(got, ref):
    assert got.keys() == ref.keys()
    for k in ref:
        assert np.array_equal(got[k], ref[k], equal_nan=True), k


@pytest.mark.parametrize("name", ["cfs_check_edges", "cfs_check_trajectories", "cfs_rrt_find_routes"])
def test_host_form_is_device_form(hctx, cfg, name):
    """the host form returns the bits of its device form (pageable caller buffers against device buffers)"""
    _set(hctx, cfg)
    host = _run(hctx, name, cfg, "pageable")
    dev = _run(hctx, name + "_device", cfg, "device")
    keys = RRT_OUT if name == "cfs_rrt_find_routes" else ENTRIES[name][5]
    _same({k: dev[k] for k in keys}, {k: host[k] for k in keys})
    if name == "cfs_rrt_find_routes":
        assert host["rnd_used"].min() > 0


@pytest.mark.parametrize("name", HOST)
def test_pageable_is_pinned(hctx, cfg, name):
    """numpy (pageable) and pinned torch caller buffers give the same bits"""
    _set(hctx, cfg)
    _same(_run(hctx, name, cfg, "pinned"), _run(hctx, name, cfg, "pageable"))


@pytest.mark.parametrize("name", list(ENTRIES))
def test_same_errors(hctx, cfg, name):
    """NULL ctx; each missing piece of state the entry needs (CFS_E_STATE) and 0 once it is there; invalid scalars and every
    required buffer NULL (CFS_E_ARG); a count of 0 returns 0 and changes no statistic"""
    lib = _lib.load()
    params, need, bad, required, count, _ = ENTRIES[name]
    bufs = _buffers(cfg, "device" if name.endswith("_device") else "pageable")
    assert _call(lib, None, name, bufs, cfg) == E_ARG
    c2 = M.Context(0)
    try:
        for k, st in enumerate(STATES):
            code = _call(lib, c2._h, name, bufs, cfg)
            assert code == (E_STATE if k <= STATES.index(need) else 0), (st, code)
            _set(c2, cfg, upto=st)
        assert _call(lib, c2._h, name, bufs, cfg) == 0
    finally:
        c2.close()
    _set(hctx, cfg)
    for what, over in bad:
        assert _call(lib, hctx._h, name, bufs, cfg, **over) == E_ARG, what
    for k in required:
        assert _call(lib, hctx._h, name, bufs, cfg, **{k: None}) == E_ARG, "NULL " + k
    if count is not None:
        hctx.solve_batch(*(cfg[k][:4] for k in ("x0", "ff", "caug", "xref")), 0.1, 20)
        before = hctx.stats()
        assert _call(lib, hctx._h, name, bufs, cfg, **{count: 0}) == 0
        assert hctx.stats() == before


def test_batch_in_flight_is_completed_first(hctx, cfg):
    """cfs_solve_batch_async on pageable buffers, then a synchronous entry: the entry returns its stand-alone result, the
    batch's outputs are in the caller's buffers and cfs_get_stats describes the batch (cfs_chomp_batch: its own) before
    cfs_wait, and the cfs_wait that follows changes nothing"""
    s = _set(hctx, cfg)
    a = tuple(cfg[k] for k in ("x0", "ff", "caug", "xref"))
    eps, n = s["epsilon_O"], s["H"] * 5
    ref = hctx.solve_batch(*a, eps, K)
    ref_stats = hctx.stats()
    keys = ("u", "x", "cost_hist", "e_u_hist", "iters", "status")
    for name in HOST:
        alone = _run(hctx, name, cfg, "pageable")
        alone_stats = hctx.stats()
        o = dict(u=np.zeros((N, n)), x=np.zeros((N, 2 * n)), cost_hist=np.zeros((N, K)), e_u_hist=np.zeros((N, K)),
                 iters=np.zeros(N, dtype=np.int32), status=np.zeros(N, dtype=np.int32))
        hctx.solve_batch_ptr(N, *(_ptr(v) for v in a), eps, K, *(_ptr(o[k]) for k in keys), sync=False)
        got = _run(hctx, name, cfg, "pageable")
        _same(got, alone)
        for k in keys:
            assert np.array_equal(o[k], ref[k], equal_nan=True), (name, k)
        st = hctx.stats()
        want = alone_stats if name == "cfs_chomp_batch" else ref_stats
        assert (st["launches"], st["problem_iters"]) == (want["launches"], want["problem_iters"]), name
        hctx.wait()
        assert hctx.stats() == st, name
        for k in keys:
            assert np.array_equal(o[k], ref[k], equal_nan=True), (name, k)
