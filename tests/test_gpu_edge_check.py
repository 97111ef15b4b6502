"""-m gpu : the continuous collision checks (k_check.cu through the C ABI) against their CPU restatement (tests/check_oracle.c).

Verdicts identical on every item, s_hit / t_hit and cmin within 1e-9, evaluation counts equal up to one on at most 0.1 % of the
items (a last-bit difference of c can move a step end across the path's end)."""
import ctypes as C

import numpy as np
import pytest

import motionplanning_5d_m_b200 as M
from motionplanning_5d_m_b200 import _lib, rrt, synthetic
from tests import check_oracle as K
from tests import common
from tests.test_edge_check import SCENES, box_obstacles, random_edges

pytestmark = pytest.mark.gpu
ETA = 1e-3


def _bind(ctx, robot_name, obs):
    r = dict(M.robotproperty2(robot_name))
    r["name"] = robot_name
    ctx.set_robot(r, 2 if robot_name == "2L" else 5)
    ctx.set_obstacles(obs)


def _compare(out, ref, key):
    assert np.array_equal(out["verdict"], ref["verdict"]), np.flatnonzero(out["verdict"] != ref["verdict"])[:10]
    assert np.abs(out[key] - ref[key]).max(initial=0.0) <= 1e-9
    assert np.abs(out["cmin"] - ref["cmin"]).max(initial=0.0) <= 1e-9
    de = np.abs(out["evals"].astype(np.int64) - ref["evals"])
    assert de.max(initial=0) <= 1 and (de > 0).sum() <= 1e-3 * de.size, (de.max(initial=0), (de > 0).sum())


def _scene_obs(name):
    robot, obs, off, half = SCENES[name]
    return robot, (box_obstacles() if obs is None else obs), off, half


@pytest.mark.parametrize("name,N", [("headline", 100000), ("boxes", 20000), ("2L", 20000)])
def test_random_edges_parity(ctx, name, N):
    robot, obs, off, half = _scene_obs(name)
    _bind(ctx, robot, obs)
    rng = np.random.default_rng(101)
    a, b = random_edges(rng, N, off, half, reach=0.6 if robot != "2L" else 1.5)
    out = ctx.check_edges(a, b, eta=ETA)
    ref = K.Scene(robot, obs).check_edges(a, b, eta=ETA)
    _compare(out, ref, "s_hit")
    assert (out["verdict"] == _lib.CHECK_HIT).any() and (out["verdict"] == _lib.CHECK_CLEAR).any()


def test_rrt_tree_edges_parity(ctx):
    sc = rrt.SCENE_RRTSTAR
    _bind(ctx, "M200i", sc["obs"])
    S = 1024
    rng = np.random.default_rng(5)
    tile = lambda v: np.tile(np.asarray(v, dtype=np.float64).reshape(1, -1), (S, 1))
    tr = ctx.rrt_find_routes(tile(sc["x0"]), tile(sc["goal"]), tile(sc["goal"]), sc["region_g"], sc["region_s"], sc["sample_off"],
                             sc["ratial"], rng.random((S, rrt.NRND_DEFAULT)), star=True, want_tree=True)
    ta, tb = [], []
    for s_ in range(S):
        n = int(tr["n_nodes"][s_])
        par = tr["parent"][s_, 1:n] - 1            # 1-based parents; node 0 is the root
        ta.append(tr["nodes"][s_, par])
        tb.append(tr["nodes"][s_, 1:n])
    ta, tb = np.concatenate(ta), np.concatenate(tb)
    assert ta.shape[0] > 10000
    out = ctx.check_edges(ta, tb, eta=ETA)
    ref = K.Scene("M200i", sc["obs"]).check_edges(ta, tb, eta=ETA)
    _compare(out, ref, "s_hit")
    # the tree's nodes are feasible (d >= D); its edges need not be
    assert (out["verdict"] != _lib.CHECK_UNDECIDED).all()


@pytest.fixture(scope="module")
def headline(ctx, oracle):
    cfg = common.batch_m16ib(oracle, 4096)
    s = cfg["sys_info"]
    _bind(ctx, "M16iB", cfg["obs"])
    ctx.set_cost(s["H"], s["QQ"], s["lim"], s["MAX_input"])
    sol = ctx.solve_batch(cfg["x0"], cfg["ff"], cfg["caug"], cfg["xref"], s["epsilon_O"], s["MAX_O_ITER"])
    return cfg, sol


def test_headline_trajectories_parity(ctx, headline):
    cfg, sol = headline
    _bind(ctx, "M16iB", cfg["obs"])
    out = ctx.check_trajectories(cfg["x0"], sol["x"], sol["u"], eta=ETA)
    ref = K.Scene("M16iB", cfg["obs"]).check_trajectories(cfg["x0"], sol["x"], sol["u"], eta=ETA)
    _compare(out, ref, "t_hit")
    conv = (sol["status"] & 0xFF) == 0
    assert (out["verdict"][conv] == _lib.CHECK_HIT).any() and (out["verdict"][conv] == _lib.CHECK_CLEAR).any()
    # determinism, permutation, device form
    again = ctx.check_trajectories(cfg["x0"], sol["x"], sol["u"], eta=ETA)
    for k in out:
        assert np.array_equal(out[k], again[k])
    perm = np.random.default_rng(1).permutation(len(out["verdict"]))
    pout = ctx.check_trajectories(cfg["x0"][perm], sol["x"][perm], sol["u"][perm], eta=ETA)
    for k in out:
        assert np.array_equal(pout[k], out[k][perm])
    import torch
    dev = torch.device("cuda", ctx.device)
    t = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in (("x0", cfg["x0"]), ("x", sol["x"]), ("u", sol["u"]))}
    B, H = cfg["x0"].shape[0], cfg["sys_info"]["H"]
    v = torch.zeros(B, dtype=torch.int32, device=dev)
    th, cm = torch.zeros(B, dtype=torch.float64, device=dev), torch.zeros(B, dtype=torch.float64, device=dev)
    ev = torch.zeros(B, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    ctx.check_trajectories_ptr(B, H, t["x0"].data_ptr(), t["x"].data_ptr(), t["u"].data_ptr(), v.data_ptr(), th.data_ptr(),
                               cm.data_ptr(), ev.data_ptr(), eta=ETA, sync=True)
    dout = dict(verdict=v.cpu().numpy(), t_hit=th.cpu().numpy(), cmin=cm.cpu().numpy(), evals=ev.cpu().numpy())
    for k in out:
        assert np.array_equal(dout[k], out[k])


def test_edges_device_form_and_determinism(ctx):
    import torch
    _bind(ctx, "M16iB", [synthetic.OBS_M16IB])
    rng = np.random.default_rng(9)
    a, b = random_edges(rng, 5000, synthetic.SAMPLE_OFF, synthetic.REGION_S)
    out = ctx.check_edges(a, b)
    again = ctx.check_edges(a, b)
    perm = rng.permutation(a.shape[0])
    pout = ctx.check_edges(a[perm], b[perm])
    for k in out:
        assert np.array_equal(out[k], again[k]) and np.array_equal(pout[k], out[k][perm])
    dev = torch.device("cuda", ctx.device)
    da, db = torch.from_numpy(a).to(dev), torch.from_numpy(b).to(dev)
    N = a.shape[0]
    v, ev = torch.zeros(N, dtype=torch.int32, device=dev), torch.zeros(N, dtype=torch.int32, device=dev)
    sh, cm = torch.zeros(N, dtype=torch.float64, device=dev), torch.zeros(N, dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    ctx.check_edges_ptr(N, da.data_ptr(), db.data_ptr(), v.data_ptr(), sh.data_ptr(), cm.data_ptr(), ev.data_ptr(), sync=True)
    dout = dict(verdict=v.cpu().numpy(), s_hit=sh.cpu().numpy(), cmin=cm.cpu().numpy(), evals=ev.cpu().numpy())
    for k in out:
        assert np.array_equal(dout[k], out[k])


def test_zero_length_edges_match_node_check(ctx):
    _bind(ctx, "M16iB", [synthetic.OBS_M16IB])
    th = common.sampling_box(np.random.default_rng(4), 20000)
    feas, dmin = ctx.nodes_feasible(th)
    out = ctx.check_edges(th, th, eta=ETA)
    assert np.array_equal(out["cmin"], dmin - 0.2)                       # bit for bit
    assert np.array_equal(out["verdict"] == _lib.CHECK_HIT, dmin - 0.2 < -ETA / 2)
    assert np.array_equal(feas, out["cmin"] >= 0)
    assert (out["evals"] == 1).all()


def test_errors(ctx):
    fresh = M.Context(ctx.device)
    try:
        fresh.nj = 5
        with pytest.raises(_lib.CfsError, match=r"\(-3\)"):
            fresh.check_edges(np.zeros((1, 5)), np.zeros((1, 5)))
    finally:
        fresh.close()
    _bind(ctx, "M16iB", [synthetic.OBS_M16IB])
    z = np.zeros((1, 5))
    for eta in (0.0, -1e-3, np.nan, np.inf, 0.2 - 0.5e-4):
        with pytest.raises(_lib.CfsError, match=r"\(-1\)"):
            ctx.check_edges(z, z, eta=eta)
    with pytest.raises(_lib.CfsError, match=r"\(-1\)"):
        ctx.check_edges(z, z, max_evals=0)
    # epsilon as the margin: the same rule on obs{j}.epsilon
    _bind(ctx, "M16iB", [dict(synthetic.OBS_M16IB, epsilon=1e-3)])
    with pytest.raises(_lib.CfsError, match=r"\(-1\)"):
        ctx.check_edges(z, z, eta=1e-3, margin_is_D=False)
    ctx.check_edges(z, z, eta=1e-3, margin_is_D=True)
    e = ctx.check_edges(np.zeros((0, 5)), np.zeros((0, 5)))          # N = 0: no-op
    assert e["verdict"].size == 0
    t = ctx.check_trajectories(np.zeros((0, 10)), np.zeros((0, 100)), np.zeros((0, 50)))
    assert t["verdict"].size == 0
    rc = ctx._lib.cfs_check_edges(ctx._h, C.c_int(-1), None, None, C.c_double(1e-3), C.c_int(1), C.c_int(8), None, None, None, None)
    assert rc == -1


def test_rrtstar_cfs_check(ctx):
    robot = M.robotproperty2("M200i")
    base = rrt.rrtstar_cfs(ctx, robot, num_seed=8, rng=np.random.default_rng(21))
    plain = rrt.rrtstar_cfs(ctx, robot, num_seed=8, rng=np.random.default_rng(21), check=False)
    assert base.keys() == plain.keys()
    for k in ("winner", "cost"):
        assert base[k] == plain[k]
    assert np.array_equal(base["x"], plain["x"]) and np.array_equal(base["u"], plain["u"])
    for smooth_all in (False, True):
        a = rrt.rrtstar_cfs(ctx, robot, num_seed=8, rng=np.random.default_rng(21), smooth_all=smooth_all)
        b = rrt.rrtstar_cfs(ctx, robot, num_seed=8, rng=np.random.default_rng(21), smooth_all=smooth_all, check=True)
        for k in ("u", "x", "cost_hist", "iters", "status"):
            assert np.array_equal(a["sol"][k], b["sol"][k], equal_nan=k == "cost_hist")
        assert set(b) == set(a) | {"route_check", "traj_check", "clear"}
        assert b["route_check"].shape == (8,)
        if smooth_all:
            tv = b["traj_check"]["verdict"]
            fin = np.isfinite([b["sol"]["cost_hist"][k, max(b["sol"]["iters"][k], 1) - 1] for k in range(8)])
            if ((tv == _lib.CHECK_CLEAR) & fin & ((b["sol"]["status"] & 0xFF) < 2)).any():
                assert b["clear"] and tv[b["winner"]] == _lib.CHECK_CLEAR
        else:
            assert b["winner"] == a["winner"] and b["cost"] == a["cost"]
