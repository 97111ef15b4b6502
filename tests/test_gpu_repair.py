"""GPU tests of per-waypoint margin offsets (cfs_solve_batch_margins) and the checked solve (cfs_solve_checked)."""
import numpy as np
import pytest

from motionplanning_5d_m_b200 import _lib
from tests import check_oracle as K
from tests import common
from tests import repair_oracle as R
from tests.test_gpu_parity import BULK_DEFAULT, BULK_MODES, _compare_solve, _set
from tests.test_oracle import _golden_cases

pytestmark = pytest.mark.gpu
ETA = 1e-3
KEYS = ("u", "x", "cost_hist", "e_u_hist", "iters", "status")
LAUNCHES = {"lockstep": 44, "lockstep_warp": 64, "cta": 6, "warp_noscreen": 6, "warp_screen1": 8, "warp_screen3": 12}


def _same(a, b, keys=KEYS):
    for k in keys:
        assert np.array_equal(a[k], b[k], equal_nan=True), k


@pytest.mark.parametrize("mode", list(BULK_MODES))
def test_zero_and_constant_offsets_bitwise(ctx, oracle, mode):
    """zero offsets = cfs_solve_batch bit for bit (same launch count), a constant delta = margins m_j + delta bit for bit"""
    cfg = common.batch_m16ib(oracle, 192)
    s, obs = cfg["sys_info"], cfg["obs"]
    args = (cfg["x0"], cfg["ff"], cfg["caug"], cfg["xref"])
    d = 0.0123
    raised = [dict(o, epsilon=o["epsilon"] + d) for o in obs]
    for k, v in BULK_MODES[mode].items():
        ctx.set_option(k, v)
    try:
        _set(ctx, "M16iB", cfg["robot"], raised, s)
        ref_d = ctx.solve_batch(*args, s["epsilon_O"], s["MAX_O_ITER"])
        _set(ctx, "M16iB", cfg["robot"], obs, s)
        ref = ctx.solve_batch(*args, s["epsilon_O"], s["MAX_O_ITER"])
        z = ctx.solve_batch_margins(*args, np.zeros((192, len(obs), s["H"])), s["epsilon_O"], s["MAX_O_ITER"])
        launches = ctx.stats()["launches"]
        c = ctx.solve_batch_margins(*args, np.full((192, len(obs), s["H"]), d), s["epsilon_O"], s["MAX_O_ITER"])
    finally:
        for k, v in BULK_DEFAULT.items():
            ctx.set_option(k, v)
    _same(z, ref)
    _same(c, ref_d)
    assert launches == LAUNCHES.get(mode, 10)


@pytest.mark.parametrize("name", ["main_fanuc_psgcfs", "m16ib_script_derivest"])
def test_zero_offsets_psgcfs_derivest(ctx, oracle, name):
    ROBOT, obs, s, solver, grad, noise = _golden_cases(oracle)[name]
    _set(ctx, ROBOT, s["robot"], obs)
    ctx.set_cost(s["H"], s["QQ"], s.get("lim"), s["MAX_input"] if solver == 0 else None)
    args = (s["xR"][:, 0][None], s["ff"][None], np.array([s["caug"]]), s["x_"][None])
    ref = ctx.solve_batch(*args, s["epsilon_O"], s["MAX_O_ITER"], solver=solver, grad=grad, noise=noise)
    z = ctx.solve_batch_margins(*args, np.zeros((1, len(obs), s["H"])), s["epsilon_O"], s["MAX_O_ITER"], solver=solver, grad=grad,
                                noise=noise)
    _same(z, ref)


def test_random_offsets_vs_offset_oracle(ctx, oracle):
    cfg = common.batch_m16ib(oracle, 256)
    s, obs = cfg["sys_info"], cfg["obs"]
    _set(ctx, "M16iB", cfg["robot"], obs, s)
    rng = np.random.default_rng(11)
    off = np.where(rng.random((256, len(obs), s["H"])) < 0.1, rng.random((256, len(obs), s["H"])) * 0.01, 0.0)
    args = (cfg["x0"], cfg["ff"], cfg["caug"], cfg["xref"])
    P = common.oracle_problem(oracle, "M16iB", obs, s)
    ref = R.solve_batch_off(P, *args, off, nthreads=8)
    out = ctx.solve_batch_margins(*args, off, s["epsilon_O"], s["MAX_O_ITER"])
    _compare_solve(out, ref)


@pytest.fixture(scope="module")
def headline(ctx, oracle):
    cfg = common.batch_m16ib(oracle, 4096)
    s = cfg["sys_info"]
    _set(ctx, "M16iB", cfg["robot"], cfg["obs"], s)
    args = (cfg["x0"], cfg["ff"], cfg["caug"], cfg["xref"], s["epsilon_O"], s["MAX_O_ITER"])
    out = ctx.solve_checked(*args, eta=ETA, rounds=4, gain=2.0)
    r0 = ctx.solve_checked(*args, eta=ETA, rounds=0)
    return cfg, out, r0


def test_rounds0_is_solve_plus_check(ctx, headline):
    cfg, out, r0 = headline
    s = cfg["sys_info"]
    _set(ctx, "M16iB", cfg["robot"], cfg["obs"], s)
    sol = ctx.solve_batch(cfg["x0"], cfg["ff"], cfg["caug"], cfg["xref"], s["epsilon_O"], s["MAX_O_ITER"])
    ck = ctx.check_trajectories(cfg["x0"], sol["x"], sol["u"], eta=ETA, margin_is_D=False)
    _same(r0, sol)
    _same(r0, ck, ("verdict", "t_hit", "cmin"))
    assert (r0["rounds_used"] == 0).all() and (r0["margin_off"] == 0).all()


def test_increments_match_restatement(ctx, oracle, headline):
    """k_repair_margins, fed round 0's trajectories, against restatements fed the GPU's own per-segment results of round 0 (each
    segment checked as a one-step trajectory: its t_hit is the segment's s_hit, and for a HIT segment cmin is the clearance at the
    witness; one obstacle).  Bit for bit against gain (eta - c) with the max rule, evaluated in numpy.  The C restatement
    (tests/repair_oracle.c) fed the same verdicts and s_hit evaluates c itself with libm's sincos and the oracle's distance, whose
    last bits differ from the device's FK: within 1e-8."""
    cfg, out, r0 = headline
    s = cfg["sys_info"]
    _set(ctx, "M16iB", cfg["robot"], cfg["obs"], s)
    r1 = ctx.solve_checked(cfg["x0"], cfg["ff"], cfg["caug"], cfg["xref"], s["epsilon_O"], s["MAX_O_ITER"], eta=ETA, rounds=1)
    idx = np.nonzero((r0["verdict"] == K.HIT) & ((r0["status"] & 0xFF) < 2))[0]
    assert len(idx) > 50
    nj, H = 5, s["H"]
    X = np.concatenate([cfg["x0"][idx][:, None, :], r0["x"][idx].reshape(len(idx), H, 2 * nj)], axis=1)
    ck = ctx.check_trajectories(X[:, :-1].reshape(-1, 2 * nj), X[:, 1:].reshape(-1, 2 * nj), r0["u"][idx].reshape(-1, nj), eta=ETA,
                                margin_is_D=False)
    sv, ss, cm = (ck[k].reshape(len(idx), H) for k in ("verdict", "t_hit", "cmin"))
    inc = np.where((sv == K.HIT) & (cm < -0.5 * ETA), 2.0 * (ETA - cm), 0.0)
    exp = np.maximum(inc, np.concatenate([inc[:, 1:], np.zeros((len(idx), 1))], axis=1))[:, None, :]
    acc = r1["rounds_used"][idx] == 1  # accepted re-solves return their offsets; failed ones keep round 0's (zero)
    assert acc.sum() > 0.9 * len(idx)
    got = r1["margin_off"][idx]
    assert np.array_equal(got[acc], exp[acc])
    assert (got[~acc] == 0).all()
    rest = np.setdiff1d(np.arange(len(r0["verdict"])), idx)
    assert (r1["margin_off"][rest] == 0).all()
    sc = K.Scene("M16iB", cfg["obs"], margin_is_D=False)
    cres = np.zeros((len(idx), sc.nobs, H))
    R.repair_increments(sc, cfg["x0"][idx], r0["x"][idx], r0["u"][idx], sv, ss, ETA, 2.0, cres)
    assert np.array_equal(cres > 0, exp > 0) and np.abs(cres - exp).max() <= 1e-8, np.abs(cres - exp).max()


def test_checked_headline(ctx, oracle, headline):
    cfg, out, r0 = headline
    s = cfg["sys_info"]
    sc = K.Scene("M16iB", cfg["obs"], margin_is_D=False)
    conv0 = (r0["status"] & 0xFF) == 0
    hit0 = conv0 & (r0["verdict"] == K.HIT)
    fixed = hit0 & (out["verdict"] == K.CLEAR)
    assert hit0.sum() > 300 and fixed.sum() >= 0.8 * hit0.sum(), (hit0.sum(), fixed.sum())
    # every CLEAR answer is CLEAR under the CPU check on the returned arrays, and passes a dense sample
    clear = np.nonzero(out["verdict"] == K.CLEAR)[0]
    ck = sc.check_trajectories(cfg["x0"][clear], out["x"][clear], out["u"][clear], eta=ETA)
    assert (ck["verdict"] == K.CLEAR).all()
    dt, nj, H = s["robot"]["delta_t"], 5, s["H"]
    rep = clear[out["rounds_used"][clear] > 0]
    tau = np.linspace(0.0, dt, 64)
    for b in rep:
        pts = np.concatenate([K.segment_points(cfg["x0"][b], out["x"][b], out["u"][b], nj, dt, k, tau) for k in range(H)])
        assert sc.clearance(pts).min() >= -ETA, b
    # problems with status >= 2 after round 0 are round 0's, byte for byte
    failed = (r0["status"] & 0xFF) >= 2
    for k in KEYS + ("verdict", "t_hit", "cmin"):
        assert np.array_equal(out[k][failed], r0[k][failed], equal_nan=True), k
    # the restated loop (oracle solves, CPU checks): same rounds and verdicts except within the parity noise
    P = common.oracle_problem(oracle, "M16iB", cfg["obs"], s)
    # A problem may differ only where the oracle and its FMA twin already differ (DESIGN.md section 2) or where a checked cmin
    # or a repair witness of the oracle's loop lies within 1e-6 of the -eta/2 threshold.
    a = (cfg["x0"], cfg["ff"], cfg["caug"], cfg["xref"])
    ref = R.checked_solve(P, sc, *a, eta=ETA, rounds=4, gain=2.0)
    twn = R.checked_solve(P, sc, *a, eta=ETA, rounds=4, gain=2.0, twin=True)
    mis = (ref["rounds_used"] != out["rounds_used"]) | (ref["verdict"] != out["verdict"])
    twin_ex = (ref["rounds_used"] != twn["rounds_used"]) | (ref["verdict"] != twn["verdict"]) | (ref["status"] != twn["status"])
    near_ex = np.minimum(ref["near"], twn["near"]) < 1e-6
    bad = np.nonzero(mis & ~twin_ex & ~near_ex)[0]
    assert len(bad) == 0, (bad[:20], out["rounds_used"][bad[:20]], ref["rounds_used"][bad[:20]], mis.sum(), twin_ex.sum())
    # relative cost change of the repaired problems is small
    it0, it = r0["iters"][fixed], out["iters"][fixed]
    c0 = r0["cost_hist"][fixed, it0 - 1]
    c1 = out["cost_hist"][fixed, it - 1]
    assert np.median(np.abs(c1 / c0 - 1)) < 1e-3


def test_determinism_permutation_device_form(ctx, headline):
    import torch
    cfg, out, r0 = headline
    s = cfg["sys_info"]
    _set(ctx, "M16iB", cfg["robot"], cfg["obs"], s)
    B = 1024
    a = (cfg["x0"][:B], cfg["ff"][:B], cfg["caug"][:B], cfg["xref"][:B], s["epsilon_O"], s["MAX_O_ITER"])
    o1 = ctx.solve_checked(*a, eta=ETA)
    o2 = ctx.solve_checked(*a, eta=ETA)
    for k in o1:
        assert np.array_equal(o1[k], o2[k], equal_nan=True), k
    perm = np.random.default_rng(3).permutation(B)
    op = ctx.solve_checked(*(v[perm] for v in a[:4]), *a[4:], eta=ETA)
    for k in o1:
        assert np.array_equal(op[k], o1[k][perm], equal_nan=True), k
    dev = torch.device("cuda", ctx.device)
    T = lambda v: torch.from_numpy(np.ascontiguousarray(v)).to(dev)
    n, K_ = s["H"] * 5, s["MAX_O_ITER"]
    t_in = [T(v) for v in a[:4]]
    d = dict(u=torch.zeros(B, n, dtype=torch.float64, device=dev), x=torch.zeros(B, 2 * n, dtype=torch.float64, device=dev),
             cost_hist=torch.zeros(B, K_, dtype=torch.float64, device=dev), e_u_hist=torch.zeros(B, K_, dtype=torch.float64, device=dev),
             iters=torch.zeros(B, dtype=torch.int32, device=dev), status=torch.zeros(B, dtype=torch.int32, device=dev),
             verdict=torch.zeros(B, dtype=torch.int32, device=dev), t_hit=torch.zeros(B, dtype=torch.float64, device=dev),
             cmin=torch.zeros(B, dtype=torch.float64, device=dev), rounds_used=torch.zeros(B, dtype=torch.int32, device=dev),
             margin_off=torch.zeros(B, 1, s["H"], dtype=torch.float64, device=dev))
    torch.cuda.synchronize()
    p = {k: v.data_ptr() for k, v in d.items()}
    ctx.solve_checked_ptr(B, *(t.data_ptr() for t in t_in), s["epsilon_O"], K_, p["u"], p["x"], p["cost_hist"], p["e_u_hist"],
                          p["iters"], p["status"], p["verdict"], p["t_hit"], p["cmin"], p["rounds_used"], p["margin_off"], eta=ETA)
    for k in o1:
        assert np.array_equal(d[k].cpu().numpy(), o1[k], equal_nan=True), k
    # the margins entry's device form with the returned offsets reproduces the host form
    m = dict(u=torch.zeros_like(d["u"]), x=torch.zeros_like(d["x"]), ch=torch.zeros_like(d["cost_hist"]),
             eu=torch.zeros_like(d["e_u_hist"]), it=torch.zeros_like(d["iters"]), st=torch.zeros_like(d["status"]))
    ctx.solve_batch_margins_ptr(B, *(t.data_ptr() for t in t_in), d["margin_off"].data_ptr(), s["epsilon_O"], K_, m["u"].data_ptr(),
                                m["x"].data_ptr(), m["ch"].data_ptr(), m["eu"].data_ptr(), m["it"].data_ptr(), m["st"].data_ptr())
    h = ctx.solve_batch_margins(*a[:4], o1["margin_off"], s["epsilon_O"], K_)
    assert np.array_equal(m["u"].cpu().numpy(), h["u"]) and np.array_equal(m["st"].cpu().numpy(), h["status"])
    # the returned offsets reproduce the returned solution, for every problem (zero offsets where rounds_used is 0)
    assert (o1["rounds_used"] > 0).any()
    for k in ("u", "x", "iters", "status"):
        assert np.array_equal(h[k], o1[k]), k


def test_errors(ctx, oracle):
    cfg = common.batch_m16ib(oracle, 8)
    s, obs = cfg["sys_info"], cfg["obs"]
    _set(ctx, "M16iB", cfg["robot"], obs, s)
    a = (cfg["x0"], cfg["ff"], cfg["caug"], cfg["xref"], s["epsilon_O"], s["MAX_O_ITER"])
    for kw in (dict(eta=0.0), dict(eta=-1e-3), dict(eta=obs[0]["epsilon"]), dict(rounds=-1), dict(gain=0.0), dict(gain=np.nan),
               dict(max_evals=0)):
        with pytest.raises(_lib.CfsError):
            ctx.solve_checked(*a, **kw)
    for bad in (-1e-3, np.nan, np.inf):
        off = np.zeros((8, len(obs), s["H"]))
        off[3, 0, 7] = bad
        with pytest.raises(_lib.CfsError):
            ctx.solve_batch_margins(*a[:4], off, *a[4:])
    # the device form checks the offsets on the device
    import torch
    dev = torch.device("cuda", ctx.device)
    T = lambda v: torch.from_numpy(np.ascontiguousarray(v)).to(dev)
    n, K_, H = s["H"] * 5, s["MAX_O_ITER"], s["H"]
    t_in = [T(v) for v in a[:4]]
    outs = [torch.zeros(8, n, dtype=torch.float64, device=dev), torch.zeros(8, 2 * n, dtype=torch.float64, device=dev),
            torch.zeros(8, K_, dtype=torch.float64, device=dev), torch.zeros(8, K_, dtype=torch.float64, device=dev),
            torch.zeros(8, dtype=torch.int32, device=dev), torch.zeros(8, dtype=torch.int32, device=dev)]
    for bad in (-1e-3, np.nan, np.inf):
        off = np.zeros((8, len(obs), H))
        off[5, 0, 11] = bad
        d_off = T(off)
        with pytest.raises(_lib.CfsError, match="negative or non-finite"):
            ctx.solve_batch_margins_ptr(8, *(t.data_ptr() for t in t_in), d_off.data_ptr(), s["epsilon_O"], K_,
                                        *(o.data_ptr() for o in outs))
    # no robot / no obstacles: rejected by the library (raw entry, no Python-side guard)
    c2 = _lib.Context(ctx.device)
    try:
        vd, th, cm, ru = (torch.zeros(8, dtype=dt_, device=dev) for dt_ in (torch.int32, torch.float64, torch.float64, torch.int32))
        ptrs = [t.data_ptr() for t in t_in] + [s["epsilon_O"], K_] + [o.data_ptr() for o in outs] + [v.data_ptr() for v in (vd, th, cm, ru)]
        with pytest.raises(_lib.CfsError, match="robot not set"):
            c2.solve_checked_ptr(8, *ptrs, eta=ETA)
        c2.set_robot(dict(cfg["robot"], name="M16iB"), 5)
        c2.set_cost(s["H"], s["QQ"], s["lim"], s["MAX_input"])
        with pytest.raises(_lib.CfsError, match="obstacles not set"):
            c2.solve_checked_ptr(8, *ptrs, eta=ETA)
        with pytest.raises(_lib.CfsError, match="obstacles not set"):
            c2.solve_checked(*a)
    finally:
        c2.close()


def test_optimizer_check_keyword(ctx, oracle):
    """BatchCFS.optimizer(check=...) and CFS_FANUC(...).optimizer(check=...) run the checked solve; check=None is unchanged"""
    import motionplanning_5d_m_b200 as M
    cfg = common.batch_m16ib(oracle, 128)
    s = cfg["sys_info"]
    bc = M.BatchCFS(cfg["obs"], s, "M16iB", ctx=ctx)
    a = (cfg["x0"], cfg["ff"], cfg["caug"], cfg["xref"])
    plain = bc.optimizer(*a)
    chk = bc.optimizer(*a, check=dict(eta=ETA, rounds=2))
    ref = ctx.solve_checked(*a, s["epsilon_O"], s["MAX_O_ITER"], eta=ETA, rounds=2)
    for k in ref:
        assert np.array_equal(chk[k], ref[k], equal_nan=True), k
    _same(plain, ctx.solve_batch(*a, s["epsilon_O"], s["MAX_O_ITER"]))
    ROBOT, robot, obs, s1 = common.main_fanuc_config()
    base = M.CFS_FANUC(obs, s1, ROBOT, ctx=ctx).optimizer()
    opt = M.CFS_FANUC(obs, s1, ROBOT, ctx=ctx).optimizer(check=dict(eta=ETA))
    one = ctx.solve_checked(s1["xR"][:, 0][None], s1["ff"][None], np.array([s1["caug"]]), s1["x_"][None], s1["epsilon_O"],
                            s1["MAX_O_ITER"], eta=ETA)
    assert np.array_equal(opt.u, one["u"][0]) and np.array_equal(opt.x_, one["x"][0]) and opt.status == one["status"][0]
    assert opt.verdict == one["verdict"][0] and opt.rounds_used == one["rounds_used"][0]
    assert np.array_equal(opt.margin_off, one["margin_off"][0])
    if one["rounds_used"][0] == 0:
        assert np.array_equal(opt.u, base.u)
    assert not hasattr(base, "verdict")
