"""CPU tests of the checked solve's restatement: the offset oracle (tests/repair_oracle.c on a copy of oracle/cfs_oracle.c),
the repair increments, and the round loop of cfs_solve_checked (tests/repair_oracle.py)."""
import numpy as np
import pytest

from motionplanning_5d_m_b200 import synthetic
from tests import check_oracle as K
from tests import common
from tests import repair_oracle as R
from tests.test_oracle import _golden_cases

ETA = 1e-3


def _same(a, b):
    for k in ("u", "x", "cost_hist", "e_u_hist", "iters", "status"):
        assert np.array_equal(a[k], b[k], equal_nan=True), k


@pytest.mark.parametrize("name", ["main_fanuc_cfs", "main_fanuc_psgcfs", "main_2l_cfs", "m16ib_script_derivest",
                                  "m16ib_script_alt_numjac", "rrtstar_cfs"])
def test_offset_oracle_null_and_zero_equal_oracle(oracle, name):
    """NULL offsets and all-zero offsets reproduce the oracle bit for bit on the golden cases"""
    ROBOT, obs, s, solver, grad, noise = _golden_cases(oracle)[name]
    P = common.oracle_problem(oracle, ROBOT, obs, s, solver=solver, grad=grad)
    args = (s["xR"][:, 0][None], s["ff"][None], np.array([s["caug"]]), s["x_"][None])
    ref = P.solve_batch(*args, noise=noise)
    _same(R.solve_batch_off(P, *args, None, noise=noise), ref)
    _same(R.solve_batch_off(P, *args, np.zeros((1, len(obs), s["H"])), noise=noise), ref)


def test_constant_offset_equals_raised_margin(oracle):
    """a constant delta on every waypoint is a solve with margins m_j + delta, bit for bit"""
    cfg = common.batch_m16ib(oracle, 24)
    s, obs = cfg["sys_info"], cfg["obs"]
    d = 0.0123
    P = common.oracle_problem(oracle, "M16iB", obs, s)
    Pm = common.oracle_problem(oracle, "M16iB", obs, s, margin=[o["epsilon"] + d for o in obs])
    args = (cfg["x0"], cfg["ff"], cfg["caug"], cfg["xref"])
    _same(R.solve_batch_off(P, *args, np.full((24, len(obs), s["H"]), d)), Pm.solve_batch(*args))


def _scene2():
    o1 = dict(synthetic.OBS_M16IB)
    o2 = dict(o1, l=o1["l"] + np.array([[0.0], [0.3], [0.0]]))
    return K.Scene("M16iB", [o1, o2], margin_is_D=False)


def _witness(scene, x0, x, u, k, s):
    nj = scene.nj
    p = x0 if k == 0 else x[(k - 1) * 2 * nj:k * 2 * nj]
    return (p[:nj] + p[nj:2 * nj] * s) + ((0.5 * s) * s) * u[k * nj:(k + 1) * nj]


@pytest.mark.parametrize("nobs", [1, 2])
def test_increments_hand_computed(nobs):
    """hits on segment 0 (waypoint 0 never raised), on two adjacent segments (max, not sum), per obstacle"""
    sc = _scene2() if nobs == 2 else K.Scene("M16iB", [synthetic.OBS_M16IB], margin_is_D=False)
    rng = np.random.default_rng(5)
    H, nj = 6, 5
    x0 = np.concatenate([synthetic.SAMPLE_OFF, np.zeros(nj)])[None]
    x = (np.tile(x0, H) + rng.normal(0, 0.05, (1, 2 * nj * H)))
    u = rng.normal(0, 0.1, (1, nj * H))
    sv = np.zeros((1, H), dtype=np.int32)
    ss = np.full((1, H), -1.0)
    sv[0, [0, 2, 3]] = K.HIT
    ss[0, [0, 2, 3]] = [0.01, 0.02, 0.0]
    # a margin larger than any distance puts every witness below -eta/2; the second obstacle's is smaller, so its increments
    # differ from the first's
    sc.margin = np.ascontiguousarray(np.array([50.0, 40.0])[:sc.nobs])
    eta, gain = ETA, 2.0
    off = np.zeros((1, sc.nobs, H))
    R.repair_increments(sc, x0, x, u, sv, ss, eta, gain, off)
    inc = np.zeros((H, sc.nobs))
    for k in (0, 2, 3):
        th = _witness(sc, x0[0], x[0], u[0], k, ss[0, k])
        for j in range(sc.nobs):
            c = K.Scene.__new__(K.Scene)
            c.r, c.nj, c.nobs = sc.r, sc.nj, 1
            c.obs = np.ascontiguousarray(sc.obs[j * 7:(j + 1) * 7])
            c.margin = np.ascontiguousarray(sc.margin[j:j + 1])
            cj = c.clearance(th)[0]
            inc[k, j] = gain * (eta - cj) if cj < -eta / 2 else 0.0
    exp = np.zeros((sc.nobs, H))
    for i in range(1, H + 1):  # waypoint i: segments i-1 and i
        exp[:, i - 1] = np.maximum(inc[i - 1], inc[i] if i < H else 0.0)
    assert np.array_equal(off[0], exp)
    assert (inc > 0).sum() == 3 * sc.nobs and (off[0][:, 0] == inc[0]).all()  # segment 0 raises waypoint 1 only (0 is x0)
    assert (off[0][:, 2] == np.maximum(inc[2], inc[3])).all() and (inc[2] != inc[3]).all()  # between two hits: the max
    assert (off[0][:, 1] == inc[2]).all() and (off[0][:, 3] == inc[3]).all() and (off[0][:, 4:] == 0).all()
    # accumulation: a second call adds the same increments
    R.repair_increments(sc, x0, x, u, sv, ss, eta, gain, off)
    assert np.array_equal(off[0], exp + exp)


def _dense_clear(scene, x0, x, u, nj, dt, eta, npts=64):
    H = u.shape[0] // nj
    tau = np.linspace(0.0, dt, npts)
    return min(scene.clearance(K.segment_points(x0, x, u, nj, dt, k, tau)).min() for k in range(H)) >= -eta


def test_checked_loop_headline_256(oracle):
    """The restated round loop on 256 headline problems (H = 50, eta = 1 mm, gain 2, 4 rounds): every CLEAR trajectory passes a
    dense brute-force sample (64 points per segment, c >= -eta), and at least 80 % of the converged-and-HIT problems end CLEAR.
    Measured: 21 of the 202 converged problems are HIT after the first solve; all 21 end CLEAR."""
    cfg = common.batch_m16ib(oracle, 256)
    s, obs = cfg["sys_info"], cfg["obs"]
    P = common.oracle_problem(oracle, "M16iB", obs, s)
    sc = K.Scene("M16iB", obs, margin_is_D=False)
    args = (cfg["x0"], cfg["ff"], cfg["caug"], cfg["xref"])
    out = R.checked_solve(P, sc, *args, eta=ETA, rounds=4, gain=2.0)
    base = R.checked_solve(P, sc, *args, eta=ETA, rounds=0)
    conv0 = (base["status"] & 0xFF) == 0
    hit0 = conv0 & (base["verdict"] == K.HIT)
    assert conv0.sum() == 202 and hit0.sum() == 21, (conv0.sum(), hit0.sum())
    fixed = hit0 & (out["verdict"] == K.CLEAR)
    assert fixed.sum() >= 0.8 * hit0.sum(), (fixed.sum(), hit0.sum())
    cand = (base["verdict"] == K.HIT) & ((base["status"] & 0xFF) < 2)  # repaired: HIT and converged or MAX_ITER
    assert (out["rounds_used"][~cand] == 0).all() and (out["rounds_used"][fixed] >= 1).all()
    dt, nj = s["robot"]["delta_t"], 5
    for b in np.nonzero(out["verdict"] == K.CLEAR)[0]:
        assert _dense_clear(sc, cfg["x0"][b], out["x"][b], out["u"][b], nj, dt, ETA), b
    # untouched: problems never repaired are round 0's bit for bit
    same = out["rounds_used"] == 0
    for k in ("u", "x", "iters", "status"):
        assert np.array_equal(out[k][same], base[k][same]), k
