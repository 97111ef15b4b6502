"""Parity against the REAL reference: outputs of the unmodified Lib/CFS_FANUC.m / Lib/PSGCFS_FANUC.m (MATLAB + quadprog) written by
matlab/make_reference_golden.m into tests/golden/reference/<case>_ref.bin.  MATLAB cannot run in the build container, so these
files are absent until a MATLAB owner produces them; the tests then pin the oracle (CPU) and the CUDA path (-m gpu) to MATLAB at
north_star's tolerances (trajectory 1e-6 rad, cost 1e-6 relative, same iteration count).  The input fixtures that script reads
are always checked (they must round-trip and agree with the configurations the other tests use)."""
import glob
import os

import numpy as np
import pytest

from motionplanning_5d_m_b200 import fixture_io
from tests import common
from tests.golden import export_fixtures

HERE = os.path.dirname(os.path.abspath(__file__))
REF = sorted(glob.glob(os.path.join(HERE, "golden", "reference", "*_ref.bin")))
ROBOTS = ["M16iB", "M200i", "2L"]


def _problem(fx):
    ROBOT = ROBOTS[int(fx["robot_id"])]
    obs = [{"l": fx["obs_l"][:, :, j], "D": float(np.ravel(fx["obs_D"])[j]), "epsilon": float(np.ravel(fx["obs_epsilon"])[j])}
           for j in range(fx["obs_l"].shape[2])]
    s = dict(H=int(fx["H"]), njoint=int(fx["njoint"]), QQ=fx["QQ"], ff=np.ravel(fx["ff"]), caug=float(fx["caug"]),
             xR=np.ravel(fx["x0"])[:, None], x_=np.ravel(fx["x_"]), lim=np.ravel(fx["lim"]) if int(fx["has_lim"]) else None,
             MAX_input=np.ravel(fx["MAX_input"]), epsilon_O=float(fx["epsilon_O"]), MAX_O_ITER=int(fx["MAX_O_ITER"]),
             alpha=float(fx["alpha"]))
    noise = fx["noise"].T[None] if "noise" in fx else None
    return ROBOT, obs, s, int(fx["solver_id"]), noise


def test_fixtures_match_the_configurations_and_round_trip(tmp_path, oracle):
    """the fixtures make_reference_golden.m reads hold exactly the golden configurations; solving FROM a fixture reproduces the
    frozen oracle golden of the same case (so MATLAB and the oracle are fed identical numbers).  The arrays the config builders
    compute with BLAS / LAPACK (QQ, ff, caug, Aaug, Baug, alpha) match the committed fixture to rounding (common.frozen_inputs),
    every other array exactly."""
    g = common.golden("cases.npz")
    for name, arrays in export_fixtures.cases().items():
        p = tmp_path / (name + ".bin")
        fixture_io.write_fixture(str(p), arrays)
        fx = fixture_io.read_fixture(str(p))
        assert set(fx) == set(arrays) and all(np.array_equal(fx[k], np.asarray(arrays[k], dtype=np.float64)) for k in fx), name
        committed = os.path.join(HERE, "golden", "fixtures", name + ".bin")
        assert os.path.exists(committed), "run python tests/golden/export_fixtures.py"
        cf = fixture_io.read_fixture(committed)
        assert set(cf) == set(fx), name
        for k in fx:
            if k in ("QQ", "ff", "caug", "Aaug", "Baug", "alpha"):
                common.assert_rounding_close(fx[k], cf[k], (name, k))
            else:
                assert np.array_equal(cf[k], fx[k]), (name, k)
        ROBOT, obs, s, solver, noise = _problem(cf)
        P = common.oracle_problem(oracle, ROBOT, obs, s, solver=solver)
        r = P.solve_batch(s["xR"][:, 0][None], s["ff"][None], np.array([s["caug"]]), s["x_"][None], noise=noise)
        assert int(r["iters"][0]) == int(g[name + ".iters"]) and int(r["status"][0]) == int(g[name + ".status"])
        assert np.array_equal(r["x"][0], g[name + ".x"]), name


def _compare(name, ref, out):
    it = int(round(float(ref["iter_O"]))) - 1                       # iter_O = completed iterations + 1 (CFS_FANUC.m:77)
    assert int(out["iters"][0]) == it, (name, int(out["iters"][0]), it)
    assert np.abs(out["x"][0] - np.ravel(ref["x_"])).max() < 1e-6, name
    assert np.abs(out["u"][0] - np.ravel(ref["u"])).max() < 1e-6, name
    cm = np.ravel(ref["cost_all"])
    assert np.all(np.abs(out["cost_hist"][0, :it] - cm[:it]) <= 1e-6 * np.abs(cm[:it])), name


@pytest.mark.skipif(not REF, reason="no MATLAB reference goldens (matlab/make_reference_golden.m has not been run): parity unpinned above the leaves")
@pytest.mark.parametrize("path", REF)
def test_oracle_against_matlab(path, oracle):
    name = os.path.basename(path)[:-8]
    fx = fixture_io.read_fixture(os.path.join(HERE, "golden", "fixtures", name + ".bin"))
    ROBOT, obs, s, solver, noise = _problem(fx)
    P = common.oracle_problem(oracle, ROBOT, obs, s, solver=solver)
    out = P.solve_batch(s["xR"][:, 0][None], s["ff"][None], np.array([s["caug"]]), s["x_"][None], noise=noise)
    _compare(name, fixture_io.read_fixture(path), out)


@pytest.mark.gpu
@pytest.mark.skipif(not REF, reason="no MATLAB reference goldens (matlab/make_reference_golden.m has not been run)")
@pytest.mark.parametrize("path", REF)
def test_gpu_against_matlab(path, ctx):
    import motionplanning_5d_m_b200 as M
    name = os.path.basename(path)[:-8]
    fx = fixture_io.read_fixture(os.path.join(HERE, "golden", "fixtures", name + ".bin"))
    ROBOT, obs, s, solver, noise = _problem(fx)
    r = dict(M.robotproperty2(ROBOT))
    r["name"] = ROBOT
    ctx.set_robot(r, s["njoint"])
    ctx.set_obstacles(obs)
    ctx.set_cost(s["H"], s["QQ"], s["lim"], None if solver else s["MAX_input"])
    out = ctx.solve_batch(s["xR"][:, 0][None], s["ff"][None], np.array([s["caug"]]), s["x_"][None], s["epsilon_O"], s["MAX_O_ITER"],
                          solver=solver, noise=noise, alpha=s["alpha"])
    _compare(name, fixture_io.read_fixture(path), out)
