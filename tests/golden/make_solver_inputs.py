#!/usr/bin/env python
"""Freeze the solver inputs of the golden configurations that the config builders compute with BLAS / LAPACK products and SIMD
sums (QQ, ff, caug, alpha; tests/common.py frozen_inputs):

    python tests/golden/make_solver_inputs.py      ->  tests/golden/solver_inputs.npz

The values written must be the ones the goldens of cases.npz and stl_boxes.npz were computed from: the script checks that the
oracle reproduces every one of those goldens bit for bit from them, and writes nothing otherwise."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)


def main():
    import motionplanning_5d_m_b200 as M
    import oracle as O
    from tests import common
    inp, box = common.golden("inputs.npz"), common.golden("stl_boxes.npz")
    configs = {"main_fanuc": common.main_fanuc_config(), "main_2l": common.main_2l_config(),
               "m16ib_script": common.main_cfs_m16ib_config(inp["xuori"]), "rrtstar": common.rrtstar_route_config(inp["route_wp"]),
               "box_solve1": ("M16iB", None, None, M.make_sys_info(M.robotproperty2("M16iB"), 5, 30, box["solve1.theta0"],
                                                                  box["solve1.thetag"]))}
    alt = [dict(configs["m16ib_script"][2][0], l=np.array(common.OBS_M16_SCRIPT_ALT))]
    boxes = [{"shape": "box", "l": box["box_l"][:, :, j], "D": float(box["box_D"][j]), "epsilon": float(box["box_epsilon"][j])}
             for j in range(box["box_l"].shape[2])]
    s = configs["main_fanuc"][3]
    noise = np.random.default_rng(123).normal(0.0, 0.1, size=(1, s["MAX_O_ITER"], s["H"] * 5))
    cases = [  # (golden file, golden name, config, obstacles or None for the config's own, solver, grad, noise)
        ("cases.npz", "main_fanuc_cfs", "main_fanuc", None, 0, 0, None), ("cases.npz", "main_fanuc_psgcfs", "main_fanuc", None, 1, 0, noise),
        ("cases.npz", "main_2l_cfs", "main_2l", None, 0, 0, None), ("cases.npz", "m16ib_script_derivest", "m16ib_script", None, 0, 1, None),
        ("cases.npz", "m16ib_script_alt_derivest", "m16ib_script", alt, 0, 1, None),
        ("cases.npz", "m16ib_script_alt_numjac", "m16ib_script", alt, 0, 0, None), ("cases.npz", "rrtstar_cfs", "rrtstar", None, 0, 0, None),
        ("stl_boxes.npz", "solve1", "box_solve1", boxes, 0, 0, None)]
    for gname, name, cfg, obs, solver, grad, nz in cases:
        ROBOT, _, obs0, s = configs[cfg]
        P = common.oracle_problem(O, ROBOT, obs or obs0, s, solver=solver, grad=grad)
        r = P.solve_batch(s["xR"][:, 0][None], s["ff"][None], np.array([s["caug"]]), s["x_"][None], noise=nz)
        g = common.golden(gname)
        for k in ("x", "u", "iters", "status"):
            assert np.array_equal(r[k][0], g["%s.%s" % (name, k)]), (name, k, "these inputs are not the ones the golden came from")
    out = {"%s.%s" % (cfg, k): np.asarray(configs[cfg][3].get(k, 0.0), dtype=np.float64) for cfg in configs for k in common.FROZEN_KEYS}
    path = os.path.join(HERE, "solver_inputs.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
