"""Cost of joint position limits (cfs_set_joint_limits) on the 4096-problem headline batch.

M16iB, H = 50, one capsule obstacle.  Two configurations: the sampling box SAMPLE_OFF +- REGION_S on all 4096 problems (every
start and goal lies inside it; the rows rarely bind), and the active limits of the tests (joints 3 and 5 at SAMPLE_OFF +-
0.5 REGION_S, tests/test_limits.py) on the problems whose start lies inside them (upper and lower rows bind in about half).
Runs the plain solve, the plain solve through the margin-offset instantiations (all-zero offsets: the kernels the limits
instantiations extend, same results) and the limited solve alternately (median of --reps each, host clock around the
synchronous host entry: copies included), then the plain and limited forms of one checked solve (eta = 1 mm, 4 rounds).
Reports ms per batch; the shares of the problems with status < 2 that end with a joint on an upper / a lower limit (within
1e-9: such a row active in the final QP) and outside the limits; the bulk and heavy tiers' times of one extra run with the
tiers serialised (timing level 2); the largest working set; status counts.  The library does not count escalations to the
heavy tier; its serialised time and the largest working set stand for them.  Writes one JSON line (default
profiles/r05_limits.json); an infinite limit is written as null.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import oracle as O  # noqa: E402
from motionplanning_5d_m_b200 import _lib, synthetic  # noqa: E402
from tests import common  # noqa: E402
from tests.test_limits import inside_box, limit_box  # noqa: E402


def measure(ctx, cfg, s, idx, limits, reps):
    lo, hi = limits
    B = len(idx)
    a = tuple(np.ascontiguousarray(cfg[k][idx]) for k in ("x0", "ff", "caug", "xref")) + (s["epsilon_O"], s["MAX_O_ITER"])
    zero = np.zeros((B, len(cfg["obs"]), s["H"]))

    def run(limited, checked):
        ctx.set_joint_limits(*((lo, hi) if limited == "limits" else (None, None)))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if checked:
            out = ctx.solve_checked(*a, eta=1e-3, rounds=4, gain=2.0)
        elif limited == "offsets":
            out = ctx.solve_batch_margins(*a[:4], zero, *a[4:])
        else:
            out = ctx.solve_batch(*a)
        ms = (time.perf_counter() - t0) * 1e3
        return ms, out, ctx.stats()

    fin = lambda v: [float(x) if np.isfinite(x) else None for x in v]
    res = dict(problems=B, qmin=fin(lo), qmax=fin(hi))
    for checked in (False, True):
        kinds = ("plain", "limits") if checked else ("plain", "offsets", "limits")
        for lim in kinds:
            run(lim, checked)  # warm-up
        t = {k: [] for k in kinds}
        for _ in range(reps):
            for lim in kinds:
                t[lim].append(run(lim, checked)[0])
        for lim in kinds:
            _, out, _ = run(lim, checked)
            ctx.set_timing(2)  # tiers serialised: the heavy tier's own time
            st = run(lim, checked)[2]
            ctx.set_timing(1)
            th = out["x"].reshape(B, s["H"], 10)[:, :, :5]
            good = (out["status"] & 0xFF) < 2
            up = (np.abs(th - hi) <= 1e-9).any(axis=(1, 2))
            dn = (np.abs(th - lo) <= 1e-9).any(axis=(1, 2))
            outside = ((th > hi + 1e-9) | (th < lo - 1e-9)).any(axis=(1, 2))
            key = ("checked_" if checked else "solve_") + lim
            res[key] = dict(ms_median=float(np.median(t[lim])), ms_all=[round(v, 3) for v in t[lim]],
                            share_upper_active=float(up[good].mean()), share_lower_active=float(dn[good].mean()),
                            share_outside_limits=float(outside[good].mean()),
                            converged=int(((out["status"] & 0xFF) == 0).sum()), max_iter=int(((out["status"] & 0xFF) == 1).sum()),
                            infeasible=int(((out["status"] & 0xFF) == 2).sum()), numerical=int(((out["status"] & 0xFF) == 3).sum()),
                            ms_bulk_serialised=float(st["ms_bulk"]), ms_heavy_serialised=float(st["ms_heavy"]),
                            max_working_set=int(st["max_active"]), launches=int(st["launches"]))
            if checked:
                res[key]["clear"] = int((out["verdict"] == 0).sum())
    ctx.set_joint_limits(None, None)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_limits.json"))
    ap.add_argument("--B", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    cfg = common.batch_m16ib(O, args.B)
    s = cfg["sys_info"]
    ctx = _lib.Context(0)
    ctx.set_robot(dict(cfg["robot"], name="M16iB"), 5)
    ctx.set_obstacles(cfg["obs"])
    ctx.set_cost(s["H"], s["QQ"], s["lim"], s["MAX_input"])
    box = (synthetic.SAMPLE_OFF - synthetic.REGION_S, synthetic.SAMPLE_OFF + synthetic.REGION_S)
    sel = inside_box(cfg)
    res = {"sampling_box": measure(ctx, cfg, s, np.arange(args.B), box, args.reps),
           "active_limits": measure(ctx, cfg, s, sel, limit_box(), args.reps)}
    ctx.set_joint_limits(None, None)
    q = lambda f: subprocess.check_output(["nvidia-smi", "--query-gpu=" + f, "--format=csv,noheader"], text=True).split("\n")[0].strip()
    line = dict(what="joint position limits, headline batch", B=args.B, H=s["H"], escalations="not counted by the library",
                device=torch.cuda.get_device_name(0), power_limit=q("power.limit"), sm_clock=q("clocks.sm"), **res)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write(json.dumps(line) + "\n")
    print(json.dumps(line))


if __name__ == "__main__":
    main()
