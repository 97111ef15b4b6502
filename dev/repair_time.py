"""Per-round cost and effect of the checked solve (cfs_solve_checked_device) on the 4096-problem headline batch.

M16iB, H = 50, one capsule obstacle, eta = 1 mm, gain 2, 4 rounds.  Round r's time is taken with CUDA events around a
checked solve with rounds = r minus the one with rounds = r - 1 (each after a warm-up), since the rounds run inside one call.
Writes one JSON line (default profiles/r03_repair.json): per round the HIT fraction of the problems converged after round 0,
the problems re-solved, ms; the relative cost change of the repaired problems; the re-solves that became infeasible.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import oracle as O  # noqa: E402
from motionplanning_5d_m_b200 import _lib  # noqa: E402
from tests import common  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_repair.json"))
    ap.add_argument("--B", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    eta, gain, R = 1e-3, 2.0, 4
    cfg = common.batch_m16ib(O, args.B)
    s = cfg["sys_info"]
    ctx = _lib.Context(0)
    robot = dict(cfg["robot"], name="M16iB")
    ctx.set_robot(robot, 5)
    ctx.set_obstacles(cfg["obs"])
    ctx.set_cost(s["H"], s["QQ"], s["lim"], s["MAX_input"])
    dev = torch.device("cuda", 0)
    B, n, K, H = args.B, s["H"] * 5, s["MAX_O_ITER"], s["H"]
    T = lambda v: torch.from_numpy(np.ascontiguousarray(v)).to(dev)
    tin = [T(cfg[k]) for k in ("x0", "ff", "caug", "xref")]
    f64 = lambda *sh: torch.zeros(*sh, dtype=torch.float64, device=dev)
    i32 = lambda *sh: torch.zeros(*sh, dtype=torch.int32, device=dev)

    def run(rounds):
        o = dict(u=f64(B, n), x=f64(B, 2 * n), cost_hist=f64(B, K), e_u_hist=f64(B, K), iters=i32(B), status=i32(B), verdict=i32(B),
                 t_hit=f64(B), cmin=f64(B), rounds_used=i32(B), margin_off=f64(B, 1, H))
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ctx.solve_checked_ptr(B, *(t.data_ptr() for t in tin), s["epsilon_O"], K, *(o[k].data_ptr() for k in (
            "u", "x", "cost_hist", "e_u_hist", "iters", "status", "verdict", "t_hit", "cmin", "rounds_used", "margin_off")),
            eta=eta, rounds=rounds, gain=gain, sync=True)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), {k: v.cpu().numpy() for k, v in o.items()}

    ms, res = [], []
    for r in range(R + 1):
        run(r)  # warm-up
        t = sorted(run(r)[0] for _ in range(args.reps))
        ms.append(t[len(t) // 2])
        res.append(run(r)[1])
    r0 = res[0]
    conv0 = (r0["status"] & 0xFF) == 0
    rounds = []
    for r in range(R + 1):
        o = res[r]
        rounds.append(dict(round=r, hit_fraction_of_converged=float(((o["verdict"] == 1) & conv0).sum() / conv0.sum()),
                           resolved=int((o["rounds_used"] == r).sum()) if r else B,
                           ms=float(ms[r] - (ms[r - 1] if r else 0.0))))
    # problems re-solved in round r: those whose candidate was produced in r plus the failed candidates; count them from the
    # selection rule instead: HIT with status < 2 after round r - 1
    for r in range(1, R + 1):
        p = res[r - 1]
        prev_sel = (p["verdict"] == 1) & ((p["status"] & 0xFF) < 2)
        if r > 1:
            prev_sel &= res[r - 1]["rounds_used"] == r - 1
        rounds[r]["resolved"] = int(prev_sel.sum())
    o = res[R]
    hit0 = conv0 & (r0["verdict"] == 1)
    rep = hit0 & (o["rounds_used"] > 0)
    c0 = r0["cost_hist"][rep, r0["iters"][rep] - 1]
    c1 = o["cost_hist"][rep, o["iters"][rep] - 1]
    dc = c1 / c0 - 1
    # still HIT but re-solved fewer than R times: a re-solve failed (INFEASIBLE / NUMERICAL) and the problem stopped repairing
    infeasible = int((hit0 & (o["rounds_used"] < R) & (o["verdict"] == 1)).sum())
    name = torch.cuda.get_device_name(0)
    try:
        import subprocess
        pl = subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], text=True).split("\n")[0].strip()
    except Exception:
        pl = "unknown"
    line = dict(what="cfs_solve_checked_device, headline batch", B=B, H=H, eta=eta, gain=gain, rounds=R, device=name, power_limit=pl,
                converged_after_round0=int(conv0.sum()), hit_after_round0=int(hit0.sum()),
                cleared=int((hit0 & (o["verdict"] == 0)).sum()), still_hit=int((hit0 & (o["verdict"] == 1)).sum()),
                stopped_hit_before_last_round=infeasible,
                cost_change_repaired_median=float(np.median(dc)) if len(dc) else None,
                cost_change_repaired_max=float(np.max(np.abs(dc))) if len(dc) else None,
                per_round=rounds, ms_total_rounds=ms)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write(json.dumps(line) + "\n")
    print(json.dumps(line))


if __name__ == "__main__":
    main()
