"""Device time of the continuous collision checks (k_check.cu), one JSON line on stdout.

  python dev/check_time.py [--batch 4096] [--horizon 50] [--seeds 1024] [--reps 20] [--eta 1e-3]

1. The headline batch (synthetic.batch_config_m16ib, seed 20261018: M16iB, one capsule, H = 50) is solved by the library; then
   cfs_check_trajectories_device runs on the solution resident in HBM (B*H segments), 2 warm-up launches, `reps` launches
   bracketed by CUDA events.  The HIT fraction of the batch at eta = 1 mm is printed (all problems, and converged ones).
2. Every tree edge of `seeds` RRT* trees of the RRTstar_CFS scene (M200i, two capsules) through cfs_check_edges_device, timed
   the same way.
Rates: items/s and clearance evaluations/s; achieved FP64 rate = evals * (555 + 325 * n_obs) FLOP / kernel time (FK of five
links ~555 FLOP, one link-axis distance ~65 FLOP per link and obstacle), against cfs_measure_fp64_peak measured in the same run,
and the evaluation histogram (log2 bins).  The GPU's name and power limit are read in the same run.  Nothing is written to the
repository tree.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import motionplanning_5d_m_b200 as M  # noqa: E402
from motionplanning_5d_m_b200 import _lib, rrt, synthetic  # noqa: E402


def gpu_info(index):
    try:
        q = subprocess.check_output(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                                     "--format=csv,noheader"], text=True, timeout=30).strip()
        name, plim, clk = [v.strip() for v in q.split(",")]
        return dict(gpu=name, power_limit=plim, sm_max_clock=clk)
    except Exception as e:  # the measurement stands without it, but says so
        return dict(gpu=torch.cuda.get_device_name(index), power_limit="unavailable (%s)" % type(e).__name__)


def timed(ctx, st, fn, reps):
    """ms per call of fn, which enqueues on the context's stream; the context runs on `st` so that the events bracket its
    kernels (torch's default stream is stream 0, which cfs_set_stream would read as "the context's own stream")"""
    ctx.set_stream(st.cuda_stream)
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for _ in range(reps):
        fn()
    b.record(st)
    torch.cuda.synchronize()
    ctx.set_stream(None)
    return a.elapsed_time(b) / reps


def hist(evals):
    ev = np.asarray(evals, dtype=np.int64)
    edges = [0, 1, 2, 4, 8, 16, 32, 64, 128, 256, 512, 1024, 2048, 4096, 1 << 30]
    h, _ = np.histogram(ev, bins=edges)
    return {("%d-%d" % (lo, hi - 1)): int(c) for lo, hi, c in zip(edges[:-1], edges[1:], h) if c}


def rates(ms, items, evals, nobs, peak_tf):
    fl = float(np.sum(evals)) * (555 + 325 * nobs)
    tf = fl / (ms * 1e-3) / 1e12
    return dict(ms=round(ms, 4), items=int(items), evals=int(np.sum(evals)), items_per_s=items / (ms * 1e-3),
                evals_per_s=float(np.sum(evals)) / (ms * 1e-3), fp64_tflops=tf, fp64_share_of_peak=tf / peak_tf,
                evals_hist=hist(evals))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--horizon", type=int, default=50)
    ap.add_argument("--seeds", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--eta", type=float, default=1e-3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("check_time.py measures on the GPU; no CUDA device is visible")
    dev = torch.device("cuda", 0)
    ctx = M.Context(0)
    info = gpu_info(0)
    peak_tf, _ = ctx.measure_fp64_peak()

    # 1. trajectories of the headline batch
    ctx.set_robot(dict(M.robotproperty2("M16iB"), name="M16iB"), 5)
    ctx.set_obstacles([synthetic.OBS_M16IB])
    cfg = synthetic.batch_config_m16ib(args.batch, lambda c: ctx.nodes_feasible(c)[0], horizon=args.horizon)
    s = cfg["sys_info"]
    ctx.set_cost(s["H"], s["QQ"], s["lim"], s["MAX_input"])
    sol = ctx.solve_batch(cfg["x0"], cfg["ff"], cfg["caug"], cfg["xref"], s["epsilon_O"], s["MAX_O_ITER"])
    B, H = args.batch, args.horizon
    t = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in (("x0", cfg["x0"]), ("x", sol["x"]), ("u", sol["u"]))}
    v = torch.zeros(B, dtype=torch.int32, device=dev)
    th, cm = torch.zeros(B, dtype=torch.float64, device=dev), torch.zeros(B, dtype=torch.float64, device=dev)
    ev = torch.zeros(B, dtype=torch.int32, device=dev)
    st = torch.cuda.Stream(dev)
    run = lambda: ctx.check_trajectories_ptr(B, H, t["x0"].data_ptr(), t["x"].data_ptr(), t["u"].data_ptr(), v.data_ptr(),
                                             th.data_ptr(), cm.data_ptr(), ev.data_ptr(), eta=args.eta, sync=False)
    ms_t = timed(ctx, st, run, args.reps)
    verdict, evals = v.cpu().numpy(), ev.cpu().numpy()
    conv = (sol["status"] & 0xFF) == 0
    traj = rates(ms_t, B * H, evals, 1, peak_tf)
    traj.update(trajectories=B, segments=B * H, hit_fraction=float((verdict == _lib.CHECK_HIT).mean()),
                hit_fraction_converged=float((verdict[conv] == _lib.CHECK_HIT).mean()), converged=int(conv.sum()),
                undecided=int((verdict == _lib.CHECK_UNDECIDED).sum()))

    # 2. every tree edge of `seeds` RRT* trees
    sc = rrt.SCENE_RRTSTAR
    ctx.set_robot(dict(M.robotproperty2("M200i"), name="M200i"), 5)
    ctx.set_obstacles(sc["obs"])
    S = args.seeds
    rng = np.random.Generator(np.random.Philox(synthetic.SEED))
    tile = lambda a: np.tile(np.asarray(a, dtype=np.float64).reshape(1, -1), (S, 1))
    tr = ctx.rrt_find_routes(tile(sc["x0"]), tile(sc["goal"]), tile(sc["goal"]), sc["region_g"], sc["region_s"], sc["sample_off"],
                             sc["ratial"], rng.random((S, rrt.NRND_DEFAULT)), star=True, want_tree=True)
    ta, tb = [], []
    for k in range(S):
        n = int(tr["n_nodes"][k])
        ta.append(tr["nodes"][k, tr["parent"][k, 1:n] - 1])
        tb.append(tr["nodes"][k, 1:n])
    ta, tb = np.concatenate(ta), np.concatenate(tb)
    N = ta.shape[0]
    da, db = torch.from_numpy(ta).to(dev), torch.from_numpy(tb).to(dev)
    v2, ev2 = torch.zeros(N, dtype=torch.int32, device=dev), torch.zeros(N, dtype=torch.int32, device=dev)
    sh, cm2 = torch.zeros(N, dtype=torch.float64, device=dev), torch.zeros(N, dtype=torch.float64, device=dev)
    run2 = lambda: ctx.check_edges_ptr(N, da.data_ptr(), db.data_ptr(), v2.data_ptr(), sh.data_ptr(), cm2.data_ptr(),
                                       ev2.data_ptr(), eta=args.eta, sync=False)
    ms_e = timed(ctx, st, run2, args.reps)
    edges = rates(ms_e, N, ev2.cpu().numpy(), len(sc["obs"]), peak_tf)
    edges.update(seeds=S, hit_fraction=float((v2.cpu().numpy() == _lib.CHECK_HIT).mean()))

    line = dict(metric="continuous_check", eta=args.eta, fp64_peak_tflops=peak_tf, trajectories=traj, tree_edges=edges, **info)
    print(json.dumps(line))
    ctx.close()


if __name__ == "__main__":
    main()
