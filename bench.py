#!/usr/bin/env python
"""bench.py -- BASELINE.json's headline metric: 5-DoF CFS trajectories/sec (M16iB, batch 4096, horizon 50).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one rank per GPU under torchrun)
  python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm's CPU port (oracle/) on host cores
  python bench.py --config psgcfs|rrtstar ...              # the other BASELINE.json configurations (parity cases with a number)
  python bench.py ... --dump-outputs DIR                   # + the last timed step's results as DIR/<name>.npy (float64)

--config cfs (default, the headline; BASELINE.json configs[2]).  One "step" = one pass of the hot path over one batch:
CFS_FANUC.optimizer run to the reference's stop rule for every problem of a 4096-problem synthetic batch.
  value  whole-job throughput with the inputs resident in HBM (cfs_solve_batch_device).  The K timed steps are issued
         round-robin on --contexts library contexts (each its own stream and buffer set), so the rare heavy-tier
         stragglers of batch k overlap the bulk of batch k+1 -- the GPU analogue of the reference's parfor workers;
         `latency_ms_single_batch` is one batch alone on an idle GPU.
  e2e    the same K steps through the host-pointer C-ABI call (cfs_solve_batch_async / cfs_wait) with pinned host
         buffers: H2D of every input and D2H of every result inside the timed region, copies of batch k+1 overlapping
         the kernels of batch k.  `e2e_pageable`: the same with pageable buffers (what a MATLAB caller passes).
--config psgcfs (configs[3]): PSGCFS_FANUC.optimizer on an M200i batch with host-drawn noise, sharded over the ranks.
--config rrtstar (configs[4]): RRTstar_CFS.m -- per rank and step, S RRT seeds of one scene grown on the device, every found
         route resampled + smoothed by CFS, the cheapest trajectory selected; over ranks the winner is chosen by an NCCL
         best-of (all-gather of costs, the winner contributes its trajectory) -- min(routeL) of s_Parallel_rrt.m:27 continued
         over GPUs.
Multi-GPU (cfs, psgcfs): every rank solves its own batches (weak scaling, no data-path collective); the per-problem
(cost, status) of the last step are all-gathered over NCCL once, inside the timed region (the final gather of north_star).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# One hardware queue per stream: with the default of 8 connections, the copies of one context queue behind the persistent
# kernels of another (false dependencies) and the e2e pipeline loses 40 % (measured: 2.75 -> 1.98 ms per step).
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

F_WAYPOINT_NUMJAC = 9680.0   # algorithmic FLOPs of one num_jac gradient (11 dist_arm evaluations), SURVEY.md section 8d
F_WAYPOINT_DERIVEST = 162080.0
METRIC = {"cfs": ("cfs_trajectories_per_sec", "trajectories/s"), "psgcfs": ("psgcfs_trajectories_per_sec", "trajectories/s"),
          "rrtstar": ("rrtstar_cfs_seeds_per_sec", "seeds/s")}
# dram__bytes_read.sum + dram__bytes_write.sum of the dominant launch, one `ncu --set full` capture (profiles/README.md)
DRAM_BYTES_PER_LAUNCH = {"cfs": None}
try:
    DRAM_BYTES_PER_LAUNCH.update(json.load(open(os.path.join(ROOT, "profiles", "dram_traffic.json"))))
except Exception:
    pass


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=96)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cfs", choices=["cfs", "psgcfs", "rrtstar"])
    ap.add_argument("--batch", type=int, default=0, help="problems (cfs 4096, psgcfs 2048) / RRT seeds (rrtstar 1024) per GPU and step")
    ap.add_argument("--horizon", type=int, default=0, help="cfs 50, psgcfs 30, rrtstar 40")
    ap.add_argument("--grad", default="numjac", choices=["numjac", "derivest"])
    ap.add_argument("--contexts", type=int, default=0, help="library contexts (streams + buffer sets) the steps rotate over (cfs and psgcfs 24, rrtstar 8)")
    ap.add_argument("--cpu-reps", type=int, default=3, help="CPU baseline: passes of the oracle over the same batch")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the arrays the timed path computed in its last step as "
                    "DIR/<name>.npy (float64, at most 64 MB in all), to compare two builds on the same seeded inputs")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    a.batch = a.batch or {"cfs": 4096, "psgcfs": 2048, "rrtstar": 1024}[a.config]
    a.horizon = a.horizon or {"cfs": 50, "psgcfs": 30, "rrtstar": 40}[a.config]
    a.contexts = a.contexts or {"cfs": 24, "psgcfs": 24, "rrtstar": 8}[a.config]
    return a


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md clocks line)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        if os.environ.get("BENCH_NO_CLOCKS"):
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([time.perf_counter()] + [c.strip() for c in line.split(",")])

    def mark(self):
        """start of the timed region: samples taken before it (warm-up) are only used if none fall inside it"""
        self.t_mark = time.perf_counter()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        inside = [r[1:] for r in self.rows if r[0] >= getattr(self, "t_mark", 0.0)]
        window = "timed region" if inside else "warm-up + timed region (no sample fell inside the timed region)"
        for r in (inside or [r[1:] for r in self.rows]):
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for nm, val in zip(names, r[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


DUMP_BYTES = 64 * 10 ** 6 - 4096  # 64 MB in all, less room for the .npy headers


def dump_outputs(path, arrays):
    """--dump-outputs: every array as <path>/<name>.npy in float64 (exact for the int32 iteration counts and status words).
    Above DUMP_BYTES in all, the same fixed seeded sample of rows is kept of every array whose first dimension is the batch
    (the largest one), and the sampled row indices go to rows.npy."""
    os.makedirs(path, exist_ok=True)
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    rows = max(a.shape[0] for a in arrays.values())
    per_row = sum(a.nbytes for a in arrays.values() if a.shape[0] == rows) / rows
    rest = sum(a.nbytes for a in arrays.values() if a.shape[0] != rows)
    if rest + per_row * rows > DUMP_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(rows, int((DUMP_BYTES - rest) // (per_row + 8)), replace=False))
        arrays = {k: a[keep] if a.shape[0] == rows else a for k, a in arrays.items()}
        arrays["rows"] = keep.astype(np.float64)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)
    print("bench.py: %d arrays (%.1f MB) written to %s" % (len(arrays), sum(a.nbytes for a in arrays.values()) / 1e6, path),
          file=sys.stderr, flush=True)


def bind_to_gpu_numa(index):
    """Multi-rank runs: keep this rank's threads (and hence its first-touch pinned staging buffers) on the CPU cores local to
    its GPU (sysfs local_cpulist of the GPU's PCI function).  Returns a short description for the JSON line, or None."""
    try:
        bus = subprocess.check_output(["nvidia-smi", "-i", str(index), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                                      text=True, timeout=20).strip().lower()
        if bus.startswith("00000000:"):
            bus = bus[4:]
        cpus = set()
        for part in open("/sys/bus/pci/devices/%s/local_cpulist" % bus).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return "%s: %d local cores" % (bus, len(cpus))
    except Exception:
        return None


def cpu_count():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def workload_text(args):
    if args.config == "psgcfs":
        return ("batched PSGCFS (BASELINE.json configs[3]): %d random start/goal pairs per GPU, LR Mate 200iD (M200i) capsules, "
                "horizon %d, the obstacle / weights of main_FANUC.m, host-drawn normrnd noise per outer iteration, 20 outer "
                "iterations (PSGCFS never meets the stop rule: eval.x_old stays ones)" % (args.batch, args.horizon))
    if args.config == "rrtstar":
        return ("RRTstar_CFS.m (BASELINE.json configs[4]): per GPU and step %d RRT seeds of the script's scene (M200i, two "
                "obstacle capsules) grown on the device from a host-drawn uniform stream, every found route resampled "
                "(cubicpolytraj, horizon %d) and smoothed by CFS, cheapest trajectory selected; NCCL best-of over the ranks"
                % (args.batch, args.horizon))
    return ("batched CFS (BASELINE.json configs[2]): %d random start/goal pairs per GPU, M16iB capsules, horizon %d, "
            "1 obstacle capsule, %s gradients, every problem run to the reference stop rule (eps 0.1, <= 20 outer "
            "iterations)" % (args.batch, args.horizon, "num_jac" if args.grad == "numjac" else "DERIVEST"))


def make_oracle_problem(O, cfg, grad, solver=0):
    s = cfg["sys_info"]
    return O.Problem(O.robot(cfg["ROBOT"]), s["H"], list(cfg["obs"]),
                     [o["epsilon"] if solver == 0 else o["D"] for o in cfg["obs"]], s["QQ"], s["lim"],
                     s["MAX_input"] if solver == 0 else None, s["epsilon_O"], s["MAX_O_ITER"], solver=solver, grad=grad,
                     alpha=s.get("alpha", 0.0))


def oracle_feasible(O, ROBOT, obs):
    r = O.robot(ROBOT)
    o6 = [O.obs6(o) for o in obs]
    return lambda cand: np.array([all(O.dist_arm(r, th, o)[0] >= ob["D"] for o, ob in zip(o6, obs)) for th in cand])


def oracle_batch(args, O):
    from motionplanning_5d_m_b200 import synthetic
    if args.config == "psgcfs":
        return synthetic.batch_config_m200i_psgcfs(args.batch, oracle_feasible(O, "M200i", [synthetic.OBS_M200I]), horizon=args.horizon)
    return synthetic.batch_config_m16ib(args.batch, oracle_feasible(O, "M16iB", [synthetic.OBS_M16IB]), horizon=args.horizon)


# ---- CPU legs (oracle port: MATLAB / Octave are not installed and the reference is MATLAB-only) ---------------------------------
def cpu_rrtstar_step(O, sc, rnd, H, cores):
    """One rrtstar step on the host: orc_rrt_find_route per seed (threads over seeds; ctypes releases the GIL), then the CFS
    stage set-up (RRTstar_CFS.m:96-187) and the oracle's CFS for every found route.  Returns (#seeds, best cost)."""
    from concurrent.futures import ThreadPoolExecutor

    import motionplanning_5d_m_b200 as M
    from motionplanning_5d_m_b200 import problem
    rob = O.robot("M200i")
    seg, D = [o["l"] for o in sc["obs"]], [o["D"] for o in sc["obs"]]

    def tree(k):
        return O.rrt_find_route(rob, seg, D, sc["x0"], sc["goal"], sc["region_g"], sc["region_s"], sc["sample_off"], sc["goal"],
                                sc["ratial"], rnd[k], star=False)
    with ThreadPoolExecutor(max_workers=cores) as ex:
        trees = list(ex.map(tree, range(rnd.shape[0])))
    routes = [t["route"] for t in trees if t is not None and not t["fail"]]
    if not routes:
        return rnd.shape[0], np.inf
    robot = M.robotproperty2("M200i")
    Aaug, Baug, Qaug, QQ = problem.build_cost_matrices(robot, 5, H, problem.Q_RRTSTAR, problem.R_MAIN_FANUC, 10.0)
    dt = robot["delta_t"]
    samp = [problem.cubicpolytraj(r.T, np.arange(len(r)) * dt, np.linspace(0, (len(r) - 1) * dt, H + 1)) for r in routes]
    x0 = np.stack([np.concatenate([s_[:, 0], np.zeros(5)]) for s_ in samp])
    gaug = np.stack([np.tile(np.concatenate([s_[:, -1], np.zeros(5)]), H) for s_ in samp])
    xref = np.stack([np.concatenate([np.concatenate([s_[:, i], np.zeros(5)]) for i in range(1, H + 1)]) for s_ in samp])
    ff, caug = problem.build_linear_term(Aaug, Baug, Qaug, x0, gaug)
    P = O.Problem(rob, H, seg, [o["epsilon"] for o in sc["obs"]], QQ, np.ones(5),
                  np.tile(np.array([1, 1, np.pi, np.pi, np.pi]) * dt, H), 0.1, 20)
    out = P.solve_batch(x0, ff, caug, xref, nthreads=cores)
    ok = ((out["status"] & 0xFF) < 2) & (out["iters"] > 0)
    fin = np.where(ok, out["cost_hist"][np.arange(len(routes)), np.maximum(out["iters"], 1) - 1], np.inf)
    return rnd.shape[0], float(fin.min())


def cpu_leg(args, O, cfg, steps, warm, cores, sample):
    """`steps` passes of the oracle over the first `sample` units of the seeded workload on `cores` threads -> (units/s, s, out)"""
    from motionplanning_5d_m_b200 import rrt
    if args.config == "rrtstar":
        rnd = np.random.default_rng(20261018).random((sample, rrt.NRND_DEFAULT))
        run = lambda: cpu_rrtstar_step(O, rrt.SCENE_RRTSTAR, rnd, args.horizon, cores)
    else:
        psg = args.config == "psgcfs"
        P = make_oracle_problem(O, cfg, 1 if args.grad == "derivest" else 0, solver=1 if psg else 0)
        nz = cfg["noise"][:sample] if psg else None
        run = lambda: P.solve_batch(cfg["x0"][:sample], cfg["ff"][:sample], cfg["caug"][:sample], cfg["xref"][:sample], noise=nz,
                                    nthreads=cores)
    for _ in range(warm):
        run()
    t0 = time.perf_counter()
    for _ in range(steps):
        out = run()
    dt = time.perf_counter() - t0
    return sample * steps / dt, dt, out


def run_reference(args, rank):
    """The reference algorithm on the host CPU.  MATLAB / Octave are not installed and the reference is pure MATLAB
    (nothing to pip-install), so this arm times the C port of the same algorithm (oracle/) on every host core, on the same
    seeded workload and the same batch per step as the b200 arm."""
    if rank != 0:
        return
    import oracle as O
    O.build()
    cores = cpu_count()
    cfg = None if args.config == "rrtstar" else oracle_batch(args, O)
    sample = args.batch if args.config != "rrtstar" else min(args.batch, 256)
    val, dt, out = cpu_leg(args, O, cfg, args.steps, min(args.warmup, 1), cores, sample)
    metric, unit = METRIC[args.config]
    line = {"impl": "reference", "metric": metric, "value": val, "unit": unit, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_text(args), "batch_per_gpu": args.batch, "horizon": args.horizon,
                       "sample_per_step": sample},
            "cpu_baseline": {"value": val, "unit": unit, "cores": cores, "kind": "port",
                             "sample": "%d units/step of the same seeded workload, %d steps, threads over problems / seeds" % (sample, args.steps)},
            "e2e": {"value": val, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "MATLAB/Octave unavailable offline and the reference is MATLAB-only: the C port of the reference "
                    "algorithm (oracle/cfs_oracle.c) is timed on all host cores"}
    if args.config != "rrtstar":
        line["ms_per_cfs_iter"] = 1e3 * dt / args.steps / max(int(out["iters"].max()), 1)
        line["converged_trajectories_per_sec"] = val * float(((out["status"] & 0xFF) == 0).mean())
    print(json.dumps(line), flush=True)


# ---- b200 arm ---------------------------------------------------------------------------------------------------------------------
class Env:
    pass


def make_env(args):
    import torch
    import torch.distributed as dist
    e = Env()
    e.torch, e.dist = torch, dist
    e.rank = int(os.environ.get("RANK", "0"))
    e.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    e.world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this framework has no CPU fallback")
    torch.cuda.set_device(e.local_rank)
    e.dev = torch.device("cuda", e.local_rank)
    e.numa = bind_to_gpu_numa(e.local_rank) if (e.world > 1 and not os.environ.get("BENCH_NO_NUMA")) else None  # N = 1 keeps every core for the CPU baseline leg
    if e.world > 1:
        dist.init_process_group("nccl", device_id=e.dev)
    e.main_stream = torch.cuda.Stream(device=e.dev)
    e.flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=e.dev)  # 256 MB > 126 MB L2
    e.launches = 0
    e.outputs = None  # --dump-outputs: host copies of the last timed step's results (rank 0)
    return e


def barrier(e):
    if e.world > 1:
        e.dist.barrier()
    e.torch.cuda.synchronize(e.dev)


def max_over_ranks(e, vals):
    t = e.torch.tensor(vals, dtype=e.torch.float64, device=e.dev)
    if e.world > 1:
        e.dist.all_reduce(t, op=e.dist.ReduceOp.MAX)
    return [float(v) for v in t]


def run_steps(e, ctxs, streams, steps, issue, host, after=None):
    """issue `steps` batches round-robin over the contexts; device ms between the first issue and the last completion"""
    torch = e.torch
    NC = len(ctxs)
    t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_begin.record(e.main_stream)
    for st in streams:
        st.wait_event(t_begin)
    t_host = time.perf_counter()
    for k in range(steps):
        c = k % NC
        if host and k >= NC:
            ctxs[c].wait()  # the host buffers of this context are about to be reused
        issue(c)
        e.launches += ctxs[c].stats()["launches"]
    e.host_issue_ms = (time.perf_counter() - t_host) * 1e3
    if after is not None:
        after((steps - 1) % NC)
    for st in streams:
        ev = torch.cuda.Event()
        ev.record(st)
        e.main_stream.wait_event(ev)
    t_end.record(e.main_stream)
    torch.cuda.synchronize(e.dev)
    for ctx in ctxs:
        ctx.wait()
    return t_begin.elapsed_time(t_end)


def out_set(e, B, n, K, pin):
    torch = e.torch
    mk = (lambda *sh, dt=torch.float64: torch.empty(sh, dtype=dt).pin_memory()) if pin else \
        (lambda *sh, dt=torch.float64: torch.empty(sh, dtype=dt, device=e.dev))
    return dict(u=mk(B, n), x=mk(B, 2 * n), cost=mk(B, K), eu=mk(B, K), iters=mk(B, dt=torch.int32), status=mk(B, dt=torch.int32))


def base_line(args, e, ms_dev, units_per_step):
    metric, unit = METRIC[args.config]
    return {"metric": metric, "value": e.world * units_per_step * args.steps / (ms_dev * 1e-3), "unit": unit, "n_gpus": e.world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic"}


def bench_solver(args, e):
    """--config cfs / psgcfs"""
    torch = e.torch
    import motionplanning_5d_m_b200 as M
    from motionplanning_5d_m_b200 import _lib, multi_gpu, problem, synthetic
    psg = args.config == "psgcfs"
    B, H, nj, NC = args.batch, args.horizon, 5, max(1, args.contexts)
    n, N = H * nj, 2 * H * nj
    grad_mode = _lib.GRAD_DERIVEST if args.grad == "derivest" else _lib.GRAD_NUMJAC
    solver = _lib.SOLVER_PSGCFS if psg else _lib.SOLVER_CFS
    ROBOT = "M200i" if psg else "M16iB"
    obs = [synthetic.OBS_M200I] if psg else [synthetic.OBS_M16IB]
    robot = dict(M.robotproperty2(ROBOT))
    robot["name"] = ROBOT
    ctxs, streams = [], []
    for c in range(NC):
        ctx = M.Context(e.local_rank)
        st = torch.cuda.Stream(device=e.dev)
        ctx.set_stream(st.cuda_stream)
        ctx.set_robot(robot, nj)
        ctx.set_obstacles(obs)
        for kv in filter(None, os.environ.get("BENCH_OPTS", "").split(",")):  # development: library scheduling options
            ctx.set_option(kv.split("=")[0], int(kv.split("=")[1]))
        ctxs.append(ctx)
        streams.append(st)
    feas = lambda cand: ctxs[0].nodes_feasible(cand)[0]
    mkcfg = (lambda sd: synthetic.batch_config_m200i_psgcfs(B, feas, horizon=H, seed=sd)) if psg else \
        (lambda sd: synthetic.batch_config_m16ib(B, feas, horizon=H, seed=sd))
    seed0 = synthetic.SEED + 1000 * int(os.environ.get("BENCH_SEED_RANK", e.rank))  # development: another rank's batches
    cfgs = [mkcfg(seed0 + c) for c in range(NC)]
    s = cfgs[0]["sys_info"]
    eps_o, K, alpha = float(s["epsilon_O"]), int(s["MAX_O_ITER"]), float(s.get("alpha", 0.0))
    for ctx in ctxs:
        ctx.set_cost(H, s["QQ"], s["lim"], None if psg else s["MAX_input"])
    setup_ms = ctxs[0].stats()["ms_setup"]
    names_in = ("x0", "ff", "caug", "xref") + (("noise",) if psg else ())
    d_in = [{k: torch.from_numpy(cfgs[c][k]).to(e.dev) for k in names_in} for c in range(NC)]
    d_out = [out_set(e, B, n, K, False) for _ in range(NC)]
    h_in = [{k: torch.from_numpy(cfgs[c][k]).pin_memory() for k in names_in} for c in range(NC)]
    h_out = [out_set(e, B, n, K, True) for _ in range(NC)]
    torch.cuda.synchronize(e.dev)

    def issue(c, host):
        i, o = (h_in[c], h_out[c]) if host else (d_in[c], d_out[c])
        ctxs[c].solve_batch_ptr(B, i["x0"].data_ptr(), i["ff"].data_ptr(), i["caug"].data_ptr(), i["xref"].data_ptr(),
                                eps_o, K, o["u"].data_ptr(), o["x"].data_ptr(), o["cost"].data_ptr(), o["eu"].data_ptr(),
                                o["iters"].data_ptr(), o["status"].data_ptr(), solver=solver, grad=grad_mode,
                                noise=i["noise"].data_ptr() if psg else 0, alpha=alpha, device=not host, sync=False)

    p_in = [{k: np.array(cfgs[c][k]) for k in names_in} for c in range(min(NC, 8))]      # pageable (numpy) buffers
    p_out = [dict(u=np.empty((B, n)), x=np.empty((B, N)), cost=np.empty((B, K)), eu=np.empty((B, K)),
                  iters=np.empty(B, dtype=np.int32), status=np.empty(B, dtype=np.int32)) for _ in range(min(NC, 8))]

    def issue_pageable(c):
        i, o = p_in[c % len(p_in)], p_out[c % len(p_out)]
        ptr = lambda a: a.ctypes.data
        ctxs[c].solve_batch_ptr(B, ptr(i["x0"]), ptr(i["ff"]), ptr(i["caug"]), ptr(i["xref"]), eps_o, K, ptr(o["u"]), ptr(o["x"]),
                                ptr(o["cost"]), ptr(o["eu"]), ptr(o["iters"]), ptr(o["status"]), solver=solver, grad=grad_mode,
                                noise=ptr(i["noise"]) if psg else 0, alpha=alpha, device=False, sync=False)

    def final_gather(c):
        """the one collective of the job: (cost, status) of the last step's problems from every rank (north_star: NCCL only
        for the final all-gather of per-problem costs)"""
        if e.world > 1:
            with torch.cuda.stream(streams[c]):
                fc = multi_gpu.final_cost(d_out[c]["cost"], d_out[c]["iters"])
                multi_gpu.gather_results({"cost": fc, "status": d_out[c]["status"]}, e.world * B)

    sampler = ClockSampler(e.local_rank)
    sampler.start()  # nvidia-smi needs up to a second to deliver its first row on an 8-GPU box: started before the warm-up
    W = max(args.warmup, 3)
    run_steps(e, ctxs, streams, max(W, NC), lambda c: issue(c, False), False, after=final_gather)  # incl. NCCL's lazy set-up
    run_steps(e, ctxs, streams, max(W, NC), lambda c: issue(c, True), True)
    barrier(e)
    # ---- timed: device-resident ---------------------------------------------------------------------------------------------
    e.flush.zero_()
    barrier(e)
    sampler.mark()
    e.launches = 0
    ms_dev = run_steps(e, ctxs, streams, args.steps, lambda c: issue(c, False), False,
                       after=None if os.environ.get("BENCH_NO_GATHER") else final_gather)
    barrier(e)
    if args.dump_outputs and e.rank == 0:  # what cfs_solve_batch_device returned for the last timed step's batch
        e.outputs = {k: v.cpu().numpy() for k, v in d_out[(args.steps - 1) % NC].items()}
    rank_ms = [ms_dev]
    if e.world > 1:  # every rank's own device time (diagnostic: the value uses the max)
        t_all = torch.zeros(e.world, dtype=torch.float64, device=e.dev)
        e.dist.all_gather_into_tensor(t_all, torch.tensor([ms_dev], dtype=torch.float64, device=e.dev))
        rank_ms = [float(v) for v in t_all]
    if os.environ.get("BENCH_QUICK"):  # development: resident leg only
        clk = sampler.stop()
        info = [None] * e.world
        mine = {"rank": e.rank, "issue_ms": round(e.host_issue_ms, 2), "sm_mhz": clk.get("sm_mhz"), "numa": e.numa,
                "cores": cpu_count(), "seed0": seed0}
        if e.world > 1:
            e.dist.all_gather_object(info, mine)
        else:
            info = [mine]
        if e.rank == 0:
            print(json.dumps({"quick_ranks": info}), flush=True)
        if e.rank == 0:
            print(json.dumps({"quick": True, "n_gpus": e.world, "ms_per_step": max(rank_ms) / args.steps,
                              "rank_ms_per_step": [v / args.steps for v in rank_ms], "clocks": clk}), flush=True)
        return
    wp_ctx = [ctxs[c].stats()["grad_waypoints"] for c in range(min(NC, args.steps))]
    wp_timed = sum(wp_ctx[k % NC] for k in range(args.steps))
    conv_ctx = [float(((d_out[c]["status"] & 0xFF) == 0).double().mean()) for c in range(min(NC, args.steps))]
    conv_frac = float(np.mean([conv_ctx[k % NC] for k in range(args.steps)]))
    # ---- timed: end to end through the host-pointer C ABI ------------------------------------------------------------------------
    e.flush.zero_()
    barrier(e)
    ms_e2e = run_steps(e, ctxs, streams, args.steps, lambda c: issue(c, True), True)
    barrier(e)
    launches_timed = e.launches
    clocks = sampler.stop()
    e2e_out = {k: h_out[0][k].numpy().copy() for k in ("x", "status", "iters", "cost")}
    ms_dev, ms_e2e = max_over_ranks(e, [ms_dev, ms_e2e])
    # ---- e2e with pageable host buffers (what a MATLAB caller passes: mxGetPr memory), staged inside the library -------------------
    NP = min(NC, 8)
    run_steps(e, ctxs[:NP], streams[:NP], NP, issue_pageable, True)
    barrier(e)
    ms_page = run_steps(e, ctxs[:NP], streams[:NP], args.steps, issue_pageable, True)
    barrier(e)
    (ms_page,) = max_over_ranks(e, [ms_page])

    # ---- one batch alone, per-tier CUDA events inside the library (timing level 2) --------------------------------------------------
    ctx0 = ctxs[0]
    ctx0.set_timing(2)
    lat = []
    for _ in range(3):
        e.flush.zero_()
        torch.cuda.synchronize(e.dev)
        issue(0, False)
        ctx0.wait()
        lat.append(ctx0.stats())
    stt = min(lat, key=lambda d: d["ms_total"])
    ctx0.set_timing(1)
    lat1 = []
    for _ in range(3):
        e.flush.zero_()
        torch.cuda.synchronize(e.dev)
        issue(0, False)
        ctx0.wait()
        lat1.append(ctx0.stats()["ms_total"])
    iters = d_out[0]["iters"].cpu().numpy()
    status = d_out[0]["status"].cpu().numpy()
    fused = stt["launches"] <= 12
    grad_phase = None
    if fused and not psg and args.grad == "numjac":
        # clock64 split of the warp tier (profiled instantiation of the kernel, timing level 3): the gradient code's own rate
        ctx0.set_timing(3)
        issue(0, False)
        ctx0.wait()
        wp = ctx0.warp_profile()
        ctx0.set_timing(1)
        if wp[0] > 0 and wp[4] > 0:
            grad_phase = {"cycles_gradient": int(wp[0]), "cycles_qp": int(wp[1]), "cycles_problems": int(wp[2]), "gradient_passes": int(wp[3]),
                          "resident_warps": int(wp[4]), "share_of_warp_cycles": float(wp[0]) / float(wp[2])}
    fp64_tf, fp64_mhz = ctx0.measure_fp64_peak()
    f_wp = F_WAYPOINT_DERIVEST if args.grad == "derivest" else F_WAYPOINT_NUMJAC
    grad_flops = f_wp * stt["grad_waypoints"]
    th_all = cfgs[0]["xref"].reshape(B, H, 2 * nj)[:, :, :nj].reshape(-1, nj)
    k1_ms = ctx0.time_dist_grad(th_all, grad=grad_mode, reps=10)
    k1_tf = f_wp * th_all.shape[0] / (k1_ms * 1e-3) / 1e12
    ms_sg, sg_status_equal = None, None
    if not psg:
        # e2e from start/goal pairs: the mains' problem set-up (main_FANUC.m:38-103) done on the device
        for ctx in ctxs:
            ctx.set_cost_blocks(H, problem.Q_MAIN_FANUC, problem.R_MAIN_FANUC, 50.0, s["lim"], s["MAX_input"])
        h_sg = [dict(t0=torch.from_numpy(np.ascontiguousarray(cfgs[c]["theta0"])).pin_memory(),
                     tg=torch.from_numpy(np.ascontiguousarray(cfgs[c]["thetag"])).pin_memory()) for c in range(NC)]

        def issue_sg(c):
            o = h_out[c]
            ctxs[c].solve_start_goal_ptr(B, h_sg[c]["t0"].data_ptr(), h_sg[c]["tg"].data_ptr(), eps_o, K, o["u"].data_ptr(), 0,
                                         o["cost"].data_ptr(), 0, o["iters"].data_ptr(), o["status"].data_ptr(), grad=grad_mode,
                                         sync=False)
        run_steps(e, ctxs, streams, NC, issue_sg, True)
        barrier(e)
        ms_sg = run_steps(e, ctxs, streams, args.steps, issue_sg, True)
        barrier(e)
        sg_status_equal = bool((h_out[0]["status"].numpy() == e2e_out["status"]).all())
        (ms_sg,) = max_over_ranks(e, [ms_sg])
    if fused:
        dom_ms, dom_name = stt["ms_bulk"] + stt["ms_heavy"], "k_cfs_warp (screen + bulk launches) + k_cfs_fused (heavy tier)"
    else:
        dom_ms = stt["ms_grad"] if stt["ms_grad"] >= stt["ms_qp"] else stt["ms_qp"]
        dom_name = "k_grad_%s" % args.grad if stt["ms_grad"] >= stt["ms_qp"] else "k_qp (+ k_psg_point, k_dgemm, k_psg_cost)"
    share = dom_ms / stt["ms_total"] if stt["ms_total"] else 1.0
    amort_ms = ms_dev / args.steps * share
    flops_per_launch = f_wp * wp_timed / args.steps
    ach_tf = flops_per_launch / (amort_ms * 1e-3) / 1e12
    ach_single_tf = grad_flops / (dom_ms * 1e-3) / 1e12 if dom_ms > 0 else 0.0
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    bytes_per_problem = 8.0 * ((2 * nj + n + 1 + N) + 3 * n + (n + N + 2 * K) + 1 + (n * K if psg else 0))
    hbm_ach = bytes_per_problem * B / (stt["ms_total"] * 1e-3) / 1e9
    if e.rank != 0:
        return
    h2d = sum(int(t.numel() * t.element_size()) for t in h_in[0].values())
    d2h = sum(int(t.numel() * t.element_size()) for t in h_out[0].values())
    line = base_line(args, e, ms_dev, B)
    unit = line["unit"]
    line.update({
        "config": {"workload": workload_text(args), "batch_per_gpu": B, "horizon": H,
                   "l2": "%d rotating buffer sets (one seeded batch each, %.0f MB of inputs+state+outputs in total) "
                         "> 126 MB L2; 256 MB flush before each timed region" % (NC, NC * B * (bytes_per_problem + 8 * 4 * n) / 1e6),
                   "contexts": NC, "seed": synthetic.SEED, "numa_binding": e.numa,
                   "parallelism": "independent problems sharded over %d GPU(s), no data-path collective; one NCCL all-gather "
                                  "of (cost,status) at the end of the timed region" % e.world},
        "e2e_arrays": {"value": e.world * B * args.steps / (ms_e2e * 1e-3), "unit": unit,
                       "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / args.steps,
                       "api": "cfs_solve_batch_async + cfs_wait (host pointers, pinned): every array of the class contract in "
                              "(x0, ff, caug, x_) and out (u, x_, cost_all, e_u_all, iters, status), H2D + solve + D2H of every "
                              "step inside the timed events, %d contexts in rotation" % NC},
        "e2e_pageable": {"value": e.world * B * args.steps / (ms_page * 1e-3), "unit": unit, "steps": args.steps,
                         "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": ms_page / args.steps,
                         "api": "the same entry with pageable (numpy / mxGetPr-like) caller buffers: the library stages them "
                                "through its own pinned buffers (one memcpy each way), %d contexts in rotation" % NP},
        "gpu_launches": int(launches_timed),
        "gpu_launches_note": "kernels launched by libcfs_b200 inside the two timed regions (device-resident + e2e), counted by "
                             "the library per solve (cfs_stats.launches: %d per step)" % int(stt["launches"]),
        "clocks": clocks,
        "rank_ms_per_step": [v / args.steps for v in rank_ms],
        "converged_trajectories_per_sec": e.world * B * args.steps / (ms_dev * 1e-3) * conv_frac,
        "latency_ms_single_batch": float(min(lat1)),
        "ms_per_cfs_iter": float(min(lat1)) / max(int(iters.max()), 1),
        "problem_iters_per_sec": float(stt["problem_iters"]) * args.steps / (ms_dev * 1e-3),
        "roofline": {"bound": "fp64", "kernel": dom_name,
                     "achieved": ach_tf, "peak": fp64_tf, "unit": "TFLOP/s", "frac": ach_tf / fp64_tf if fp64_tf else None,
                     "traffic": DRAM_BYTES_PER_LAUNCH.get(args.config) if (B == 4096 and H == 50) else None,
                     "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum summed over one step's four solver launches "
                                       "(screen, heavy#1, bulk, heavy#2), single-pass ncu run without replay save/restore "
                                       "(profiles/r02_dram_single_pass.csv; the --set full capture inflates writes, profiles/README.md)",
                     "peak_source": "measured here by cfs_measure_fp64_peak (DFMA micro-benchmark; MEASURED_PEAKS.json "
                                    "has no FP64 entry), implied SM clock %.0f MHz" % fp64_mhz,
                     "algorithmic_flops_per_launch": flops_per_launch, "avg_launch_ms": amort_ms,
                     "avg_launch_ms_basis": "timed region / steps x share_of_step: the %d timed steps overlap on %d "
                                            "streams, so this is the GPU time one step's solver launches cost in the timed region" % (args.steps, NC),
                     "single_launch": {"ms": dom_ms, "achieved": ach_single_tf,
                                       "frac": ach_single_tf / fp64_tf if fp64_tf else None,
                                       "note": "one batch alone on an idle GPU, tiers serialised (timing level 2)"},
                     "note": "algorithmic FLOPs = %.0f per waypoint gradient x %.0f waypoint gradients per step (SURVEY.md 8d); the "
                             "solver kernels also run the QP, roll-out and stop rule" % (f_wp, wp_timed / args.steps),
                     "share_of_step": share},
        "roofline_gradient_phase": None if grad_phase is None else dict(grad_phase, **{
            "bound": "fp64", "unit": "TFLOP/s", "peak": fp64_tf,
            "achieved": F_WAYPOINT_NUMJAC * grad_phase["gradient_passes"] * H * len(obs) /
                        (grad_phase["cycles_gradient"] / grad_phase["resident_warps"] / (fp64_mhz * 1e6)) / 1e12,
            "note": "the gradient code of the path that actually runs (k_cfs_warp's get_con phase, clock64 per warp): "
                    "algorithmic FLOPs of the gradient passes / (gradient-phase warp-cycles / resident warps) -- the rate the "
                    "kernel would sustain if every resident warp were in its gradient phase; frac = achieved / peak"}),
        "roofline_k1": {"bound": "fp64", "kernel": "k_grad_%s stand-alone" % args.grad, "achieved": k1_tf, "peak": fp64_tf,
                        "unit": "TFLOP/s", "frac": k1_tf / fp64_tf if fp64_tf else None, "waypoints": int(th_all.shape[0]),
                        "avg_launch_ms": k1_ms},
        "roofline_hbm": {"bound": "hbm", "achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_ach / hbm_peak,
                         "note": "%.1f KB algorithmic bytes per problem (inputs + v0 + outputs, once per solve)" % (bytes_per_problem / 1e3)},
        "breakdown_ms": {"single_batch_total_pipelined_tiers": float(min(lat1)), "single_batch_total_serialised_tiers": stt["ms_total"],
                         "bulk_tier": stt["ms_bulk"], "heavy_tier": stt["ms_heavy"], "grad_lockstep": stt["ms_grad"],
                         "qp_lockstep": stt["ms_qp"], "setup_once": setup_ms},
        "solve_stats": {"converged": int(((status & 0xFF) == 0).sum()), "max_iter": int(((status & 0xFF) == 1).sum()),
                        "infeasible": int(((status & 0xFF) == 2).sum()), "numerical": int(((status & 0xFF) == 3).sum()),
                        "mean_iters": float(iters.mean()), "max_iters": int(iters.max()),
                        "qp_steps": int(stt["qp_steps"]), "max_working_set": int(stt["max_active"])},
    })
    if line.get("roofline_gradient_phase"):
        g_ = line["roofline_gradient_phase"]
        g_["frac"] = g_["achieved"] / g_["peak"] if g_["peak"] else None
    if ms_sg is None:
        line["e2e"] = line["e2e_arrays"]
    else:
        line["e2e"] = {"value": e.world * B * args.steps / (ms_sg * 1e-3), "unit": unit,
                       "h2d_bytes_per_step": int(2 * B * nj * 8), "d2h_bytes_per_step": int(B * (n + K) * 8 + 2 * B * 4),
                       "ms_per_step": ms_sg / args.steps, "status_equal_to_array_path": sg_status_equal,
                       "api": "cfs_set_cost_blocks + cfs_solve_start_goal_async + cfs_wait, the documented batch entry (INTEGRATION.md): "
                              "start/goal pairs in from pinned host memory, the mains' set-up (straight-line reference, ff, caug: "
                              "main_FANUC.m:38-103) built on the device, u + cost history + iters + status back to the host "
                              "(x_ is the roll-out of u and is copied only on request); e2e_arrays is the array entry with "
                              "every input and output of the class contract copied"}
    if e.world == 1:
        # bounded CPU sample of the same workload: the oracle port on all host cores and on one, plus a parity check
        import oracle as O
        O.build()
        cores = cpu_count()
        S = B if args.grad == "numjac" else min(B, 256)
        c0 = cfgs[0]
        val, dt, ref = cpu_leg(args, O, c0, args.cpu_reps, 0, cores, S)
        S1 = min(S, 128)
        val1, dt1, _ = cpu_leg(args, O, c0, 1, 0, 1, S1)
        line["cpu_baseline"] = {"value": val, "unit": unit, "cores": cores, "kind": "port",
                                "sample": "%d passes over %d problems of the same batch, C port of the reference "
                                          "algorithm (oracle/), OpenMP over problems" % (args.cpu_reps, S), "seconds": dt,
                                "single_thread": {"value": val1, "unit": unit, "cores": 1, "sample": "%d problems" % S1, "seconds": dt1}}
        xg, sg, ig = (e2e_out[k][:S] for k in ("x", "status", "iters"))
        ok = ((ref["status"] & 0xFF) < 2) & ((ref["status"] & 0xFF) == (sg & 0xFF))
        dxp = np.abs(xg - ref["x"]).max(axis=1)
        dxp[~ok] = 0.0
        # conditioning probe: the twin oracle (same C restatement compiled with FMA contraction: a second faithful FP64
        # evaluation whose roundings differ in the last place); where the two CPU builds disagree the problem amplifies
        # rounding noise (DESIGN.md "parity noise floor")
        P = make_oracle_problem(O, c0, 1 if args.grad == "derivest" else 0, solver=1 if psg else 0)
        twin = P.solve_batch(c0["x0"][:S], c0["ff"][:S], c0["caug"][:S], c0["xref"][:S], noise=c0["noise"][:S] if psg else None,
                             nthreads=cores, use_twin=True)
        sens = np.abs(twin["x"] - ref["x"]).max(axis=1)
        cond = (sens < 1e-8) & (twin["status"] == ref["status"]) & (twin["iters"] == ref["iters"])
        well = ok & cond
        same = ((ref["status"] & 0xFF) == (sg & 0xFF)) & (ref["iters"] == ig)
        line["parity_sample"] = {"problems": S, "status_equal": bool(((ref["status"] & 0xFF) == (sg & 0xFF)).all()),
                                 "iters_equal": bool((ref["iters"] == ig).all()),
                                 "status_and_iters_equal_on_well_conditioned": bool(same[cond].all()),
                                 "touch_flag_equal": bool(((ref["status"] & 0x100) == (sg & 0x100)).all()),
                                 "max_abs_dx": float(dxp.max()) if ok.any() else None,
                                 "max_abs_dx_well_conditioned": float(dxp[well].max()) if well.any() else None,
                                 "ill_conditioned_problems": int((~cond).sum()),
                                 "ill_conditioned_rule": "the oracle and its FMA-contracted twin build (oracle/Makefile) differ by > 1e-8 in x, or in status / iteration count",
                                 "max_twin_difference": float(sens[ok].max()) if ok.any() else None,
                                 "problems_over_1e-6": int((dxp > 1e-6).sum()),
                                 "also_in": "tests/test_gpu_configs.py (pytest -m gpu, all 4096 problems)"}
    print(json.dumps(line), flush=True)


def bench_rrtstar(args, e):
    """--config rrtstar: RRT seeds -> CFS smoothing of every found route -> best-of (within the GPU, then over ranks by NCCL)"""
    torch = e.torch
    import motionplanning_5d_m_b200 as M
    from motionplanning_5d_m_b200 import multi_gpu, problem, rrt
    S, H, nj, NC, K, MAXIT = args.batch, args.horizon, 5, max(1, args.contexts), 20, 400
    n, cap, nrnd = H * nj, MAXIT + 2, rrt.NRND_DEFAULT
    sc = rrt.SCENE_RRTSTAR
    robot = dict(M.robotproperty2("M200i"))
    robot["name"] = "M200i"
    lim, mi = np.ones(5), np.tile(np.array([1, 1, np.pi, np.pi, np.pi]) * robot["delta_t"], H)
    ctxs, streams = [], []
    for c in range(NC):
        ctx = M.Context(e.local_rank)
        st = torch.cuda.Stream(device=e.dev)
        ctx.set_stream(st.cuda_stream)
        ctx.set_robot(robot, nj)
        ctx.set_obstacles(sc["obs"])
        ctx.set_cost_blocks(H, problem.Q_RRTSTAR, problem.R_MAIN_FANUC, 10.0, lim, mi)
        ctxs.append(ctx)
        streams.append(st)
    f64 = dict(dtype=torch.float64, device=e.dev)
    tile = lambda v: torch.from_numpy(np.tile(np.asarray(v, dtype=np.float64)[None], (S, 1))).to(e.dev)
    d_x0, d_goal = tile(sc["x0"]), tile(sc["goal"])
    d_par = torch.from_numpy(np.concatenate([sc["region_g"], sc["region_s"], sc["sample_off"], sc["ratial"]])).to(e.dev)
    rng = np.random.Generator(np.random.Philox(20261018 + 1000 * e.rank))
    h_rnd = [torch.from_numpy(rng.random((S, nrnd))).pin_memory() for _ in range(NC)]
    d_rnd = [t.to(e.dev) for t in h_rnd]
    buf = [dict(routes=torch.zeros((S, cap, nj), **f64), ints=[torch.zeros(S, dtype=torch.int32, device=e.dev) for _ in range(5)],
                u=torch.zeros((S, n), **f64), x=torch.zeros((S, 2 * n), **f64), c=torch.zeros((S, K), **f64),
                eu=torch.zeros((S, K), **f64), it=torch.zeros(S, dtype=torch.int32, device=e.dev),
                st=torch.zeros(S, dtype=torch.int32, device=e.dev), best=torch.zeros(2 * n + 2, **f64)) for _ in range(NC)]
    h_best = [torch.zeros(2 * n + 2, dtype=torch.float64).pin_memory() for _ in range(NC)]
    torch.cuda.synchronize(e.dev)

    def issue(c, host):
        b = buf[c]
        with torch.cuda.stream(streams[c]):
            if host:
                d_rnd[c].copy_(h_rnd[c], non_blocking=True)  # MATLAB's rand stream comes from the host (RRT_FANUC.m:108,111)
            i = b["ints"]
            ctxs[c].rrt_find_routes_device_ptr(S, False, d_x0.data_ptr(), d_goal.data_ptr(), d_goal.data_ptr(), d_par.data_ptr(), 0.5,
                                               MAXIT, d_rnd[c].data_ptr(), nrnd, b["routes"].data_ptr(), i[0].data_ptr(),
                                               i[1].data_ptr(), i[2].data_ptr(), i[3].data_ptr(), i[4].data_ptr())
            ctxs[c].solve_routes_var_ptr(S, cap, i[4].data_ptr(), b["routes"].data_ptr(), 0.1, K, b["u"].data_ptr(), b["x"].data_ptr(),
                                         b["c"].data_ptr(), b["eu"].data_ptr(), b["it"].data_ptr(), b["st"].data_ptr(), device=True,
                                         sync=False)
            # best-of within the GPU: argmin of the final cost over the seeds that produced a trajectory (s_Parallel_rrt.m:27)
            fc = multi_gpu.final_cost(b["c"], b["it"])
            fc = torch.where(((b["st"] & 0xFF) < 2) & torch.isfinite(fc), fc, torch.full_like(fc, float("inf")))
            cost, idx = fc.min(dim=0)
            status = torch.where(torch.isinf(cost), torch.full((1,), 2, dtype=torch.int32, device=e.dev),
                                 torch.zeros(1, dtype=torch.int32, device=e.dev))
            # ... then over the ranks: all-gather of the costs, the winning rank contributes its trajectory (NCCL)
            win, bestc, pay = multi_gpu.best_of(cost.reshape(1), status, {"x": b["x"][idx].reshape(1, -1)})
            b["best"][0] = bestc[0]
            b["best"][1] = win[0].double()
            b["best"][2:] = pay["x"][0]
            if host:
                h_best[c].copy_(b["best"], non_blocking=True)

    sampler = ClockSampler(e.local_rank)
    sampler.start()
    W = max(args.warmup, 3)
    run_steps(e, ctxs, streams, max(W, NC), lambda c: issue(c, False), False)
    run_steps(e, ctxs, streams, max(W, NC), lambda c: issue(c, True), False)
    barrier(e)
    e.flush.zero_()
    barrier(e)
    sampler.mark()
    e.launches = 0
    ms_dev = run_steps(e, ctxs, streams, args.steps, lambda c: issue(c, False), False)
    barrier(e)
    if args.dump_outputs and e.rank == 0:  # the last timed step: per-seed routes and CFS results, and the best-of
        b = buf[(args.steps - 1) % NC]
        i = b["ints"]
        e.outputs = {k: v.cpu().numpy() for k, v in dict(best=b["best"], routes=b["routes"], route_len=i[0], tree_nodes=i[1], fail=i[2],
                                                         u=b["u"], x=b["x"], cost=b["c"], eu=b["eu"], iters=b["it"], status=b["st"]).items()}
    e.flush.zero_()
    barrier(e)
    ms_e2e = run_steps(e, ctxs, streams, args.steps, lambda c: issue(c, True), False)
    barrier(e)
    launches_timed = e.launches + 2 * args.steps  # + the RRT kernel and its route_len kernel per step (not in cfs_stats)
    clocks = sampler.stop()
    ms_dev, ms_e2e = max_over_ranks(e, [ms_dev, ms_e2e])
    # ---- one step alone: stage times ------------------------------------------------------------------------------------------------
    torch.cuda.synchronize(e.dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    b, i = buf[0], buf[0]["ints"]
    with torch.cuda.stream(streams[0]):
        ev[0].record(streams[0])
        ctxs[0].rrt_find_routes_device_ptr(S, False, d_x0.data_ptr(), d_goal.data_ptr(), d_goal.data_ptr(), d_par.data_ptr(), 0.5, MAXIT,
                                           d_rnd[0].data_ptr(), nrnd, b["routes"].data_ptr(), i[0].data_ptr(), i[1].data_ptr(),
                                           i[2].data_ptr(), i[3].data_ptr(), i[4].data_ptr())
        ev[1].record(streams[0])
        ctxs[0].solve_routes_var_ptr(S, cap, i[4].data_ptr(), b["routes"].data_ptr(), 0.1, K, b["u"].data_ptr(), b["x"].data_ptr(),
                                     b["c"].data_ptr(), b["eu"].data_ptr(), b["it"].data_ptr(), b["st"].data_ptr(), device=True, sync=False)
        ev[2].record(streams[0])
    torch.cuda.synchronize(e.dev)
    ctxs[0].wait()
    ms_rrt, ms_cfs = ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])
    stt = ctxs[0].stats()
    found = int((i[4] >= 2).sum())
    nodes = i[1].cpu().numpy().astype(np.float64)
    used = i[3].cpu().numpy().astype(np.float64)
    fp64_tf, fp64_mhz = ctxs[0].measure_fp64_peak()
    # algorithmic FLOPs of the tree growth (SURVEY.md 8d): every sample = one nearest-neighbour scan over the tree so far
    # (3 * nj per node) + one feasibility test (555 + 325 * O); a sample consumes 1 + nj * bi = 3.5 uniform numbers on average
    samples = used / 3.5
    rrt_flops = float((samples * (555 + 325 * len(sc["obs"]))).sum() + (samples * 0.5 * nodes * 3 * nj).sum())
    cfs_flops = F_WAYPOINT_NUMJAC / 880.0 * (555 + 325 * len(sc["obs"])) * stt["grad_waypoints"] / len(sc["obs"])
    dom_rrt = ms_rrt >= ms_cfs
    dom_ms, dom_fl = (ms_rrt, rrt_flops) if dom_rrt else (ms_cfs, cfs_flops)
    share = dom_ms / (ms_rrt + ms_cfs)
    amort_ms = ms_dev / args.steps * share
    if e.rank != 0:
        return
    line = base_line(args, e, ms_dev, S)
    unit = line["unit"]
    line.update({
        "config": {"workload": workload_text(args), "seeds_per_gpu_and_step": S, "horizon": H, "contexts": NC, "numa_binding": e.numa,
                   "l2": "%d rotating buffer sets (%.0f MB of random streams, trees and trajectories) > 126 MB L2; 256 MB flush "
                         "before each timed region" % (NC, NC * S * (nrnd + cap * nj + 4 * n + 2 * K) * 8 / 1e6),
                   "parallelism": "every rank grows and smooths its own seeds of the SAME scene; per step one NCCL best-of "
                                  "(all-gather of the best cost per rank, all-reduce in which the winner contributes its trajectory)"},
        "e2e": {"value": e.world * S * args.steps / (ms_e2e * 1e-3), "unit": unit, "h2d_bytes_per_step": int(S * nrnd * 8),
                "d2h_bytes_per_step": int((2 * n + 2) * 8), "ms_per_step": ms_e2e / args.steps,
                "api": "cfs_rrt_find_routes_device + cfs_solve_routes_device per step, the uniform stream copied from pinned host "
                       "memory and the winning trajectory + cost copied back inside the timed events"},
        "gpu_launches": int(launches_timed), "clocks": clocks,
        "breakdown_ms": {"one_step_alone_rrt": ms_rrt, "one_step_alone_cfs_stage": ms_cfs},
        "solve_stats": {"seeds": S, "routes_found": found, "mean_tree_nodes": float(nodes.mean()),
                        "best_cost_last_step": float(buf[(args.steps - 1) % NC]["best"][0])},
        "roofline": {"bound": "fp64", "kernel": "k_rrt_find_routes" if dom_rrt else "CFS stage (k_cfs_warp + k_cfs_fused)",
                     "achieved": dom_fl / (amort_ms * 1e-3) / 1e12, "peak": fp64_tf, "unit": "TFLOP/s",
                     "frac": dom_fl / (amort_ms * 1e-3) / 1e12 / fp64_tf if fp64_tf else None, "traffic": None,
                     "algorithmic_flops_per_launch": dom_fl, "avg_launch_ms": amort_ms, "share_of_step": share,
                     "peak_source": "cfs_measure_fp64_peak (DFMA micro-benchmark), implied SM clock %.0f MHz" % fp64_mhz,
                     "note": "tree growth is sequential per seed (every sample is steered from the nearest node of the tree so far): "
                             "the kernel is bound by dependent-issue latency, not by the FP64 pipe"},
    })
    if e.world == 1:
        import oracle as O
        O.build()
        cores = cpu_count()
        Sc = min(S, 256)
        val, dt, _ = cpu_leg(args, O, None, 1, 0, cores, Sc)
        line["cpu_baseline"] = {"value": val, "unit": unit, "cores": cores, "kind": "port", "seconds": dt,
                                "sample": "%d seeds: orc_rrt_find_route per seed (threads over seeds) + the oracle's CFS on every found route" % Sc}
    print(json.dumps(line), flush=True)


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args, int(os.environ.get("RANK", "0")))
        return
    e = make_env(args)
    if args.config == "rrtstar":
        bench_rrtstar(args, e)
    else:
        bench_solver(args, e)
    if e.outputs is not None:
        o = e.outputs
        for k in ("cost", "eu"):  # NaN after each problem's last iteration (include/cfs_b200.h): written as 0, iters.npy has the length
            o[k] = np.where(np.arange(o[k].shape[1]) < o["iters"][:, None], o[k], 0.0)
        dump_outputs(args.dump_outputs, o)
    if e.world > 1:
        e.dist.destroy_process_group()


if __name__ == "__main__":
    main()
