#!/usr/bin/env python
"""bench.py -- tuned-MPC solves/sec (batched Pmpc.step, fp64) on the CSTR config of BASELINE.json.

  python bench.py --gpus N --steps K --warmup W            B200 arm (under torchrun for N > 1, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K ...  CPU arm: the oracle port of the reference loop on host cores
  python bench.py --config lq|evaporation|unicycle|awe9 ...  the other BASELINE.json configs at their own batch sizes
  python bench.py --scaling strong ...                     fixed 2^20 instances in total, split over the ranks
  python bench.py --dump-outputs DIR ...                   also write the last timed step's u0 / status as DIR/*.npy

A "step" = one pass of the hot path over one batch: `ctrl.reset(); ctrl.step(X0)` for B = 2^20 seeded initial states
per GPU (the alpha-sweep loop of tunempc/closed_loop_tools.py:43-68 as one batched call).  Weak scaling: every rank
solves its own 2^20-instance shard, no collective on the solve path; NCCL is used only for the statistics.
Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

if "reference" in sys.argv:
    # CPU arm: one single-threaded worker process per core -- keep the BLAS / OpenMP pools from oversubscribing the box
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
        os.environ[_v] = "1"

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "tuned-MPC solves/sec (batched step, fp64)"
UNIT = "solves/s"


# BASELINE.json configs: fixture, default batch per GPU, MPC steps per bench step (closed loop), workload text
CONFIGS = {
    "cstr": dict(B=1 << 20, cl=1, text="cstr N=20 tuned NMPC (examples/cstr)"),
    "lq": dict(B=1 << 10, cl=1, text="convex LQR N=10 tuned MPC (examples/convex_lqr.py)"),
    "evaporation": dict(B=1 << 18, cl=1, text="evaporation process N=30 tuned NMPC, collocation, state constraints (examples/evaporation_process)"),
    "unicycle": dict(B=1 << 16, cl=100, text="unicycle p=N=30 periodic tuned MPC, 100-step closed loop, plant = model (examples/unicycle)"),
    "awe9": dict(B=1 << 14, cl=40, text="AWE-shaped stand-in (configs.awe9: nx=9 nu=3 ns=3 nsc=3 nh=17 N=20 p=40, slacks us/usc, nonlinear rows g, "
                                        "L1 slack cost), 40-step closed loop over one period, plant = model (examples/awe_system dimensions)"),
}


def sample_x0(pb, B, seed, name="cstr"):
    """SURVEY.md section 8(d): the examples' own perturbation recipes, seeded (cstr: cA sweep alpha in [-0.1, 1.0] of
    examples/cstr/main.py:124-131 plus 1e-2*|x_s| jitter); same generator as the golden fixtures."""
    from tunempc_b200 import configs
    return configs.sample_x0(name, pb, B, seed)


def load_problem(name="cstr"):
    from tunempc_b200.problem import MpcProblem
    return MpcProblem.load(os.path.join(ROOT, "tests", "golden", "problem_%s.npz" % name))


def algorithmic_flops_per_stage_lin(exact=True, name="cstr"):
    """SURVEY.md section 8(d): fp64 add/mul/div = 1, FMA = 2, op counts of the generated model code (modelgen).
    RK4 models: the formula of SURVEY 8(d).  Discrete models: one evaluation (M = 1/4 of an RK4 step).  Collocation models:
    per finite element 4 Newton iterations (3 stage evaluations f + J, LU of the 3nx x 3nx iteration matrix, one solve), then
    one solve per first-order direction and per second-order pair against the same factorisation (tm_colloc_stage)."""
    from tunempc_b200 import configs, modelgen
    import tempfile
    m = configs.CONFIGS[name]()["model"]
    with tempfile.TemporaryDirectory() as d:
        oc = modelgen.generate_header(m, os.path.join(d, "m.h"))
    nx, nu, M = m.nx, m.nu, m.rk_steps
    nz = nx + nu
    c_f, c_J = oc["c_f"], oc["c_J"] - oc["c_f"]
    c_H = (oc["c_H"] - oc["c_J"]) + oc["c_bilin"]
    if getattr(m, "discrete", False):
        f_gn = c_f + c_J + 2 * nx * nx * nz
        f_ex = f_gn + c_H + 2 * nz * nz * nx + 2 * nx * nz * nz
        return (f_ex if exact else f_gn), c_f
    if getattr(m, "integrator", "rk") == "collocation":
        n = 3 * nx
        lu, sol = 2 * n ** 3 // 3, 2 * n * n
        newton = 4 * (3 * (c_f + c_J) + lu + sol)
        first = nz * (3 * 2 * nx * nz + sol)
        second = (nz * (nz + 1) // 2) * (3 * (c_H // max(nz * (nz + 1) // 2, 1) + 2 * nz * nz + 2 * nx * nx) + sol)
        f_gn = M * (newton + first)
        return (f_gn + M * second if exact else f_gn), M * newton
    f_gn = M * (4 * (c_f + c_J + 2 * nx * nx * nz) + 16 * nx * (1 + nz))
    f_ex = f_gn + M * 4 * (c_H + 2 * nz * nz * nx + 2 * nx * nz * nz)
    f_dyn = M * (4 * c_f + 16 * nx)
    return (f_ex if exact else f_gn), f_dyn


class ClockSampler(threading.Thread):
    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.idx = gpu_index
        self.stop_ev = threading.Event()
        self.rows = []

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self.stop_ev.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop_ev.wait(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(self.rows), "power_w_max": max(float(r[2]) for r in self.rows)}


# ------------------------------------------------------------------------------------------------------------
def _oracle_worker(args):
    idx_list, seed, name = args
    from threadpoolctl import threadpool_limits
    from oracle import reference_port as rp
    pb = load_problem(name)
    ctrl = rp.Pmpc(pb)
    X0 = sample_x0(pb, max(idx_list) + 1, seed, name)
    t = time.perf_counter()
    with threadpool_limits(limits=1):
        for i in idx_list:
            ctrl.reset()                                   # closed_loop_tools.py:68
            ctrl.step(X0[i])                               # closed_loop_tools.py:56
    return time.perf_counter() - t, len(idx_list)


def _twin_worker(args):
    """compiled CPU baseline (BASELINE.md B2): the solver source of the CUDA library compiled as a sequential host program
    (tests/twin, test infrastructure), one process per core, each on its own chunk of the sample"""
    lo, hi, seed, name, build_dir = args
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from twin.twin import Twin
    from tunempc_b200.problem import build_tables
    pb = load_problem(name)
    X0 = sample_x0(pb, hi, seed, name)[lo:hi]
    tw = Twin(pb, build_tables(pb), build_dir=build_dir)
    tw.reset(hi - lo)
    t = time.perf_counter()
    o = tw.step(X0)
    return time.perf_counter() - t, hi - lo, int((o["status"] == 0).sum())


def compiled_cpu_baseline(name, per_core=48, seed=1000):
    import multiprocessing as mp
    import tempfile
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from twin.twin import build as twin_build
    cores = len(os.sched_getaffinity(0))
    n = cores * per_core
    with tempfile.TemporaryDirectory(prefix="tmpc_twin_") as d:   # the benchmark writes nothing into the tree (it may be read-only)
        jobs = [(c * per_core, (c + 1) * per_core, seed, name, d) for c in range(cores)]
        twin_build(name, d)                                # g++ once, before the pool forks
        t0 = time.perf_counter()
        with mp.get_context("fork").Pool(cores) as pool:
            res = pool.map(_twin_worker, jobs)
        dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "%d x0 of the same distribution (%d per core, %d converged), the CUDA library's solver source compiled with g++ -O2 "
                      "as a sequential host program (tests/twin), one process per core" % (n, per_core, sum(r[2] for r in res))}


def run_reference_arm(args):
    """CPU arm: the oracle port of `for x0: ctrl.reset(); ctrl.step(x0)` on all host cores (one process per core)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    from oracle import reference_port as rp
    name = args.config
    rp.build((name,))
    backend = "qpOASES_e (reference tree, oracle/_ref)" if rp.qpoases_available() else "dense null-space + Goldfarb-Idnani (oracle fallback: oracle/_ref missing)"
    cores = len(os.sched_getaffinity(0))
    per_core = 6 if name != "awe9" else 1          # ~2 s of CPU work per core and step
    n = cores * per_core
    chunks = [list(range(c, n, cores)) for c in range(cores)]
    ctx = mp.get_context("fork")
    times = []
    with ctx.Pool(cores) as pool:
        for s in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            pool.map(_oracle_worker, [(c, 1000 + s, name) for c in chunks])
            dt = time.perf_counter() - t0
            if s >= args.warmup:
                times.append(dt)
    tot = sum(times)
    val = n * len(times) / tot
    line = {"metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * tot / len(times), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "impl": "reference",
            "config": {"workload": "%s, exact Hessian, reset+step per x0" % CONFIGS[name]["text"],
                       "sample": "%d x0 per step (bounded sample of the workload of the B200 arm)" % n},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "qp_backend": backend,
                             "sample": "%d instances per step (oracle port: numpy + C stage functions + QP backend), %d steps" % (n, len(times))},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    try:
        line["cpu_baseline_compiled"] = compiled_cpu_baseline(name)
    except Exception as e:
        line["cpu_baseline_compiled"] = {"value": None, "sample": "failed: %r" % (e,)}
    print(json.dumps(line))


def ncu_traffic():
    """DRAM bytes per unit of the dominant kernels from the newest committed `ncu --set full` capture
    (profiles/ncu_traffic.json, written by tools/ncu_traffic.py from the .ncu-rep of the same code)."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as fh:
            return json.load(fh)
    except Exception:
        return {}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write each (B, ...) array as out_dir/<name>.npy (float64) for output-by-output comparison of two builds.  Inputs are
    seeded, so the same arguments give the same rows; above 64 MB in all, the same fixed seeded sample of rows is kept
    from every array (its indices go to rows.npy)."""
    host = {k: np.asarray(v.cpu().numpy() if hasattr(v, "cpu") else v, dtype=np.float64) for k, v in arrays.items()}
    B = next(iter(host.values())).shape[0]
    row_bytes = sum(a[0].nbytes for a in host.values())
    if B * row_bytes > DUMP_LIMIT_BYTES:
        n = (DUMP_LIMIT_BYTES - 4096) // (row_bytes + 8)            # 4 KB for the .npy headers
        rows = np.sort(np.random.default_rng(0).choice(B, n, replace=False))
        host = {k: a[rows] for k, a in host.items()}
        host["rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in host.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


# ------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--config", default="cstr", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=0, help="instances per GPU per step (default: the config's BASELINE.json size)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="strong: the batch is the TOTAL, split over the ranks")
    ap.add_argument("--hessian", default="exact")
    ap.add_argument("--cpu-sample", type=int, default=40, help="x0 of the batch timed on the CPU oracle port (about 12 s)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (u0, status) as DIR/<name>.npy, to compare two builds "
                         "(B200 arm on one GPU only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs writes the outputs of the B200 arm on one GPU: not with --impl reference or more than one rank")
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist
    from tunempc_b200.pmpc import Pmpc

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 arm has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout for the one JSON line
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    name = args.config
    cfg = CONFIGS[name]
    pb = load_problem(name)
    pb.hessian_approximation = args.hessian
    ctrl = Pmpc(pb, device=local)
    B = args.batch or cfg["B"]
    if args.scaling == "strong":
        B = B // world                                    # fixed total work
    CL = cfg["cl"]
    W = max(args.warmup, 3)
    K = args.steps
    nbatches = 2
    X0_host = [torch.from_numpy(sample_x0(pb, B, 100 + 17 * rank + i, name)).pin_memory() for i in range(nbatches)]
    X0_dev = [x.to(dev) for x in X0_host]
    peak_tf = ctrl.fp64_peak_tflops()
    acc = {"lin_ms": 0.0, "qp_ms": 0.0, "post_ms": 0.0, "n_lin": 0, "n_qp": 0, "n_it": 0, "n_launch": 0, "n_dyn": 0}

    def account():
        t = ctrl.timing()
        c = ctrl.counters()
        acc["lin_ms"] += t["lin_ms"]; acc["qp_ms"] += t["qp_ms"]; acc["post_ms"] += t["post_ms"]
        acc["n_lin"] += c["stage_linearisations"]; acc["n_qp"] += c["qp_solves"]; acc["n_it"] += c["sqp_iterations"]
        acc["n_launch"] += c["kernel_launches"]; acc["n_dyn"] += c["ls_dynamics_evals"]

    # ---- one bench step: reset + step (cl = 1) or a CL-step closed loop with the model as plant (unicycle) ----
    def one_step(x, count=False):
        ctrl.reset()
        if CL == 1:
            u = ctrl.step(x, outputs="u0")
            if count:
                account()
            return u
        X = x
        host = isinstance(X, np.ndarray)
        for _ in range(CL):
            U = ctrl.step(X, outputs="u0")
            if count:
                account()
            if host:                                      # end-to-end arm: state and input cross the boundary every MPC step
                X = ctrl.plant_step(torch.as_tensor(X, device=dev), torch.as_tensor(U, device=dev)).cpu().numpy()
            else:
                X = ctrl.plant_step(X, U)
        return U

    # ---- device-resident arm: inputs already in HBM --------------------------------------------------------
    for i in range(W):
        one_step(X0_dev[i % nbatches])
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        U_last = one_step(X0_dev[i % nbatches], count=True)
    e1.record()
    barrier()
    ms_dev = e0.elapsed_time(e1)
    status = ctrl.status
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"u0": U_last, "status": status})
    flags = ctrl.log["flags"][-1]
    stat_hist = torch.bincount(status.to(torch.int64), minlength=6)[:6].to(torch.float64)
    # per-bit counts: [no flag, GN fallback (1), damped step (2), GN re-solve (4), non-convex primal step (8)]
    fl_hist = torch.stack([(flags == 0).sum()] + [((flags & b) != 0).sum() for b in (1, 2, 4, 8)]).to(torch.float64)

    # ---- end-to-end arm: host buffers through the C ABI (tmpc_step_host), H2D + D2H inside the timed region ----
    x_np = [x.numpy() for x in X0_host]
    one_step(x_np[0])
    barrier()
    t0 = time.perf_counter()
    for i in range(K):
        one_step(x_np[i % nbatches])
    torch.cuda.synchronize()
    ms_e2e_local = 1e3 * (time.perf_counter() - t0)
    barrier()
    sampler.stop_ev.set()
    sampler.join(timeout=2)

    tvec = torch.tensor([ms_dev, ms_e2e_local], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tvec, op=dist.ReduceOp.MAX)              # max over ranks
        dist.all_reduce(stat_hist, op=dist.ReduceOp.SUM)         # closed-loop statistics: the only collectives
        dist.all_reduce(fl_hist, op=dist.ReduceOp.SUM)
    ms_dev, ms_e2e = float(tvec[0]), float(tvec[1])

    if rank == 0:
        lin_ms, qp_ms, post_ms = acc["lin_ms"], acc["qp_ms"], acc["post_ms"]
        n_lin, n_qp = acc["n_lin"], acc["n_qp"]
        f_lin, f_dyn = algorithmic_flops_per_stage_lin(args.hessian == "exact", name)
        ach = (n_lin * f_lin) / (lin_ms * 1e-3) / 1e12 if lin_ms > 0 else 0.0
        # Algorithmic bytes: a stage task reads (x,u,lam_dyn) and writes its record xf | S | W; a QP reads its N records + w and
        # writes (d, lam).  Measured DRAM traffic: profiles/ncu_traffic.json (ncu --set full of this code, tools/ncu_traffic.py).
        nzm = pb.nx + pb.nu                                # the linearisation record holds model variables only (no slack columns)
        npair = nzm * (nzm + 1) // 2
        lin_alg_bytes_per_task = 8.0 * (pb.nx + pb.nu + pb.nx) + 8.0 * (pb.nx + pb.nx * nzm + npair)
        qp_alg_bytes = 8.0 * (pb.N * (pb.nx + pb.nx * nzm + npair) + 2 * pb.n_w + pb.n_g + pb.nx)
        tr = ncu_traffic().get(name, {})
        lin_tr, qp_tr = tr.get("lin", {}), tr.get("qp", {})
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
                hbm_peak = float(json.load(fh)["hbm_gbs"])
            hbm_src = "MEASURED_PEAKS.json hbm_gbs"
        except Exception:
            hbm_peak, hbm_src = 6550.0, "fallback (B200_PROFILING.md)"
        qp_ach = n_qp * qp_alg_bytes / (qp_ms * 1e-3) / 1e9 if qp_ms > 0 else 0.0
        solves = world * B * K * CL
        roof_lin = {"bound": "fp64", "kernel": lin_tr.get("kernel", "k_lin2 / k_lin"), "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s",
                    "frac": ach / peak_tf if peak_tf else None,
                    "traffic": lin_tr["dram_bytes_per_task"] * B * pb.N if "dram_bytes_per_task" in lin_tr else None,
                    "traffic_note": "ncu dram read+write per full-batch launch: %s B per stage task (capture %s), algorithmic %.0f B"
                                    % (lin_tr.get("dram_bytes_per_task"), lin_tr.get("capture"), lin_alg_bytes_per_task),
                    "peak_source": "in-run DFMA micro-benchmark (tmpc_fp64_peak); MEASURED_PEAKS.json has no FP64 figure",
                    "flops_per_stage_linearisation": f_lin, "stage_linearisations": int(n_lin),
                    "hbm_GBps_boundary_io": (B * K * CL * 8 * (pb.nx + pb.nu) + 0.0) / (ms_dev * 1e-3) / 1e9}
        roof_qp = {"bound": "hbm", "kernel": qp_tr.get("kernel", "k_qp_thread (+ k_qp0, k_qp)"), "achieved": qp_ach, "peak": hbm_peak, "unit": "GB/s",
                   "frac": qp_ach / hbm_peak,
                   "traffic": qp_tr["dram_bytes_per_qp"] * B if "dram_bytes_per_qp" in qp_tr else None,
                   "note": "algorithmic %.0f B per QP (records + w in, d + lam out); measured DRAM traffic %s B per QP (capture %s)"
                           % (qp_alg_bytes, qp_tr.get("dram_bytes_per_qp"), qp_tr.get("capture")),
                   "peak_source": hbm_src}
        lin_dominant = lin_ms >= 0.8 * qp_ms            # the linearisation is the named kernel unless the QP clearly dominates
        line = {
            "metric": METRIC, "value": solves / (ms_dev * 1e-3), "unit": UNIT, "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "%s, %s Hessian, B=%d x0 per GPU per step, %s" % (cfg["text"], args.hessian, B,
                                   "reset+step" if CL == 1 else "reset + %d closed-loop steps" % CL),
                       "l2": "working set %.1f GB per step >> L2; %d alternating input batches" % (B * 8.0 * (3 * pb.n_w + 3 * pb.n_g + pb.N * (pb.nx + pb.nx * nzm + npair)) / 1e9, nbatches),
                       "x0": "seeded perturbation recipe of the example (tunempc_b200.configs.sample_x0), seed 100+17*rank+i"},
            "e2e": {"value": solves / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": B * pb.nx * 8 * CL,
                    "d2h_bytes_per_step": (B * pb.nu * 8 + 3 * B * 4) * CL + (B * pb.nx * 8 * CL if CL > 1 else 0)},
            "gpu_launches": int(acc["n_launch"]),
            "kernel_ms": {"k_lin": lin_ms, "k_qp": qp_ms, "k_post": post_ms, "step_total": ms_dev},
            "clocks": sampler.summary(),
            "roofline": roof_lin if lin_dominant else roof_qp,
            ("roofline_qp" if lin_dominant else "roofline_lin"): roof_qp if lin_dominant else roof_lin,
            "stats": {"sqp_iter_mean": acc["n_it"] / (B * K * CL), "qp_solves": int(n_qp), "ls_dynamics_evals": int(acc["n_dyn"]),
                      "status_hist": [int(v) for v in stat_hist.tolist()], "flags_hist": [int(v) for v in fl_hist.tolist()],
                      "flags_hist_keys": ["none", "gn_fallback", "damped", "gn_resolve", "nonconvex_step"]},
        }
        # ---- CPU baselines on bounded samples of the same workload: the oracle port on one core, the compiled twin on all ----
        try:
            from oracle import reference_port as rp
            oc = rp.Pmpc(load_problem(name))
            n = args.cpu_sample if pb.n_w < 300 else min(args.cpu_sample, 6)     # the dense 369-variable QPs of awe9 take seconds each
            xs = x_np[0][:n]
            from threadpoolctl import threadpool_limits
            with threadpool_limits(limits=1):              # "cores": 1 means one thread, BLAS included
                t0 = time.perf_counter()
                for i in range(n):
                    oc.reset()
                    oc.step(xs[i])
                dt = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": n / dt, "unit": UNIT, "cores": 1, "kind": "port",
                                    "qp_backend": "qpOASES_e (reference tree, oracle/_ref)" if rp.qpoases_available() else "dense fallback",
                                    "sample": "first %d x0 of the same batch, oracle port (numpy + C stage functions + QP backend)" % n}
        except Exception as e:   # the oracle is a checker, its absence must not hide the GPU number
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 1, "kind": "port", "sample": "failed: %r" % (e,)}
        if args.cpu_sample > 1:
            try:
                line["cpu_baseline_compiled"] = compiled_cpu_baseline(name)
            except Exception as e:
                line["cpu_baseline_compiled"] = {"value": None, "sample": "failed: %r" % (e,)}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
