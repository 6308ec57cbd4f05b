"""awe9 tracking vs awe9 economic MPC on one GPU: the same seeded x0, a closed loop of --steps MPC steps with the device plant step,
at each batch size.  One JSON line per (arm, batch): solves/s, SQP iterations per solve, ms per SQP iteration of the batch, the
status histogram, and the GPU name and power limit read in the same run.

The economic arm is configs.awe9_problem(..., mpc_type='economic'): a problem of the shape of the paper's AWE economic MPC (nx 9,
nu 3, ns 3, nsc 3, N 20, p 40, exact Hessian of a non-tracking cost), not its economic optimum.  The paper's 213 ms (economic)
and 13 ms (tracking) per SQP iteration are acados on one CPU core and one instance: context for the economic / tracking ratio,
not a like-for-like speed-up.

  python tools/bench_economic.py [--batches 16384 65536] [--steps 40] [--warmup 3]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info(device):
    import torch
    name = torch.cuda.get_device_name(device)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(device)],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out


def run_arm(pb, X0, steps, warmup, device):
    import torch
    from tunempc_b200.pmpc import Pmpc
    ctrl = Pmpc(pb, device=device)
    X0t = torch.tensor(X0, device="cuda:%d" % device)
    for _ in range(warmup):                                             # warm-up loop: module load, first-QP tables, allocations
        ctrl.reset(X0t.shape[0])
        X = X0t
        for _ in range(2):
            X = ctrl.plant_step(X, ctrl.step(X, outputs="u0"))
    torch.cuda.synchronize()
    ctrl.reset(X0t.shape[0])
    X = X0t
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    iters, hist = [], np.zeros(6, dtype=np.int64)
    ms = 0.0
    for _ in range(steps):
        e0.record()
        U = ctrl.step(X, outputs="u0")
        e1.record()
        e1.synchronize()
        ms += e0.elapsed_time(e1)
        iters.append(ctrl.log["iter"][-1].double().mean().item())
        hist += np.bincount(ctrl.status.cpu().numpy(), minlength=6)[:6]
        X = ctrl.plant_step(X, U)
    B = X0.shape[0]
    it = float(np.mean(iters))
    return {"B": B, "steps": steps, "solves_per_s": B * steps / (ms * 1e-3), "sqp_iter_per_solve": it,
            "ms_per_step": ms / steps, "ms_per_sqp_iteration_batch": ms / steps / it, "status_hist": hist.tolist()}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--batches", type=int, nargs="+", default=[1 << 14, 1 << 16])
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--seed", type=int, default=2024)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_economic.py measures the GPU: no CUDA device")
    from tunempc_b200 import configs
    from tunempc_b200.lib import ModelLib
    from tunempc_b200.problem import MpcProblem
    stage = ModelLib("awe9").stage_eval
    arms = {"awe9_tracking": MpcProblem.load(os.path.join(ROOT, "tests", "golden", "problem_awe9.npz")),
            "awe9_economic": configs.awe9_problem(stage, mpc_type="economic")[0]}
    name, plim = gpu_info(a.device)
    for B in a.batches:
        X0 = configs.sample_x0("awe9", arms["awe9_tracking"], B, a.seed)
        for arm, pb in arms.items():
            r = {"arm": arm, "mpc_type": pb.mpc_type, "gpu": name, "power_limit": plim, "seed": a.seed}
            r.update(run_arm(pb, X0, a.steps, a.warmup, a.device))
            print(json.dumps(r), flush=True)


if __name__ == "__main__":
    main()
