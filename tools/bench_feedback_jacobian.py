"""Cost of the feedback Jacobian du0/dx0 (Pmpc.feedback_jacobian, tmpc_feedback_jacobian) next to the step it differentiates, on one
GPU: CSTR at 2^20 and awe9 at 2^14 and 2^16 seeded states, a closed loop of --steps MPC steps with the device plant step.  Each step
and each Jacobian call is timed with CUDA events on the current stream.  One JSON line per (config, batch): ms per step, ms per
Jacobian call, their ratio, QP solves per step, the step and Jacobian status histograms, and the GPU name and power limit read in
the same run.  The Jacobian costs about nx QP factorisations and solves per instance (one per column).

  python tools/bench_feedback_jacobian.py [--runs cstr:1048576 awe9:16384 awe9:65536] [--steps 10] [--warmup 2] [--out FILE]
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


def run(name, B, steps, warmup, device, seed):
    import torch
    from tunempc_b200 import configs
    from tunempc_b200.pmpc import Pmpc
    from tunempc_b200.problem import MpcProblem
    pb = MpcProblem.load(os.path.join(ROOT, "tests", "golden", "problem_%s.npz" % name))
    X0t = torch.tensor(configs.sample_x0(name, pb, B, seed), device="cuda:%d" % device)
    ctrl = Pmpc(pb, device=device)
    for _ in range(warmup):                                             # module load, first-QP tables, allocations
        ctrl.reset(B)
        X = X0t
        for _ in range(2):
            U = ctrl.step(X, outputs="u0")
            ctrl.feedback_jacobian()
            X = ctrl.plant_step(X, U)
    torch.cuda.synchronize()
    ctrl.reset(B)
    X = X0t
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    ms_step = ms_jac = 0.0
    qp = 0
    hist, jhist = np.zeros(6, dtype=np.int64), np.zeros(4, dtype=np.int64)
    for _ in range(steps):
        ev[0].record()
        U = ctrl.step(X, outputs="u0")
        ev[1].record()
        J, js = ctrl.feedback_jacobian()
        ev[2].record()
        ev[2].synchronize()
        ms_step += ev[0].elapsed_time(ev[1])
        ms_jac += ev[1].elapsed_time(ev[2])
        qp += ctrl.counters()["qp_solves"]
        hist += np.bincount(ctrl.status.cpu().numpy(), minlength=6)[:6]
        jhist += np.bincount(js.cpu().numpy(), minlength=4)[:4]
        X = ctrl.plant_step(X, U)
    return {"config": name, "B": B, "nx": pb.nx, "steps": steps, "ms_per_step": ms_step / steps, "ms_per_jacobian": ms_jac / steps,
            "jacobian_over_step": ms_jac / ms_step, "qp_solves_per_step_per_instance": qp / steps / B,
            "status_hist": hist.tolist(), "jstatus_hist": jhist.tolist()}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--runs", nargs="+", default=["cstr:%d" % (1 << 20), "awe9:%d" % (1 << 14), "awe9:%d" % (1 << 16)])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--seed", type=int, default=2024)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_feedback_jacobian.py measures the GPU: no CUDA device")
    gpu, plim = gpu_info(a.device)
    for spec in a.runs:
        name, B = spec.split(":")
        r = {"gpu": gpu, "power_limit": plim, "seed": a.seed}
        r.update(run(name, int(B), a.steps, a.warmup, a.device, a.seed))
        line = json.dumps(r)
        print(line, flush=True)
        if a.out:
            with open(a.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
