"""Cost of the solution VJP (Pmpc.solution_vjp, tmpc_solution_vjp) next to the step it differentiates and to the feedback Jacobian,
on one GPU: CSTR at 2^20 and awe9 at 2^14 and 2^16 seeded states, a closed loop of --steps MPC steps with the device plant step.
Each step, Jacobian and VJP call is timed with CUDA events on the current stream.  Two VJP forms: the last step's own solutions
(W = NULL: its linearisation records are reused) and the step's returned solution passed back (copied and linearised again, the
form autograd uses).  One JSON line per (config, batch): ms per step, per Jacobian and per VJP, the ratios, the share of the
re-linearisation in the stored-solution form, the status histograms, and the GPU name and power limit read in the same run.

  python tools/bench_solution_vjp.py [--runs cstr:1048576 awe9:16384 awe9:65536] [--steps 10] [--warmup 2] [--out FILE]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_feedback_jacobian import gpu_info  # noqa: E402


def run(name, B, steps, warmup, device, seed):
    import torch
    from tunempc_b200 import configs
    from tunempc_b200.pmpc import Pmpc
    from tunempc_b200.problem import MpcProblem
    pb = MpcProblem.load(os.path.join(ROOT, "tests", "golden", "problem_%s.npz" % name))
    dev = "cuda:%d" % device
    X0t = torch.tensor(configs.sample_x0(name, pb, B, seed), device=dev)
    g = torch.Generator(device=dev).manual_seed(seed)
    vu = torch.randn((B, pb.nu), dtype=torch.float64, device=dev, generator=g)
    vw = torch.randn((B, pb.n_w), dtype=torch.float64, device=dev, generator=g)
    ctrl = Pmpc(pb, device=device)

    def one_step(X, ev=None):
        rec = (lambda i: ev[i].record()) if ev else (lambda i: None)
        rec(0)
        U = ctrl.step(X, outputs="all")
        rec(1)
        _, js = ctrl.feedback_jacobian()
        rec(2)
        _, vs = ctrl.solution_vjp(v_u0=vu, v_w=vw)
        rec(3)
        _, ve = ctrl.solution_vjp(v_u0=vu, v_w=vw, w=ctrl.w_sol, lam_g=ctrl.lam_g, status=ctrl.status, phase=ctrl.last_phase)
        rec(4)
        return U, js, vs, ve

    for _ in range(warmup):                                             # module load, first-QP tables, allocations
        ctrl.reset(B)
        X = X0t
        for _ in range(2):
            U = one_step(X)[0]
            X = ctrl.plant_step(X, U)
    torch.cuda.synchronize()
    ctrl.reset(B)
    X = X0t
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    ms = np.zeros(4)
    jhist, vhist = np.zeros(4, dtype=np.int64), np.zeros(4, dtype=np.int64)
    agree = True
    for _ in range(steps):
        U, js, vs, ve = one_step(X, ev)
        ev[4].synchronize()
        ms += [ev[i].elapsed_time(ev[i + 1]) for i in range(4)]
        jhist += np.bincount(js.cpu().numpy(), minlength=4)[:4]
        vhist += np.bincount(ve.cpu().numpy(), minlength=4)[:4]
        agree &= bool(torch.equal(js, vs) and torch.equal(vs, ve))
        X = ctrl.plant_step(X, U)
    ms /= steps
    return {"config": name, "B": B, "nx": pb.nx, "steps": steps, "ms_per_step": ms[0], "ms_per_jacobian": ms[1],
            "ms_per_vjp_last_step": ms[2], "ms_per_vjp_stored": ms[3], "vjp_stored_over_step": ms[3] / ms[0],
            "vjp_stored_over_jacobian": ms[3] / ms[1], "relinearisation_share_of_stored": (ms[3] - ms[2]) / ms[3],
            "jstatus_hist": jhist.tolist(), "vjp_jstatus_hist": vhist.tolist(), "jstatus_equal": agree}


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
        raise SystemExit("bench_solution_vjp.py measures the GPU: no CUDA device")
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
