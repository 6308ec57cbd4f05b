"""Feedback Jacobian du0/dx0, test infrastructure only: the CPU twin's Jacobian (tests/twin/twin_fbjac.cpp, the device routine
compiled with g++) and an independent dense KKT statement of it from the oracle's NLP classes.

At a solution (w*, lam*) of instance b the held rows are the equality rows and the inequality rows with lam* != 0 (stage-0 rows
that relax0 drops have no finite bound and are never held).  du0/dx0 is the u_0 block of dw in
    [H  J_A'; J_A  0] [dw; dlam] = [0; E],   E = identity on the init rows (g_init = x_0 - x0),
with H = hess(w, p, lam, 'exact') and J_A the rows of g(w, p, 1)'s Jacobian: numpy dense linear algebra, no device routine.
"""
import ctypes
import os
import subprocess

import numpy as np

from oracle import reference_port as rp

_TWIN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "twin")
_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

FIXTURES = ["lq", "cstr", "evaporation", "unicycle", "awe9", "evaporation_sc1", "cstr_economic", "evaporation_economic",
            "unicycle_economic"]


def relerr(a, b):
    return np.max(np.abs(a - b) / np.maximum(np.abs(b), 1.0))


def oracle_nlp(pb):
    """TrackingNlp for tuned problems; EconomicNlp (EconomicSlackNlp with slacks) with the config's l for economic ones"""
    if pb.mpc_type != "economic":
        return rp.TrackingNlp(pb)
    from tunempc_b200 import configs, tuning
    card = configs.CONFIGS[pb.name]()
    cf = tuning.lambdify_cost(card["model"], card["cost"])
    if pb.ns or pb.nsc:
        from economic_slack_support import EconomicSlackNlp
        return EconomicSlackNlp(pb, cf)
    return rp.EconomicNlp(pb, cf)


def dense_kkt_jacobian(nlp, pb, tab, x0, w, lam, phase=0):
    """du0/dx0 (nu, nx) at (w, lam) by one dense KKT solve with nx right-hand sides"""
    p0 = {"x0": np.asarray(x0, dtype=np.float64), "wref": tab.ref[phase], "H": tab.Href[phase], "q": tab.qref[phase]}
    _, Jg = nlp.g(w, p0, order=1)
    Hm = nlp.hess(w, p0, lam, "exact")
    lbg, ubg = pb.bounds()
    held = (lbg == ubg) | ((lam != 0) & np.isfinite(lbg))
    A = Jg[held]
    m = A.shape[0]
    K = np.block([[Hm, A.T], [A, np.zeros((m, m))]])
    rhs = np.zeros((pb.n_w + m, pb.nx))
    init_pos = np.nonzero(held)[0]
    for j in range(pb.nx):
        rhs[pb.n_w + int(np.nonzero(init_pos == j)[0][0]), j] = 1.0      # the init rows are the first rows of g, all held
    sol = np.linalg.solve(K, rhs)
    return sol[pb.iu(0)]


def active_set(pb, lam):
    return np.concatenate([lam[pb.g_h(k)] != 0 for k in range(pb.N)]) if pb.nh else np.zeros(0, dtype=bool)


def build_twin_fbjac(name):
    """g++-compile tests/twin/twin_fbjac.cpp into tests/twin/libtwin_fbjac_<name>.so (flags of the CPU twin, twin/twin.py)"""
    out = os.path.join(_TWIN, "libtwin_fbjac_%s.so" % name)
    srcs = [os.path.join(_TWIN, "twin_fbjac.cpp")] + [os.path.join(_ROOT, "tunempc_b200", "csrc", f) for f in
                                                       ("tmpc_core.cuh", "tmpc_qp.cuh", "gen/model_%s.h" % name)]
    if os.path.exists(out) and all(os.path.getmtime(out) >= os.path.getmtime(s) for s in srcs):
        return out
    subprocess.check_call(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-w"] + os.environ.get("TWIN_CXXFLAGS", "").split() + [
                           "-I" + os.path.join(_ROOT, "tunempc_b200/csrc"), "-I" + os.path.join(_ROOT, "tunempc_b200/csrc/gen"),
                           '-DTMPC_MODEL_HEADER="model_%s.h"' % name, srcs[0], "-o", out])
    return out


def twin_feedback_jacobian(tw, X0, out, tol=None, hessian=None, phase=None):
    """du0/dx0 (B, nu, nx) and its status (B,) on the CPU twin (twin_fbjac.cpp) at the solutions `out` of `tw.step(X0, tol=tol)`
    of a twin.Twin `tw` (or any dict with 'w', 'lam', 'status'): the stage records are linearised again at out['w'], out['lam'].
    tol: the step's tolerance (the weak-activity test reads it); phase: that step's phase (default: tw's last step)."""
    pb = tw.pb
    lib = ctypes.CDLL(build_twin_fbjac(pb.name))
    dp, ip = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int)
    p = lambda a: a.ctypes.data_as(dp)
    i = lambda a: a.ctypes.data_as(ip)
    X0 = np.ascontiguousarray(X0, dtype=np.float64).reshape(-1, pb.nx)
    B = X0.shape[0]
    hm = pb.hessian_approximation if hessian is None else hessian
    economic = getattr(pb, "mpc_type", "tuned") == "economic"
    if hm != "exact" and not economic:
        raise ValueError("the feedback Jacobian needs the exact Hessian")
    dims = np.array([pb.N, pb.nh, pb.nx_term, pb.p], dtype=np.int32)
    iopts = np.array([1, pb.max_iter, 300, tw.maxact, 1 if economic else 0, tw.reg_mode, tw.nonconvex_after], dtype=np.int32)
    dopts = np.array([pb.tol if tol is None else tol, 1e-8, 0.8, 1e-8, tw.rho_rel], dtype=np.float64)
    wref_d, H_d, q_d = pb.device_tables()
    Hs = np.ascontiguousarray(0.5 * (H_d + np.transpose(H_d, (0, 2, 1))))
    relax0 = np.zeros(max(pb.nh, 1), dtype=np.int32)
    for r in pb.relax0:
        relax0[r] = 1
    tidx = np.array(pb.term_idx, dtype=np.int32)
    C = np.ascontiguousarray(pb.C if pb.nh else np.zeros((1, pb.nz)))
    c = np.ascontiguousarray(pb.c if pb.nh else np.zeros(1))
    wref = np.ascontiguousarray(wref_d); q = np.ascontiguousarray(q_d); rdu = np.ascontiguousarray(tw.tab.ref_du)
    W = np.ascontiguousarray(out["w"], dtype=np.float64); LAM = np.ascontiguousarray(out["lam"], dtype=np.float64)
    st = np.ascontiguousarray(out["status"], dtype=np.int32)
    J = np.zeros((B, pb.nu, pb.nx)); jst = np.zeros(B, dtype=np.int32)
    ph = (tw.index - 1) % pb.p if phase is None else phase
    ret = lib.twin_feedback_jacobian(i(dims), i(iopts), p(dopts), p(wref), p(Hs), p(q), p(rdu), p(C), p(c), i(tidx), i(relax0),
                                     ctypes.c_int(ph), ctypes.c_longlong(B), p(X0), p(W), p(LAM), i(st), p(J), i(jst))
    if ret:
        raise RuntimeError("twin_feedback_jacobian returned %d" % ret)
    return J, jst
