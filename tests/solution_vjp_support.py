"""Solution VJP G = v_u0' du0/dx0 + v_w' dw/dx0, test infrastructure only: the CPU twin's VJP (tests/twin/twin_vjp.cpp, the
device routine compiled with g++) and independent dense KKT statements of it from the oracle's NLP classes.

With K = [H J_A'; J_A 0] at a solution (held rows A as in feedback_jacobian_support), the forward form is
    dw/dx0 = the w block of K^-1 [0; E]          (E = identity on the init rows)
and the adjoint form is
    v' dw/dx0 = the init-row block of [y; mu] = K^-1 [v; 0]      (K symmetric).
"""
import ctypes
import os
import subprocess

import numpy as np

from feedback_jacobian_support import FIXTURES, oracle_nlp, relerr  # noqa: F401  (re-exported for the VJP tests)

_TWIN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "twin")
_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _kkt(nlp, pb, tab, x0, w, lam, phase):
    p0 = {"x0": np.asarray(x0, dtype=np.float64), "wref": tab.ref[phase], "H": tab.Href[phase], "q": tab.qref[phase]}
    _, Jg = nlp.g(w, p0, order=1)
    Hm = nlp.hess(w, p0, lam, "exact")
    lbg, ubg = pb.bounds()
    held = (lbg == ubg) | ((lam != 0) & np.isfinite(lbg))
    A = Jg[held]
    m = A.shape[0]
    K = np.block([[Hm, A.T], [A, np.zeros((m, m))]])
    init_pos = np.nonzero(held)[0]
    init = [pb.n_w + int(np.nonzero(init_pos == j)[0][0]) for j in range(pb.nx)]   # the init rows, all held
    return K, init


def dense_kkt_dw_dx0(nlp, pb, tab, x0, w, lam, phase=0):
    """the full dw/dx0 (n_w, nx) at (w, lam): one dense KKT solve with nx right-hand sides"""
    K, init = _kkt(nlp, pb, tab, x0, w, lam, phase)
    rhs = np.zeros((K.shape[0], pb.nx))
    for j, r in enumerate(init):
        rhs[r, j] = 1.0
    return np.linalg.solve(K, rhs)[:pb.n_w]


def dense_kkt_adjoint(nlp, pb, tab, x0, w, lam, v, phase=0):
    """v' dw/dx0 (nx,) by the adjoint form: the init-row block of K^-1 [v; 0]"""
    K, init = _kkt(nlp, pb, tab, x0, w, lam, phase)
    rhs = np.zeros(K.shape[0])
    rhs[:pb.n_w] = v
    return np.linalg.solve(K, rhs)[init]


def build_twin_vjp(name):
    """g++-compile tests/twin/twin_vjp.cpp into tests/twin/libtwin_vjp_<name>.so (flags of the CPU twin, twin/twin.py)"""
    out = os.path.join(_TWIN, "libtwin_vjp_%s.so" % name)
    srcs = [os.path.join(_TWIN, "twin_vjp.cpp")] + [os.path.join(_ROOT, "tunempc_b200", "csrc", f) for f in
                                                    ("tmpc_core.cuh", "tmpc_qp.cuh", "gen/model_%s.h" % name)]
    if os.path.exists(out) and all(os.path.getmtime(out) >= os.path.getmtime(s) for s in srcs):
        return out
    subprocess.check_call(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-w"] + os.environ.get("TWIN_CXXFLAGS", "").split() + [
                           "-I" + os.path.join(_ROOT, "tunempc_b200/csrc"), "-I" + os.path.join(_ROOT, "tunempc_b200/csrc/gen"),
                           '-DTMPC_MODEL_HEADER="model_%s.h"' % name, srcs[0], "-o", out])
    return out


def twin_solution_vjp(tw, out, v_u0=None, v_w=None, tol=None, phase=None):
    """(G (B, nx), jstatus (B,)) on the CPU twin (twin_vjp.cpp) at the solutions `out` (a dict with 'w', 'lam', 'status', e.g.
    the result of `tw.step(X0, tol=tol)`) of a twin.Twin `tw`: the stage records are linearised again at out['w'], out['lam'].
    tol: the step's tolerance (the weak-activity test reads it); phase: that step's phase (default: tw's last step)."""
    pb = tw.pb
    if v_u0 is None and v_w is None:
        raise ValueError("give v_u0, v_w or both")
    lib = ctypes.CDLL(build_twin_vjp(pb.name))
    dp, ip = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int)
    p = lambda a: a.ctypes.data_as(dp) if a is not None else None
    i = lambda a: a.ctypes.data_as(ip)
    economic = getattr(pb, "mpc_type", "tuned") == "economic"
    if pb.hessian_approximation != "exact" and not economic:
        raise ValueError("the solution VJP needs the exact Hessian")
    W = np.ascontiguousarray(out["w"], dtype=np.float64).reshape(-1, pb.n_w)
    LAM = np.ascontiguousarray(out["lam"], dtype=np.float64).reshape(-1, pb.n_g)
    st = np.ascontiguousarray(out["status"], dtype=np.int32).reshape(-1)
    B = W.shape[0]
    Vu = None if v_u0 is None else np.ascontiguousarray(v_u0, dtype=np.float64).reshape(B, pb.nu)
    Vw = None if v_w is None else np.ascontiguousarray(v_w, dtype=np.float64).reshape(B, pb.n_w)
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
    G = np.zeros((B, pb.nx)); jst = np.zeros(B, dtype=np.int32)
    ph = (tw.index - 1) % pb.p if phase is None else phase
    ret = lib.twin_solution_vjp(i(dims), i(iopts), p(dopts), p(wref), p(Hs), p(q), p(rdu), p(C), p(c), i(tidx), i(relax0),
                                ctypes.c_int(ph), ctypes.c_longlong(B), p(W), p(LAM), i(st), p(Vu), p(Vw), p(G), i(jst))
    if ret:
        raise RuntimeError("twin_solution_vjp returned %d" % ret)
    return G, jst
