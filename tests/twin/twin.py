"""ctypes wrapper of the CPU twin (tests/twin/twin.cpp) -- test infrastructure only."""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(os.path.dirname(_HERE))
_dp = ctypes.POINTER(ctypes.c_double)
_ip = ctypes.POINTER(ctypes.c_int)


def _p(a):
    return a.ctypes.data_as(_dp)


def _i(a):
    return a.ctypes.data_as(_ip)


def build(name, out_dir=None):
    """g++-compile libtwin_<name>.so into out_dir (default: next to this file)"""
    out = os.path.join(out_dir or _HERE, "libtwin_%s.so" % name)
    srcs = [os.path.join(_HERE, "twin.cpp"), os.path.join(_ROOT, "tunempc_b200/csrc/tmpc_core.cuh"),
            os.path.join(_ROOT, "tunempc_b200/csrc/tmpc_qp.cuh"),
            os.path.join(_ROOT, "tunempc_b200/csrc/gen/model_%s.h" % name)]
    if os.path.exists(out) and all(os.path.getmtime(out) >= os.path.getmtime(s) for s in srcs):
        return out
    subprocess.check_call(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-w"] + os.environ.get("TWIN_CXXFLAGS", "").split() + [
                           "-I" + os.path.join(_ROOT, "tunempc_b200/csrc"), "-I" + os.path.join(_ROOT, "tunempc_b200/csrc/gen"),
                           '-DTMPC_MODEL_HEADER="model_%s.h"' % name, srcs[0], "-o", out])
    return out


class Twin:
    def __init__(self, pb, tables, maxact=32, rho_rel=1e4, reg_mode=8, nonconvex_after=10, build_dir=None, **_ignored):
        self.pb, self.tab = pb, tables
        self.lib = ctypes.CDLL(build(pb.name, build_dir))
        self.maxact, self.rho_rel, self.reg_mode = maxact, rho_rel, int(os.environ.get("TWIN_REG_MODE", reg_mode))
        self.nonconvex_after = nonconvex_after
        self.reset(1)

    def reset(self, B):
        self.B = B
        self.index = 0
        self.W = np.tile(self.tab.ref[0], (B, 1))
        self.LAM = np.tile(self.tab.ref_du[0], (B, 1))

    def stage_eval(self, x, u, order):
        pb = self.pb
        x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1, pb.nx)
        u = np.ascontiguousarray(u, dtype=np.float64).reshape(-1, pb.nu)
        n = x.shape[0]
        nzm = pb.nx + pb.nu
        xf = np.zeros((n, pb.nx)); S = np.zeros((n, pb.nx, nzm)); T = np.zeros((n, pb.nx, nzm, nzm))
        self.lib.twin_stage_eval(n, _p(x), _p(u), order, _p(xf), _p(S), _p(T))
        return (xf, S, T)[: order + 1] if order else xf

    def lin_adjoint(self, x, u, lam, order=2):
        """record xf | S (nx x nz) | W packed of the forward / adjoint linearisation (tmpc_lin3.cuh); None for non-RK4 models"""
        pb = self.pb
        x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1, pb.nx)
        u = np.ascontiguousarray(u, dtype=np.float64).reshape(-1, pb.nu)
        lam = np.ascontiguousarray(lam, dtype=np.float64).reshape(-1, pb.nx)
        n = x.shape[0]
        nzm = pb.nx + pb.nu
        lsz = pb.nx + pb.nx * nzm + nzm * (nzm + 1) // 2
        rec = np.zeros((n, lsz))
        if self.lib.twin_lin_adjoint(n, _p(x), _p(u), _p(lam), order, _p(rec)):
            return None
        return rec

    def step(self, X0, hessian=None, tol=None, shared_first_qp=False):
        pb = self.pb
        X0 = np.ascontiguousarray(X0, dtype=np.float64).reshape(-1, pb.nx)
        B = X0.shape[0]
        assert B == self.B
        dims = np.array([pb.N, pb.nh, pb.nx_term, pb.p], dtype=np.int32)
        hm = pb.hessian_approximation if hessian is None else hessian
        iopts = np.array([1 if hm == "exact" else 0, pb.max_iter, 300, self.maxact,
                          1 if getattr(pb, "mpc_type", "tuned") == "economic" else 0, self.reg_mode, self.nonconvex_after], dtype=np.int32)
        dopts = np.array([pb.tol if tol is None else tol, 1e-8, 0.8, 1e-8, self.rho_rel], dtype=np.float64)
        wref_d, H_d, q_d = pb.device_tables()
        Hs = np.ascontiguousarray(0.5 * (H_d + np.transpose(H_d, (0, 2, 1))))
        relax0 = np.zeros(max(pb.nh, 1), dtype=np.int32)
        for i in pb.relax0:
            relax0[i] = 1
        tidx = np.array(pb.term_idx, dtype=np.int32)
        G = np.zeros((B, pb.n_g)); st = np.zeros(B, dtype=np.int32); it = np.zeros(B, dtype=np.int32)
        fl = np.zeros(B, dtype=np.int32); fv = np.zeros(B); nAS = np.zeros(B, dtype=np.int32)
        nACt = np.zeros(B, dtype=np.int32); nAC = np.zeros(B, dtype=np.int32)
        Wsh = np.zeros_like(self.W); Lsh = np.zeros_like(self.LAM)
        cnt = np.zeros(24, dtype=np.int64)
        C = np.ascontiguousarray(pb.C if pb.nh else np.zeros((1, pb.nz)))
        c = np.ascontiguousarray(pb.c if pb.nh else np.zeros(1))
        wref = np.ascontiguousarray(wref_d); q = np.ascontiguousarray(q_d); rdu = np.ascontiguousarray(self.tab.ref_du)
        ret = self.lib.twin_step(_i(dims), _i(iopts), _p(dopts), _p(wref), _p(Hs), _p(q), _p(rdu), _p(C), _p(c),
                                 _i(tidx), _i(relax0), ctypes.c_int(self.index % pb.p), ctypes.c_longlong(B), _p(X0),
                                 _p(self.W), _p(self.LAM), _p(G), _i(st), _i(it), _i(fl), _p(fv), _i(nAS), _i(nACt),
                                 _i(nAC), _p(Wsh), _p(Lsh), cnt.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong)),
                                 ctypes.c_int(1 if (shared_first_qp and self.index == 0) else 0))
        if ret:
            raise RuntimeError("twin_step returned %d" % ret)
        out = dict(w=self.W.copy(), lam=self.LAM.copy(), g=G, status=st, iter=it, flags=fl, f=fv, nAS=nAS,
                   nACtot=nACt, nAC=nAC, u0=self.W[:, pb.nx:pb.nx + pb.nu].copy(), counters=cnt)
        self.W, self.LAM = Wsh, Lsh
        self.index += 1
        return out
