"""ctypes binding of the C ABI (include/tmpc.h) -- one shared library per compiled model.

Mirrors how the reference binds its only native solver: `ctypes.CDLL` on a per-model shared library and an opaque
capsule pointer (external/acados/interfaces/acados_template/acados_template/acados_ocp_solver.py:752-801).
There is no CPU fallback: if the library or a CUDA device is missing, construction raises.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)
_dp = ctypes.POINTER(ctypes.c_double)
_ip = ctypes.POINTER(ctypes.c_int32)

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-shared", "-Xcompiler", "-fPIC",
              "-std=c++17", "--threads", "4"]      # the four translation units of a model library compile side by side

EXPORTS = ["tmpc_default_opts", "tmpc_model_info", "tmpc_model_slacks", "tmpc_create", "tmpc_destroy", "tmpc_last_error",
           "tmpc_set_tables", "tmpc_reset", "tmpc_get_index", "tmpc_step", "tmpc_step_async", "tmpc_wait", "tmpc_busy", "tmpc_step_host", "tmpc_feedback_jacobian", "tmpc_solution_vjp", "tmpc_plant_step", "tmpc_plant_jacobian", "tmpc_stage_log",
           "tmpc_get_log", "tmpc_get_counters", "tmpc_get_timing", "tmpc_stage_eval_host", "tmpc_fp64_peak"]


class TmpcDims(ctypes.Structure):
    _fields_ = [("nx", ctypes.c_int32), ("nu", ctypes.c_int32), ("nh", ctypes.c_int32), ("nx_term", ctypes.c_int32),
                ("N", ctypes.c_int32), ("p", ctypes.c_int32), ("ns", ctypes.c_int32), ("nsc", ctypes.c_int32)]


class TmpcOpts(ctypes.Structure):
    _fields_ = [("hessian_exact", ctypes.c_int32), ("max_iter", ctypes.c_int32), ("max_ls_iter", ctypes.c_int32),
                ("tol", ctypes.c_double), ("lam_tresh", ctypes.c_double), ("ls_step_factor", ctypes.c_double),
                ("reg_tol", ctypes.c_double), ("term_weight", ctypes.c_double), ("max_working_set", ctypes.c_int32),
                ("economic", ctypes.c_int32)]


def lib_path(name):
    return os.path.join(_PKG, "libtmpc_%s.so" % name)


def build_model_lib(name, force=False, verbose=False):
    """nvcc-compile libtmpc_<name>.so in-tree for sm_100a (cross-compiles without a GPU)."""
    out = lib_path(name)
    srcs = [os.path.join(_PKG, "csrc", "tmpc.cu"), os.path.join(_PKG, "csrc", "tmpc_qp_thread.cu"),
            os.path.join(_PKG, "csrc", "tmpc_fbjac_thread.cu"), os.path.join(_PKG, "csrc", "tmpc_vjp_thread.cu"),
            os.path.join(_PKG, "csrc", "tmpc_qp_thread.cuh"),
            os.path.join(_PKG, "csrc", "tmpc_core.cuh"), os.path.join(_PKG, "csrc", "tmpc_lin2.cuh"),
            os.path.join(_PKG, "csrc", "tmpc_qp.cuh"), os.path.join(_PKG, "csrc", "tmpc_lin3.cuh"),
            os.path.join(_PKG, "csrc", "gen", "model_%s.h" % name), os.path.join(_ROOT, "include", "tmpc.h")]
    if not force and os.path.exists(out) and all(os.path.getmtime(out) >= os.path.getmtime(s) for s in srcs):
        return out
    cmd = ["nvcc"] + NVCC_FLAGS + ['-DTMPC_MODEL_HEADER="gen/model_%s.h"' % name, "-I" + os.path.join(_ROOT, "include"),
                                  "-I" + os.path.join(_PKG, "csrc"), srcs[0], srcs[1], srcs[2], srcs[3], "-o", out]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    subprocess.check_call(cmd)
    return out


class ModelLib:
    """loaded libtmpc_<name>.so with typed entry points"""

    def __init__(self, name):
        path = lib_path(name)
        if not os.path.exists(path):
            raise RuntimeError("CUDA library %s is missing -- run __graft_entry__.build() (there is no CPU fallback)" % path)
        self.name = name
        self.path = path
        L = self.lib = ctypes.CDLL(path)
        vp = ctypes.c_void_p
        L.tmpc_default_opts.argtypes = [ctypes.POINTER(TmpcOpts)]
        L.tmpc_model_info.restype = ctypes.c_char_p
        L.tmpc_model_info.argtypes = [_ip, _ip, _ip, _dp]
        L.tmpc_create.argtypes = [ctypes.POINTER(vp), ctypes.POINTER(TmpcDims), ctypes.POINTER(TmpcOpts), ctypes.c_int]
        L.tmpc_destroy.argtypes = [vp]
        L.tmpc_destroy.restype = None
        L.tmpc_last_error.argtypes = [vp]
        L.tmpc_last_error.restype = ctypes.c_char_p
        L.tmpc_set_tables.argtypes = [vp, _dp, _dp, _dp, _dp, _dp, _dp, _ip, _ip]
        L.tmpc_reset.argtypes = [vp, ctypes.c_int64]
        L.tmpc_get_index.argtypes = [vp, ctypes.POINTER(ctypes.c_int64)]
        L.tmpc_step.argtypes = [vp, vp, ctypes.c_int64, vp, vp, vp, vp, vp, vp, vp, vp]
        L.tmpc_step_async.argtypes = [vp, vp, ctypes.c_int64, vp, vp, vp, vp, vp, vp, vp, vp]
        L.tmpc_wait.argtypes = [vp]
        L.tmpc_busy.argtypes = [vp, _ip]
        L.tmpc_step_host.argtypes = [vp, vp, ctypes.c_int64, vp, vp, vp, vp, vp, vp, vp]
        L.tmpc_feedback_jacobian.argtypes = [vp, vp, vp, ctypes.c_int, vp]
        L.tmpc_solution_vjp.argtypes = [vp, ctypes.c_int64, vp, vp, vp, ctypes.c_int32, vp, vp, vp, vp, ctypes.c_int, vp]
        L.tmpc_plant_step.argtypes = [vp, vp, vp, ctypes.c_int64, vp, vp]
        L.tmpc_plant_jacobian.argtypes = [vp, vp, vp, ctypes.c_int64, vp, vp]
        L.tmpc_stage_log.argtypes = [vp, vp, vp, ctypes.c_int64, vp, vp, vp]
        L.tmpc_get_log.argtypes = [vp, vp, vp, vp, vp, ctypes.c_int]
        L.tmpc_get_counters.argtypes = [vp, ctypes.POINTER(ctypes.c_int64)]
        L.tmpc_get_timing.argtypes = [vp, _dp]
        L.tmpc_stage_eval_host.argtypes = [ctypes.c_int32, _dp, _dp, ctypes.c_int32, _dp, _dp, _dp]
        L.tmpc_fp64_peak.argtypes = [vp, _dp]
        nx, nu, st = ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int32()
        dt = ctypes.c_double()
        self.model_name = L.tmpc_model_info(ctypes.byref(nx), ctypes.byref(nu), ctypes.byref(st), ctypes.byref(dt)).decode()
        self.nx, self.nu, self.nz = nx.value, nu.value, nx.value + nu.value       # model dimensions (x, u)
        self.rk_steps, self.dt = st.value, dt.value
        ns, nsc = ctypes.c_int32(), ctypes.c_int32()
        L.tmpc_model_slacks.argtypes = [_ip, _ip]
        L.tmpc_model_slacks.restype = None
        L.tmpc_model_slacks(ctypes.byref(ns), ctypes.byref(nsc))
        self.ns, self.nsc = ns.value, nsc.value

    def default_opts(self):
        o = TmpcOpts()
        self.lib.tmpc_default_opts(ctypes.byref(o))
        return o

    def stage_eval(self, xs, us, order=0):
        """host evaluation of the generated model's interval map (offline tuning only)"""
        xs = np.ascontiguousarray(xs, dtype=np.float64).reshape(-1, self.nx)
        us = np.ascontiguousarray(us, dtype=np.float64).reshape(-1, self.nu)
        n = xs.shape[0]
        xf = np.zeros((n, self.nx))
        S = np.zeros((n, self.nx, self.nz))
        T = np.zeros((n, self.nx, self.nz, self.nz))
        p = lambda a: a.ctypes.data_as(_dp)
        self.lib.tmpc_stage_eval_host(n, p(xs), p(us), order, p(xf), p(S), p(T))
        return (xf, S, T)[: order + 1] if order else xf
