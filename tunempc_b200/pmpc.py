"""Batched drop-in for the reference controller object `tunempc.pmpc.Pmpc` (tracking / tuned type).

Same surface as the reference (`tunempc/pmpc.py`): constructor options and their defaults (:149-160, unknown key ->
ValueError :89-94), `step(x0) -> u0` (:371-423), `reset()` (:858-865), properties `w_sol, g_sol, log, index`
(:1120-1142).  New: `step(X0)` with `X0` of shape (B, nx) solves B independent instances in one call -- a
`torch.float64` CUDA tensor stays on the device (zero-copy through the C ABI), a numpy array goes through the
host entry point `tmpc_step_host`.  All arithmetic happens in libtmpc_<model>.so (CUDA, sm_100a); this module only
marshals pointers.  No CPU fallback: construction raises if the library or the GPU is missing.
"""
from __future__ import annotations

import copy
import ctypes

import numpy as np

from .lib import ModelLib, TmpcDims, _dp, _ip
from .problem import MpcProblem, build_tables

STATUS_NAMES = {0: "Solve_Succeeded", 1: "Maximum_Iterations_Exceeded", 2: "QP_Infeasible",
                3: "Reduced_Hessian_Not_PD", 4: "NaN_Detected", 5: "Working_Set_Overflow"}

_LOG_KEYS = ("cpu", "iter", "f", "status", "sol_x", "lam_x", "lam_g", "u0", "nACtot", "nAC", "idx_AC", "nAS", "flags")


def default_options():
    """tunempc/pmpc.py:149-160 (p_operator is given as the list of selected state indices; None = identity)"""
    return {"hessian_approximation": "exact", "ipopt_presolve": False, "max_iter": 2000, "p_operator": None,
            "slack_flag": "none"}


def problem_from_reference_args(N, sys, cost, wref, tuning, lam_g_ref, sensitivities, options):
    """The reference constructor's arguments (tunempc/pmpc.py:39-147) -> the problem IR.

    sys            model card: {'f': OdeModel or compiled-model name, 'vars': {'x': .., 'u': .. [, 'us': .., 'usc': ..]},
                   'h': (C, c) with h = C z + c >= 0 over z = (x, u, us, usc) [, 'g': the compiled model's nonlinear rows
                   h_nl(x,u) - us = 0, 'scost': (nsc,), 'gnl_x_idx': state-only rows of g]} -- what Tuner.sys returns after
                   preprocessing (tuner.py:201-207, preprocessing.py:35-155 hand CasADi Functions here)
    cost           'tracking' / 'economic', or a callable: two arguments l(x,u) -> economic, otherwise tracking
                   (the reference tells them apart by cost.n_in(), pmpc.py:97-118)
    wref           {'x': [p arrays (nx,)], 'u': [p arrays (nu,)]} or an array (p, nz)   (pmpc.py:692-706)
    tuning         {'H': [p (nz,nz)], 'q': [p (nz,)]}; required for tracking MPC (pmpc.py:117-118), ignored for economic
    lam_g_ref      {'dyn': [p (nx,)], 'h': [p (nh,)]}   (pmpc.py:709-720)
    sensitivities  {'A': [p (nx,nx)], 'B': [p (nx,nu)]}: only read when the terminal constraint is projected (pmpc.py:724-767)
    """
    import inspect
    f = sys["f"]
    name = f if isinstance(f, str) else f.name
    nx, nu = len(sys["vars"]["x"]), len(sys["vars"]["u"])
    ns = len(sys["vars"]["us"]) if "us" in sys["vars"] else 0                                # pmpc.py:50-55
    nsc = len(sys["vars"]["usc"]) if "usc" in sys["vars"] else 0                             # pmpc.py:57-62
    scost = np.asarray(sys["scost"], dtype=np.float64).ravel() if nsc else None
    if (ns > 0) != ("g" in sys):
        raise ValueError("slacks us and the nonlinear rows g come together (tunempc/preprocessing.py:78-118)")
    # state-only nonlinear constraints (pmpc.py:1107-1114): from the model card's expressions, or given explicitly
    gnl_x_idx = list(sys.get("gnl_x_idx", []))
    if ns and not isinstance(f, str) and "gnl_x_idx" not in sys:
        usym = set(f.u)
        gnl_x_idx = [i for i, e in enumerate(f.gnl) if not (set(getattr(e, "free_symbols", ())) & usym)]
    nzr, nz = nx + nu + ns, nx + nu + ns + nsc
    if isinstance(cost, str):
        economic = cost == "economic"
    else:
        economic = callable(cost) and len(inspect.signature(cost).parameters) == 2          # pmpc.py:97
    assert wref is not None, "Provide reference trajectory!"                                 # pmpc.py:134
    if isinstance(wref, dict):
        w = np.array([np.concatenate([np.ravel(wref["x"][k]), np.ravel(wref["u"][k])] + ([np.ravel(wref["us"][k])] if ns else []))
                      for k in range(len(wref["u"]))])                                         # pmpc.py:692-704
    else:
        w = np.atleast_2d(np.asarray(wref, dtype=np.float64))
    P = w.shape[0]
    if economic:
        # pmpc.py:103: no tuning required.  With slacks the stage cost is l(x,u) + scost'usc (pmpc.py:299-301,338-339): H and
        # q stay zero on (x,u,us) and device_tables() puts scost into the usc entries of q
        H, q = np.zeros((P, nzr, nzr)), np.zeros((P, nzr))
    else:
        assert tuning is not None, "Provide tuning matrices for tracking MPC!"                # pmpc.py:118
        Hs = [np.asarray(h, dtype=np.float64) for h in tuning["H"]]
        qs = [np.asarray(v, dtype=np.float64).ravel() for v in tuning["q"]]
        H = np.array(Hs * P if len(Hs) == 1 and P > 1 else Hs)
        q = np.array(qs * P if len(qs) == 1 and P > 1 else qs)
    C, c = sys.get("h", (np.zeros((0, nz)), np.zeros(0)))
    C, c = np.asarray(C, dtype=np.float64).reshape(-1, nz), np.asarray(c, dtype=np.float64).ravel()
    nh = C.shape[0]
    lam_dyn = (np.zeros((P, nx)) if lam_g_ref is None
               else np.array([np.ravel(v) for v in lam_g_ref["dyn"]], dtype=np.float64).reshape(P, nx))
    lam_h = (np.zeros((P, nh - nsc)) if lam_g_ref is None or "h" not in lam_g_ref                # the usc >= 0 rows get -scost (pmpc.py:716-720)
             else np.array([np.ravel(v) for v in lam_g_ref["h"]], dtype=np.float64).reshape(P, nh - nsc))
    lam_g = None
    if ns:
        lam_g = (np.zeros((P, ns)) if lam_g_ref is None or "g" not in lam_g_ref
                 else np.array([np.ravel(v) for v in lam_g_ref["g"]], dtype=np.float64).reshape(P, ns))
    term = (options or {}).get("p_operator")
    pb = MpcProblem(name=name, nx=nx, nu=nu, N=int(N), p=P, wref=w, H=H, q=q, C=C, c=c, lam_h_ref=lam_h, lam_dyn_ref=lam_dyn,
                    term_idx=list(range(nx)) if term is None else [int(i) for i in term],
                    S_A=None if sensitivities is None else np.array(sensitivities["A"], dtype=np.float64),
                    S_B=None if sensitivities is None else np.array(sensitivities["B"], dtype=np.float64),
                    mpc_type="economic" if economic else "tuned", ns=ns, nsc=nsc, scost=scost, lam_g_ref=lam_g,
                    gnl_x_idx=[int(i) for i in gnl_x_idx])
    if economic:
        pb.hessian_approximation = "exact"                                                     # pmpc.py:105-107
    return pb


class Pmpc:
    def __init__(self, N=None, sys=None, cost=None, wref=None, tuning=None, lam_g_ref=None, sensitivities=None, options=None,
                 device=0, solver_options=None, problem: MpcProblem = None):
        """Two ways in: the reference's own signature `Pmpc(N, sys, cost, wref, tuning, lam_g_ref, sensitivities, options)`
        (tunempc/pmpc.py:39) with `sys` a model card, or the problem IR `Pmpc(problem, options)` /
        `Pmpc(problem=problem)` (an `MpcProblem`, e.g. loaded from a fixture).  `device`: CUDA device index."""
        if isinstance(N, MpcProblem):                                    # Pmpc(problem[, options])
            problem, N = N, None
            if isinstance(sys, dict) and options is None:
                options, sys = sys, None
        if problem is None:
            problem = problem_from_reference_args(N, sys, cost, wref, tuning, lam_g_ref, sensitivities, options)
        opts = default_options()
        for k, v in (options or {}).items():
            if k in opts:
                opts[k] = v
            else:
                raise ValueError('Unknown option for Pmpc class instance: "{}"'.format(k))   # pmpc.py:94
        if opts["ipopt_presolve"]:
            raise NotImplementedError("ipopt_presolve is a host-side IPOPT call in the reference (pmpc.py:394-404); not available")
        # opts['slack_flag'] is consumed by Tuner.create_mpc, which softens the rows before this constructor runs
        # (tuner.py:171-177, preprocessing.py:120-155); here the softened rows arrive in sys['h'] / sys['vars']['usc'] / sys['scost']
        problem = copy.copy(problem)                                     # the caller's problem object is never modified
        if options and "hessian_approximation" in options:
            problem.hessian_approximation = opts["hessian_approximation"]
        if options and "max_iter" in options:
            problem.max_iter = int(opts["max_iter"])
        if opts["p_operator"] is not None:
            problem.term_idx = [int(i) for i in opts["p_operator"]]
        if problem.hessian_approximation not in ("exact", "gauss_newton"):
            raise ValueError("hessian_approximation must be 'exact' or 'gauss_newton'")
        self.__options = opts
        self.__pb = problem
        self.__tab = build_tables(problem)
        self.__lib = ModelLib(problem.name)
        L = self.__lib.lib
        if (self.__lib.nx, self.__lib.nu, self.__lib.ns, self.__lib.nsc) != (problem.nx, problem.nu, problem.ns, problem.nsc):
            raise ValueError("problem dimensions do not match compiled model '%s'" % problem.name)
        dims = TmpcDims(problem.nx, problem.nu, problem.nh, problem.nx_term, problem.N, problem.p, problem.ns, problem.nsc)
        o = self.__lib.default_opts()
        o.hessian_exact = 1 if problem.hessian_approximation == "exact" else 0
        o.economic = 1 if problem.mpc_type == "economic" else 0          # pmpc.py:97-107: exact Hessian forced
        o.max_iter = int(problem.max_iter)
        o.tol = float(problem.tol)
        for k, v in (solver_options or {}).items():
            if not hasattr(o, k):
                raise ValueError('Unknown solver option "{}"'.format(k))
            setattr(o, k, v)
        self.__h = ctypes.c_void_p()
        rc = L.tmpc_create(ctypes.byref(self.__h), ctypes.byref(dims), ctypes.byref(o), int(device))
        if rc != 0:
            raise RuntimeError("tmpc_create failed with code %d (no usable CUDA device? there is no CPU fallback)" % rc)
        self.__device = int(device)
        pb = problem
        relax0 = np.zeros(max(pb.nh, 1), dtype=np.int32)
        for i in pb.relax0:                                               # pmpc.py:293-294: h_us_idx + h_x_idx
            relax0[i] = 1
        tidx = np.ascontiguousarray(np.array(pb.term_idx, dtype=np.int32))
        C = np.ascontiguousarray(pb.C if pb.nh else np.zeros((1, pb.nz)), dtype=np.float64)
        c = np.ascontiguousarray(pb.c if pb.nh else np.zeros(1), dtype=np.float64)
        arrs = [np.ascontiguousarray(a, dtype=np.float64) for a in pb.device_tables() + (self.__tab.ref_du,)]
        p = lambda a: a.ctypes.data_as(_dp)
        self.__check(L.tmpc_set_tables(self.__h, p(arrs[0]), p(arrs[1]), p(arrs[2]), p(arrs[3]), p(C), p(c),
                                       tidx.ctypes.data_as(_ip), relax0.ctypes.data_as(_ip)))
        self.__B = 0
        self.__index = 0
        self.__out = None
        self.__pending = None
        self.__initialize_log()

    # ---- plumbing ------------------------------------------------------------------------------------
    def __check(self, rc):
        if rc != 0:
            raise RuntimeError("libtmpc: " + self.__lib.lib.tmpc_last_error(self.__h).decode())

    def __del__(self):
        try:
            if self.__h:
                self.__lib.lib.tmpc_destroy(self.__h)
                self.__h = None
        except Exception:
            pass

    def __initialize_log(self):                                       # pmpc.py:785-800
        self.__log = {k: [] for k in _LOG_KEYS}

    def reset(self, B=None):
        """pmpc.py:858-865: phase index <- 0, log cleared, warm start <- reference (for B instances)."""
        if getattr(self, "_Pmpc__pending", None) is not None:
            raise RuntimeError("reset: a step started by step_async is still in flight (call wait() first)")
        if B is not None:
            self.__B = int(B)
        self.__index = 0
        self.__initialize_log()
        self.__check(self.__lib.lib.tmpc_reset(self.__h, self.__B))

    def __ensure_batch(self, B):
        if B != self.__B:
            if self.__index != 0 and self.__B != 0:
                raise ValueError("batch size changed from %d to %d without reset()" % (self.__B, B))
            self.__B = B
            self.__index = 0                                              # tmpc_reset zeroes the device phase index too
            self.__check(self.__lib.lib.tmpc_reset(self.__h, B))

    # ---- the hot path --------------------------------------------------------------------------------
    def step(self, x0, outputs="all"):
        """One MPC feedback solve per row of x0 (pmpc.py:371-423).

        x0: (nx,), (nx,1) [reference semantics, returns (nu,) / (nu,1)], numpy (B,nx) -> numpy (B,nu), or a
        torch.float64 CUDA tensor (B,nx) -> torch CUDA tensor (B,nu).  outputs='u0' skips the (B,n_w)/(B,n_g)
        solution tensors."""
        pb = self.__pb
        L = self.__lib.lib
        if getattr(self, "_Pmpc__pending", None) is not None:
            raise RuntimeError("step: a step started by step_async is still in flight (call wait() first)")
        is_torch = type(x0).__module__.startswith("torch")
        if is_torch:
            import torch
            if x0.dtype != torch.float64 or not x0.is_cuda:
                raise TypeError("torch input must be a float64 CUDA tensor")
            if x0.dim() != 2 or x0.shape[1] != pb.nx:
                raise ValueError("expected X0 of shape (B, %d)" % pb.nx)
            if x0.device.index != self.__device:
                raise ValueError("X0 is on cuda:%s, controller on cuda:%d" % (x0.device.index, self.__device))
            X0 = x0.contiguous()
            B = X0.shape[0]
            self.__ensure_batch(B)
            phase = self.__index % pb.p
            dev = X0.device
            full = outputs == "all"
            U0 = torch.empty((B, pb.nu), dtype=torch.float64, device=dev)
            W = torch.empty((B, pb.n_w), dtype=torch.float64, device=dev) if full else None
            LAM = torch.empty((B, pb.n_g), dtype=torch.float64, device=dev) if full else None
            G = torch.empty((B, pb.n_g), dtype=torch.float64, device=dev) if full else None
            st = torch.empty(B, dtype=torch.int32, device=dev)
            it = torch.empty(B, dtype=torch.int32, device=dev)
            fl = torch.empty(B, dtype=torch.int32, device=dev)
            ptr = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
            stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            self.__check(L.tmpc_step(self.__h, ptr(X0), B, ptr(U0), ptr(W), ptr(LAM), ptr(G), ptr(st), ptr(it), ptr(fl),
                                     stream))
            self.__out = dict(u0=U0, w=W, lam_g=LAM, g=G, status=st, iter=it, flags=fl, phase=phase)
            self.__log_append(torch_dev=dev)
            self.__index += 1
            return U0
        a = np.asarray(x0, dtype=np.float64)
        single_shape = None
        if a.ndim == 1 or (a.ndim == 2 and a.shape[1] == 1 and a.shape[0] == pb.nx):
            single_shape = a.shape
            a = a.reshape(1, pb.nx)
        if a.ndim != 2 or a.shape[1] != pb.nx:
            raise ValueError("expected x0 of shape (%d,), (%d,1) or (B,%d)" % (pb.nx, pb.nx, pb.nx))
        X0 = np.ascontiguousarray(a)
        B = X0.shape[0]
        self.__ensure_batch(B)
        phase = self.__index % pb.p
        full = outputs == "all"
        U0 = np.empty((B, pb.nu))
        W = np.empty((B, pb.n_w)) if full else None
        LAM = np.empty((B, pb.n_g)) if full else None
        G = np.empty((B, pb.n_g)) if full else None
        st = np.empty(B, dtype=np.int32)
        it = np.empty(B, dtype=np.int32)
        fl = np.empty(B, dtype=np.int32)
        vp = lambda t: ctypes.c_void_p(t.ctypes.data) if t is not None else None
        self.__check(L.tmpc_step_host(self.__h, vp(X0), B, vp(U0), vp(W), vp(LAM), vp(G), vp(st), vp(it), vp(fl)))
        self.__out = dict(u0=U0, w=W, lam_g=LAM, g=G, status=st, iter=it, flags=fl, single=single_shape is not None,
                          phase=phase)
        self.__log_append()
        self.__index += 1
        if single_shape is not None:
            return U0[0].reshape((pb.nu, 1) if len(single_shape) == 2 else (pb.nu,)).copy()
        return U0

    def step_async(self, X0, outputs="u0"):
        """`step(X0)` as a non-blocking call (C ABI: tmpc_step_async): returns the output tensor U0 (B,nu) at once while a
        worker thread of the library drives the solve; what was enqueued on the current CUDA stream before the call (the
        producer of X0) is waited for on the device.  `wait()` blocks the host until the solve has finished, appends the log and
        returns U0 -- only then may U0 be read.  One step in flight per controller: call `wait()` before the next
        `step` / `step_async` / `reset`."""
        import torch
        pb = self.__pb
        if getattr(self, "_Pmpc__pending", None) is not None:
            raise RuntimeError("step_async: a step is still in flight (call wait() first)")
        if not (type(X0).__module__.startswith("torch") and X0.is_cuda and X0.dtype == torch.float64):
            raise TypeError("step_async takes a float64 CUDA tensor (B, nx)")
        if X0.dim() != 2 or X0.shape[1] != pb.nx:
            raise ValueError("expected X0 of shape (B, %d)" % pb.nx)
        X0 = X0.contiguous()
        B = X0.shape[0]
        self.__ensure_batch(B)
        phase = self.__index % pb.p
        dev = X0.device
        full = outputs == "all"
        U0 = torch.empty((B, pb.nu), dtype=torch.float64, device=dev)
        W = torch.empty((B, pb.n_w), dtype=torch.float64, device=dev) if full else None
        LAM = torch.empty((B, pb.n_g), dtype=torch.float64, device=dev) if full else None
        G = torch.empty((B, pb.n_g), dtype=torch.float64, device=dev) if full else None
        st = torch.empty(B, dtype=torch.int32, device=dev)
        it = torch.empty(B, dtype=torch.int32, device=dev)
        fl = torch.empty(B, dtype=torch.int32, device=dev)
        ptr = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        self.__check(self.__lib.lib.tmpc_step_async(self.__h, ptr(X0), B, ptr(U0), ptr(W), ptr(LAM), ptr(G), ptr(st), ptr(it),
                                                    ptr(fl), stream))
        self.__pending = dict(out=dict(u0=U0, w=W, lam_g=LAM, g=G, status=st, iter=it, flags=fl, phase=phase), dev=dev, keep=X0)
        return U0

    def busy(self):
        b = ctypes.c_int32()
        self.__check(self.__lib.lib.tmpc_busy(self.__h, ctypes.byref(b)))
        return bool(b.value)

    def wait(self):
        """block the host until the step started by `step_async` has finished; returns its U0"""
        pend = getattr(self, "_Pmpc__pending", None)
        if pend is None:
            return self.__out["u0"] if self.__out else None
        rc = self.__lib.lib.tmpc_wait(self.__h)
        self.__pending = None
        self.__check(rc)
        self.__out = pend["out"]
        self.__log_append(torch_dev=pend["dev"])
        self.__index += 1
        return self.__out["u0"]

    def __log_append(self, torch_dev=None):                           # pmpc.py:815-831
        o = self.__out
        lg = self.__log
        if self.__B == 0:                                             # empty batch: nothing ran on the device
            for k in _LOG_KEYS:
                lg[k].append(o.get({"sol_x": "w"}.get(k, k)))
            return
        lg["cpu"].append(self.timing()["step_ms"] * 1e-3)
        lg["iter"].append(o["iter"])
        lg["status"].append(o["status"])
        lg["sol_x"].append(o["w"])
        lg["lam_g"].append(o["lam_g"])
        lg["u0"].append(o["u0"])
        lg["flags"].append(o["flags"])
        f, nAS, nACt, nAC = self.__fetch_log(torch_dev)
        lg["f"].append(f)
        lg["nAS"].append(nAS)
        lg["nACtot"].append(nACt)
        lg["nAC"].append(nAC)
        lg["idx_AC"].append(nAC)                                      # the reference stores nAC here too (pmpc.py:828)

    def __fetch_log(self, torch_dev):
        L = self.__lib.lib
        B = self.__B
        if torch_dev is not None:
            import torch
            outs = [torch.empty(B, dtype=dt, device=torch_dev) for dt in (torch.float64, torch.int32, torch.int32, torch.int32)]
            self.__check(L.tmpc_get_log(self.__h, *[ctypes.c_void_p(t.data_ptr()) for t in outs], 0))
            return outs
        outs = [np.empty(B, dtype=dt) for dt in (np.float64, np.int32, np.int32, np.int32)]
        self.__check(L.tmpc_get_log(self.__h, *[ctypes.c_void_p(t.ctypes.data) for t in outs], 1))
        return outs

    def feedback_jacobian(self):
        """Feedback Jacobian du0/dx0 of the solutions of the last step (C ABI: tmpc_feedback_jacobian, definition in
        include/tmpc.h): (J, jstatus) with J (B, nu, nx), J[b, i, j] = d u0_i / d x0_j, and jstatus (B,) int32 -- 0 ok, 1 a weakly
        active row (the solution map has a kink; J holds the active set), 2 the step did not converge, 3 singular (J is NaN for
        2 and 3).  torch CUDA tensors after a torch step, numpy arrays after a numpy step, ((nu, nx), int) after a single-state
        step.  Needs the exact Hessian; leaves the warm start, the phase index and the log unchanged."""
        if getattr(self, "_Pmpc__pending", None) is not None:
            raise RuntimeError("feedback_jacobian: a step started by step_async is still in flight (call wait() first)")
        pb = self.__pb
        L = self.__lib.lib
        B = self.__B
        o = self.__out
        if o is not None and type(o["u0"]).__module__.startswith("torch"):
            import torch
            dev = o["u0"].device
            J = torch.empty((B, pb.nu, pb.nx), dtype=torch.float64, device=dev)
            js = torch.empty(B, dtype=torch.int32, device=dev)
            stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            self.__check(L.tmpc_feedback_jacobian(self.__h, ctypes.c_void_p(J.data_ptr()), ctypes.c_void_p(js.data_ptr()), 0,
                                                  stream))
            return J, js
        J = np.empty((B, pb.nu, pb.nx))
        js = np.empty(B, dtype=np.int32)
        self.__check(L.tmpc_feedback_jacobian(self.__h, ctypes.c_void_p(J.ctypes.data), ctypes.c_void_p(js.ctypes.data), 1,
                                              None))
        if o is not None and o.get("single"):
            return J[0].copy(), int(js[0])
        return J, js

    def solution_vjp(self, v_u0=None, v_w=None, w=None, lam_g=None, status=None, phase=None):
        """Vector-Jacobian product of the solution map (C ABI: tmpc_solution_vjp, definition in include/tmpc.h): (G, jstatus) with
        G (B, nx), G[b] = v_u0[b]' du0/dx0 + v_w[b]' dw/dx0, and jstatus (B,) int32 as in feedback_jacobian() (G is NaN for 2
        and 3).  One QP solve per instance whatever nx, for both cotangents together.
        v_u0 (B, nu), v_w (B, n_w): the cotangents; either may be None, not both.
        w, lam_g, status, phase: a solution as a step returned it (w_sol, lam_g, status, last_phase of that step), which may be
        several steps old; phase defaults to the last step's.  w=None: the last step's own solutions (lam_g, status and phase must
        then be None).  torch CUDA tensors for torch inputs (and after a torch step with w=None), numpy arrays otherwise;
        ((nx,), int) after a single-state step with w=None.  Needs the exact Hessian; changes nothing in the controller."""
        if getattr(self, "_Pmpc__pending", None) is not None:
            raise RuntimeError("solution_vjp: a step started by step_async is still in flight (call wait() first)")
        pb = self.__pb
        L = self.__lib.lib
        o = self.__out
        if w is None:
            if lam_g is not None or status is not None or phase is not None:
                raise ValueError("solution_vjp: lam_g, status and phase go with w")
            B, ph = self.__B, 0
            is_torch = (o is not None and type(o["u0"]).__module__.startswith("torch")) or any(
                type(v).__module__.startswith("torch") for v in (v_u0, v_w))
        else:
            if lam_g is None or status is None:
                raise ValueError("solution_vjp: w needs lam_g and status")
            ph = int(phase) if phase is not None else (o["phase"] if o is not None else 0)
            is_torch = type(w).__module__.startswith("torch")
            B = int(w.shape[0])
        if is_torch:
            import torch
            dev = torch.device("cuda", self.__device)
            f64 = lambda t: None if t is None else torch.as_tensor(t, dtype=torch.float64, device=dev).contiguous()
            i32 = lambda t: None if t is None else torch.as_tensor(t, dtype=torch.int32, device=dev).contiguous()
            args = [f64(w), f64(lam_g), i32(status), f64(v_u0), f64(v_w)]
            G = torch.empty((B, pb.nx), dtype=torch.float64, device=dev)
            js = torch.empty(B, dtype=torch.int32, device=dev)
            ptr = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
            stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            is_host = 0
        else:
            f64 = lambda t: None if t is None else np.ascontiguousarray(t, dtype=np.float64)
            i32 = lambda t: None if t is None else np.ascontiguousarray(t, dtype=np.int32)
            args = [f64(w), f64(lam_g), i32(status), f64(v_u0), f64(v_w)]
            G = np.empty((B, pb.nx))
            js = np.empty(B, dtype=np.int32)
            ptr = lambda t: ctypes.c_void_p(t.ctypes.data) if t is not None else None
            stream = None
            is_host = 1
        for a, n, name in zip(args, (pb.n_w, pb.n_g, 1, pb.nu, pb.n_w), ("w", "lam_g", "status", "v_u0", "v_w")):
            size = None if a is None else (a.numel() if is_torch else a.size)
            if size is not None and size != B * n and not (w is None and o is None):   # no step yet: the library reports it
                raise ValueError("solution_vjp: %s has %d elements, expected %d x %d" % (name, size, B, n))
        W, LAM, st, Vu, Vw = args
        self.__check(L.tmpc_solution_vjp(self.__h, B, ptr(W), ptr(LAM), ptr(st), ph, ptr(Vu), ptr(Vw), ptr(G), ptr(js), is_host,
                                         stream))
        if w is None and not is_torch and o is not None and o.get("single"):
            return G[0].copy(), int(js[0])
        return G, js

    # ---- closed loop helpers -------------------------------------------------------------------------
    def plant_step(self, X, U):
        """x+ = F(x,u) for every row (closed_loop_tools.py:102).  torch CUDA tensors in, torch CUDA tensor out."""
        import torch
        X = X.contiguous()
        U = U.contiguous()
        Xn = torch.empty_like(X)
        stream = ctypes.c_void_p(torch.cuda.current_stream(X.device).cuda_stream)
        self.__check(self.__lib.lib.tmpc_plant_step(self.__h, ctypes.c_void_p(X.data_ptr()), ctypes.c_void_p(U.data_ptr()),
                                                    X.shape[0], ctypes.c_void_p(Xn.data_ptr()), stream))
        return Xn

    def plant_jacobian(self, X, U):
        """[dF/dx | dF/du] at every row (C ABI: tmpc_plant_jacobian): torch CUDA tensors in, (B, nx, nx+nu) out."""
        import torch
        X = X.contiguous()
        U = U.contiguous()
        B = X.shape[0]
        JF = torch.empty((B, self.__pb.nx, self.__pb.nx + self.__pb.nu), dtype=torch.float64, device=X.device)
        stream = ctypes.c_void_p(torch.cuda.current_stream(X.device).cuda_stream)
        self.__check(self.__lib.lib.tmpc_plant_jacobian(self.__h, ctypes.c_void_p(X.data_ptr()), ctypes.c_void_p(U.data_ptr()), B,
                                                        ctypes.c_void_p(JF.data_ptr()), stream))
        return JF

    def stage_log(self, X, U):
        """l(x,u) and h(x,u) = C z + c for every row (closed_loop_tools.py:64-65, 98-99): torch CUDA tensors in,
        (l (B,), h (B,nh)) out."""
        import torch
        X = X.contiguous()
        U = U.contiguous()
        B = X.shape[0]
        l = torch.empty(B, dtype=torch.float64, device=X.device)
        hv = torch.empty((B, self.__pb.nh), dtype=torch.float64, device=X.device)
        stream = ctypes.c_void_p(torch.cuda.current_stream(X.device).cuda_stream)
        self.__check(self.__lib.lib.tmpc_stage_log(self.__h, ctypes.c_void_p(X.data_ptr()), ctypes.c_void_p(U.data_ptr()), B,
                                                   ctypes.c_void_p(l.data_ptr()), ctypes.c_void_p(hv.data_ptr()), stream))
        return l, hv

    def counters(self):
        out = (ctypes.c_int64 * 8)()
        self.__check(self.__lib.lib.tmpc_get_counters(self.__h, out))
        return {"sqp_iterations": out[0], "kernel_launches": out[1], "qp_solves": out[2], "stage_linearisations": out[3],
                "ls_dynamics_evals": out[4]}

    def timing(self):
        out = (ctypes.c_double * 4)()
        self.__check(self.__lib.lib.tmpc_get_timing(self.__h, out))
        return {"lin_ms": out[0], "qp_ms": out[1], "post_ms": out[2], "step_ms": out[3]}

    def fp64_peak_tflops(self):
        v = ctypes.c_double()
        self.__check(self.__lib.lib.tmpc_fp64_peak(self.__h, ctypes.byref(v)))
        return v.value

    # ---- properties of the reference object (pmpc.py:1120-1142) --------------------------------------
    @property
    def w(self):
        return self.__pb

    @property
    def w_sol(self):
        return self.__out["w"] if self.__out else None

    @property
    def g_sol(self):
        return self.__out["g"] if self.__out else None

    @property
    def lam_g(self):
        return self.__out["lam_g"] if self.__out else None

    @property
    def status(self):
        return self.__out["status"] if self.__out else None

    @property
    def last_phase(self):
        """the phase (index mod p) the last step used: the `phase` that solution_vjp() takes with that step's solution"""
        return self.__out["phase"] if self.__out else None

    @property
    def log(self):
        return self.__log

    @property
    def index(self):
        return self.__index

    @property
    def problem(self):
        return self.__pb

    @property
    def options(self):
        return dict(self.__options)

    @property
    def device(self):
        return self.__device

    @property
    def library_path(self):
        return self.__lib.path
