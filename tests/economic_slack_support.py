"""Economic MPC with slack variables: the NLP of the CPU oracle and host helpers -- test infrastructure only.

The oracle's EconomicNlp (oracle/reference_port.py) evaluates l on the whole stage vector.  With slacks the stage variables are
z = (x, u, us, usc) and the economic stage cost is l(x_k, u_k) + scost'usc_k (tunempc/pmpc.py:299-301, 338-339), so the
restatement here follows TrackingNlp: l and its derivatives act on the (x,u) slice only, the usc entries carry the linear cost
scost, and the exact Hessian adds lam_g' d2 h_nl of the slacked nonlinear rows.  Without slacks it computes what EconomicNlp
computes.  The tests use it as an independent statement of the problem: the device routines' solutions must be its KKT points.
"""
import numpy as np

from oracle import reference_port as rp


class EconomicSlackNlp(rp.EconomicNlp):
    def f(self, w, p):
        pb = self.pb
        Z, _, _, _ = self._split(w)
        J = float(sum(self.l_f(Z[k, : self.nzm]) for k in range(pb.N)))
        if pb.nsc:
            J += float(sum(pb.scost @ Z[k, pb.nzr:] for k in range(pb.N)))
        return J

    def jacf(self, w, p):
        pb = self.pb
        Z, _, _, _ = self._split(w)
        gr = np.zeros(pb.n_w)
        for k in range(pb.N):
            gr[k * pb.nz: k * pb.nz + self.nzm] = self.g_f(Z[k, : self.nzm])
            if pb.nsc:
                gr[pb.iusc(k)] = pb.scost
        return gr

    def hess(self, w, p, lam, mode):
        """always exact (pmpc.py:101-104): sym(d2l) + lam_dyn' d2F (+ lam_g' d2 h_nl) on the (x,u) block, zero on the slacks"""
        pb = self.pb
        Z, _, _, _ = self._split(w)
        Hm = np.zeros((pb.n_w, pb.n_w))
        _, _, T2 = self.g(w, p, order=2)
        for k in range(pb.N):
            zs = slice(k * pb.nz, k * pb.nz + self.nzm)
            Hk = np.asarray(self.H_f(Z[k, : self.nzm]), dtype=np.float64)
            Hm[zs, zs] = 0.5 * (Hk + Hk.T) + np.einsum("a,aij->ij", lam[pb.g_dyn(k)], T2[k])
            if pb.ns:
                Hm[zs, zs] += np.einsum("a,aij->ij", lam[pb.g_g(k)], self.gnl.hess(Z[k, : self.nzm]))
        return Hm


def cost_funs(name):
    """(l, grad l, hess l) of z = (x,u) for a config of tunempc_b200.configs (the soft variants share the base card's cost)"""
    from tunempc_b200 import configs, tuning
    cfg = configs.CONFIGS[name]()
    return tuning.lambdify_cost(cfg["model"], cfg["cost"])


def tuner_problem(tuner, mpc_type, N, opts=None):
    """the MpcProblem that `tuner.create_mpc(mpc_type, N, opts)` hands to the controller, without a device: the controller class is
    replaced by one that only runs problem_from_reference_args on the arguments create_mpc passes"""
    from tunempc_b200 import pmpc

    class _Capture:
        def __init__(self, N=None, sys=None, cost=None, wref=None, tuning=None, lam_g_ref=None, sensitivities=None,
                     options=None, device=0):
            self.problem = pmpc.problem_from_reference_args(N, sys, cost, wref, tuning, lam_g_ref, sensitivities, options)

    real = pmpc.Pmpc
    pmpc.Pmpc = _Capture
    try:
        return tuner.create_mpc(mpc_type, N, opts=opts or {}).problem
    finally:
        pmpc.Pmpc = real


def economic_problem(name):
    """(MpcProblem, config whose l is the stage cost, Tuner or None) of the economic controllers with slacks the tests use:
      awe9            configs.awe9_problem(..., mpc_type='economic'): ns 3, nsc 3, N 20, p 40
      evaporation_sc1 Tuner(configs.evaporation()).solve_ocp(); create_mpc('economic', 30, opts={'slack_flag': 'active'})
      dims9g          Tuner(configs.dims9g()).solve_ocp(); create_mpc('economic', 20): slacked nonlinear rows"""
    import os
    from tunempc_b200 import configs, modelgen
    from tunempc_b200.tuner import Tuner
    if name == "awe9":
        return configs.awe9_problem(rp.StageLib("awe9").F, mpc_type="economic")[0], "awe9", None
    if name == "evaporation_sc1":
        t = Tuner(configs.evaporation(), p=1, stage_eval=rp.StageLib("evaporation").F)
        t.solve_ocp()
        return tuner_problem(t, "economic", 30, {"slack_flag": "active"}), "evaporation", t
    card = configs.dims9g()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    modelgen.generate_header(card["model"], os.path.join(root, "tunempc_b200", "csrc", "gen", "model_dims9g.h"))
    t = Tuner(card, p=1, stage_eval=rp.StageLib("dims9g").F)
    t.solve_ocp()
    return tuner_problem(t, "economic", 20), "dims9g", t


def initial_states(name, pb, B=12):
    """seeded x0 near the reference: evaporation_sc1 with a third of them below the softened bound X2 >= 25 (non-zero slack);
    dims9g shrunk towards the steady state as in the tuned dims9g test (the hard nonlinear state row)"""
    from tunempc_b200 import configs
    xs = pb.wref[0, :pb.nx]
    if name == "evaporation_sc1":
        X0 = configs.sample_x0("evaporation_sc1", pb, B, 11)
        X0[::3, 0] = 25.0 - np.linspace(0.05, 0.8, len(X0[::3]))
        return X0
    if name == "dims9g":
        return xs + 0.08 * (configs.sample_x0("dims9g", pb, B, 3) - xs)
    return configs.sample_x0(name, pb, B, 7)


def kkt_error(nlp, pb, tab, x0, w, lam, phase=0):
    """max of |grad L|, the constraint violation and the wrong-sign inequality multipliers (CasADi: active lower => negative)
    of the NLP at (w, lam) for the initial state x0"""
    p0 = {"x0": np.asarray(x0, dtype=np.float64), "wref": tab.ref[phase], "H": tab.Href[phase], "q": tab.qref[phase]}
    g, J = nlp.g(w, p0, order=1)
    lbg, ubg = pb.bounds()
    ineq = ubg != lbg
    return max(np.abs(nlp.jacf(w, p0) + J.T @ lam).max(), (np.maximum(lbg - g, 0.0) + np.maximum(g - ubg, 0.0)).max(),
               np.maximum(lam[ineq], 0.0).max(initial=0.0))
