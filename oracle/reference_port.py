"""ORACLE -- TEST INFRASTRUCTURE ONLY.  Never imported by the product package (tunempc_b200/); only tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may use it.

CPU restatement (numpy + the plain-C stage functions of oracle/stage.c) of the reference hot path:
    Sqp.solve            tunempc/sqp_method.py:136-183   (and every helper :185-425)
    Pmpc.step/reset      tunempc/pmpc.py:371-423, :858-865, :867-906, :930-948
    NLP construction     tunempc/pmpc.py:162-369        (w/g/p layouts, bounds, tracking cost mtools.py:43-57)
with dense matrices exactly as the reference handles them (`.full()` + scipy null_space / eig).

PARITY UNPINNED: CasADi 3.5.1 (requirements.txt:3) cannot be imported here and the reference's tests hold no value
produced by Pmpc.step / Sqp.solve (SURVEY.md section 8(c)).  The port is pinned instead by (i) the LQ feedback gain
computed independently from a dense KKT solve, (ii) KKT residual checks of every solution, (iii) the QP solved by the
reference tree's own vendored qpOASES_e (oracle/_ref, built by oracle/Makefile) and cross-checked by a dense
Goldfarb-Idnani solver, (iv) finite differences of every derivative.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np
from scipy.linalg import eig, null_space

_HERE = os.path.dirname(os.path.abspath(__file__))
_dp = ctypes.POINTER(ctypes.c_double)


def _p(a):
    return a.ctypes.data_as(_dp) if a is not None else None


def build(models=("lq", "cstr", "unicycle", "evaporation", "chain", "dims9", "awe9", "evaporation_sc1")):
    """compile the C restatement (and oracle/_ref when the reference tree is present)."""
    subprocess.check_call(["make", "-s", "-C", _HERE, "MODELS=" + " ".join(models)])


class StageLib:
    """ctypes view of oracle/_build/liborc_<model>.so (oracle/stage.c)."""

    def __init__(self, name):
        path = os.path.join(_HERE, "_build", "liborc_%s.so" % name)
        if not os.path.exists(path):
            build((name,))
        self.lib = ctypes.CDLL(path)
        nx, nu, st, disc = ctypes.c_int(), ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        dt = ctypes.c_double()
        self.lib.orc_dims(ctypes.byref(nx), ctypes.byref(nu), ctypes.byref(st), ctypes.byref(dt), ctypes.byref(disc))
        self.nx, self.nu, self.nz = nx.value, nu.value, nx.value + nu.value
        self.lib.orc_F_map.argtypes = [ctypes.c_int, _dp, _dp, _dp, _dp, _dp, ctypes.c_int]

    def F(self, xs, us, order=0):
        """xs (n,nx), us (n,nu) -> xf (n,nx) [, S (n,nx,nz) [, T (n,nx,nz,nz)]]"""
        xs = np.ascontiguousarray(xs, dtype=np.float64).reshape(-1, self.nx)
        us = np.ascontiguousarray(us, dtype=np.float64).reshape(-1, self.nu)
        n = xs.shape[0]
        xf = np.zeros((n, self.nx))
        S = np.zeros((n, self.nx, self.nz)) if order >= 1 else None
        T = np.zeros((n, self.nx, self.nz, self.nz)) if order >= 2 else None
        self.lib.orc_F_map(n, _p(xs), _p(us), _p(xf), _p(S), _p(T), order)
        return (xf, S, T)[: order + 1] if order else xf


# ------------------------------------------------------------------------------------------------------
#  QP solvers:   min 1/2 d'Hd + g'd   s.t.  lba <= A d <= uba        (tunempc/sqp_method.py:158-168)
#  return (d, lam_a) with CasADi sign:  H d + g + A' lam_a = 0, lower-active => lam < 0
# ------------------------------------------------------------------------------------------------------
_qpo = None


class NonConvexQP(np.linalg.LinAlgError):
    """the dense solver's QP is not convex where it would have to be (see qp_dense)"""


class _NotPositiveDefinite(np.linalg.LinAlgError):
    """the reduced Hessian of the Goldfarb-Idnani solve has no Cholesky factor"""


def qpoases_available():
    return os.path.exists(os.path.join(_HERE, "_ref", "libqpoases_e.so"))


def qp_qpoases(H, g, A, lba, uba, lam_hint=None, info=None):
    """the reference tree's vendored qpOASES_e (oracle/_ref/libqpoases_e.so via oracle/qpoases_shim.c), cold-started as in
    the reference: lam_hint is not used."""
    if info is not None:
        info["branch"] = "qpoases"
    global _qpo
    if _qpo is None:
        _qpo = ctypes.CDLL(os.path.join(_HERE, "_ref", "libqpoases_e.so"))
        _qpo.qpo_solve.argtypes = [ctypes.c_int, ctypes.c_int, _dp, _dp, _dp, _dp, _dp, _dp, _dp,
                                   ctypes.POINTER(ctypes.c_int)]
    n, m = H.shape[0], A.shape[0]
    big = 1e20
    Hc = np.ascontiguousarray(H, dtype=np.float64)
    Ac = np.ascontiguousarray(A, dtype=np.float64)
    gc = np.ascontiguousarray(g, dtype=np.float64).ravel()
    lb = np.ascontiguousarray(np.clip(lba, -big, big), dtype=np.float64)
    ub = np.ascontiguousarray(np.clip(uba, -big, big), dtype=np.float64)
    x = np.zeros(n)
    lam = np.zeros(m)
    nwsr = ctypes.c_int(10 * (n + m))
    ret = _qpo.qpo_solve(n, m, _p(Hc), _p(gc), _p(Ac), _p(lb), _p(ub), _p(x), _p(lam), ctypes.byref(nwsr))
    if ret != 0:
        raise RuntimeError("qpOASES_e returned %d" % ret)
    return x, lam


def qp_dense(H, g, A, lba, uba, lam_hint=None, info=None, tol=1e-11):
    """own dense solver: null-space elimination of the equality rows, then Goldfarb-Idnani dual active set on the
    reduced strictly convex problem.  Exact (active-set) solution: inactive multipliers are exact zeros.

    A reduced Hessian that is not positive definite is first made so, only to find the active set; the QP is then
    re-solved on that active set with the original H (exact, free of the modification) and the result is accepted only
    as a KKT point of the original QP:
      - positive semidefinite (slack columns without curvature): a small proximal term on the null space;
      - indefinite (exact Hessian after the 'reduced' regularisation, which makes it positive definite only with the rows
        active in lam_hint held as well): rho/2 |A_S d - b_S|^2 over those held rows S, which vanishes with its gradient
        wherever they sit on their bounds, so the local minimiser on which they stay there is the one found.
    The point returned satisfies the second-order condition too: the reduced Hessian on its active set is positive
    semidefinite (a saddle point is rejected).  Raises NonConvexQP when neither gives such a point.  info (a dict), when
    given, receives the branch taken: 'gi', 'psd' or 'held'."""
    g = np.asarray(g, dtype=np.float64).ravel()
    if info is not None:
        info["branch"] = "gi"
    try:
        return _qp_dense_gi(H, g, A, lba, uba, tol)
    except _NotPositiveDefinite:
        pass
    n = H.shape[0]
    free = uba - lba != 0
    Z = null_space(A[~free]) if (~free).any() else np.eye(n)
    ev = np.linalg.eigvalsh(0.5 * (Z.T @ H @ Z + (Z.T @ H @ Z).T))
    big = max(1.0, np.abs(ev).max())
    S = None
    if ev.min() > -1e-10 * big:
        branch = "psd"
        Hm, gm = H + 1e-6 * big * Z @ Z.T, g
    else:
        branch = "held"
        if lam_hint is None:
            raise NonConvexQP("QP not convex on the null space of its equality rows")
        held = np.where(free & (lam_hint < 0) & np.isfinite(lba))[0]
        held_up = np.where(free & (lam_hint > 0) & np.isfinite(uba))[0]
        S = np.concatenate([held, held_up]).astype(int)
        bS = np.concatenate([lba[held], uba[held_up]])
        if len(S) == 0:
            raise NonConvexQP("QP not convex on the null space of its equality rows and no held rows")
        AS = A[S]
        rho = big / max(np.abs(AS).max() ** 2, 1e-300)
        for _ in range(40):
            Hm, gm = H + rho * AS.T @ AS, g - rho * AS.T @ bS
            if np.linalg.eigvalsh(0.5 * (Z.T @ Hm @ Z + (Z.T @ Hm @ Z).T)).min() > 0:
                break
            rho *= 10.0
        else:
            raise NonConvexQP("QP not convex on the face of its held rows")
    if info is not None:
        info["branch"] = branch
    try:
        d, lam = _qp_dense_gi(Hm, gm, A, lba, uba, tol)
    except _NotPositiveDefinite:
        raise NonConvexQP("QP not convex after the modification")
    if S is not None and np.abs(A[S] @ d - bS).max() > 1e-7 * max(1.0, np.abs(bS).max()):
        raise NonConvexQP("QP not convex and its held rows leave their bounds")
    # the active set found: equality rows and rows with a non-zero multiplier; exact solve of its KKT system with H
    W = np.where((~free) | (lam != 0))[0]
    bW = np.where(lam[W] > 0, uba[W], lba[W])
    m = len(W)
    K = np.block([[H, A[W].T], [A[W], np.zeros((m, m))]])
    sol = np.linalg.lstsq(K, np.concatenate([-g, bW]), rcond=None)[0]
    d = sol[:n]
    lam = np.zeros(A.shape[0])
    lam[W] = sol[n:]
    r = A @ d
    sc = max(1.0, np.abs(np.concatenate([lba[np.isfinite(lba)], uba[np.isfinite(uba)]])).max(initial=1.0))
    at_up = bW == uba[W]                                       # CasADi sign: lower-active <= 0, upper-active >= 0
    wrong = free[W] & np.where(at_up, lam[W] < -1e-10 * big, lam[W] > 1e-10 * big)
    if (np.any(r < lba - 1e-8 * sc) or np.any(r > uba + 1e-8 * sc) or wrong.any()
            or np.abs(H @ d + g + A.T @ lam).max() > 1e-8 * max(1.0, np.abs(g).max())):
        raise NonConvexQP("the modified QP's active set gives no KKT point of the QP")
    ZW = null_space(A[W]) if m else np.eye(n)
    if ZW.shape[1] and np.linalg.eigvalsh(0.5 * (ZW.T @ H @ ZW + (ZW.T @ H @ ZW).T)).min() < -1e-10 * big:
        raise NonConvexQP("the KKT point found is a saddle point of the QP")
    return d, lam


def _qp_dense_gi(H, g, A, lba, uba, tol):
    n = H.shape[0]
    eq = np.where(uba - lba == 0)[0]
    lo = np.where((uba - lba != 0) & np.isfinite(lba))[0]
    up = np.where((uba - lba != 0) & np.isfinite(uba))[0]
    Ae, be = A[eq], lba[eq]
    # inequalities as  G d >= h
    G = np.vstack([A[lo], -A[up]]) if (len(lo) + len(up)) else np.zeros((0, n))
    hh = np.concatenate([lba[lo], -uba[up]])
    owner = np.concatenate([lo, up]).astype(int)
    sign = np.concatenate([-np.ones(len(lo)), np.ones(len(up))])   # CasADi: lower-active -> negative
    if len(eq):
        Z = null_space(Ae)
        dp, *_ = np.linalg.lstsq(Ae, be, rcond=None)
        if np.linalg.norm(Ae @ dp - be, np.inf) > 1e-8 * max(1.0, np.linalg.norm(be, np.inf)):
            raise RuntimeError("QP infeasible (equalities)")
    else:
        Z = np.eye(n)
        dp = np.zeros(n)
    Hr = Z.T @ H @ Z
    Hr = 0.5 * (Hr + Hr.T)
    gr = Z.T @ (H @ dp + g)
    Gr = G @ Z
    hr = hh - G @ dp
    try:
        L = np.linalg.cholesky(Hr)
    except np.linalg.LinAlgError:
        raise _NotPositiveDefinite("reduced Hessian not positive definite")
    Hinv = lambda v: np.linalg.solve(L.T, np.linalg.solve(L, v))
    y = -Hinv(gr)
    act = []                                        # indices into G rows
    nu = np.zeros(0)
    for _ in range(20 * (len(hh) + 1)):
        s = Gr @ y - hr
        if len(s) == 0:
            break
        s[act] = 0.0
        scale = np.maximum(1.0, np.abs(hr))
        q = int(np.argmin(s / scale))
        if s[q] / scale[q] >= -tol:
            break
        nq = 0.0
        while True:
            aq = Gr[q]
            if act:
                Na = Gr[act].T                                  # (ny, m)
                HiN = Hinv(Na)
                Sm = Na.T @ HiN
                r = np.linalg.solve(Sm, Na.T @ Hinv(aq))
                z = Hinv(aq) - HiN @ r
            else:
                r = np.zeros(0)
                z = Hinv(aq)
            zn = aq @ z
            t1, jdrop = np.inf, -1
            for j in range(len(act)):
                if r[j] > 1e-14:
                    tj = nu[j] / r[j]
                    if tj < t1:
                        t1, jdrop = tj, j
            if zn <= 1e-13 * max(1.0, aq @ aq):                 # dependent: dual step only
                if not np.isfinite(t1):
                    raise RuntimeError("QP infeasible")
                nu = nu - t1 * r
                nq += t1
                act.pop(jdrop)
                nu = np.delete(nu, jdrop)
                continue
            t2 = -(aq @ y - hr[q]) / zn
            t = min(t1, t2)
            y = y + t * z
            nu = nu - t * r
            nq += t
            if t2 <= t1:
                act.append(q)
                nu = np.append(nu, nq)
                break
            act.pop(jdrop)
            nu = np.delete(nu, jdrop)
    else:
        raise RuntimeError("dense GI: iteration limit")
    d = dp + Z @ y
    lam = np.zeros(A.shape[0])
    for j, a in enumerate(act):
        lam[owner[a]] += sign[a] * nu[j]
    if len(eq):
        rhs = -(H @ d + g + A.T @ lam)
        le, *_ = np.linalg.lstsq(Ae.T, rhs, rcond=None)
        lam[eq] = le
    return d, lam


# ------------------------------------------------------------------------------------------------------
#  NLP of the tuned tracking MPC (tunempc/pmpc.py:162-369), dense
# ------------------------------------------------------------------------------------------------------
class GnlFuns:
    """the slacked nonlinear path constraints h_nl(x,u) of a model card (tunempc/preprocessing.py:78-118), lambdified
    straight from the sympy expressions: value (ns,), Jacobian (ns, nx+nu), second derivatives (ns, nx+nu, nx+nu).
    Independent of the generated C the device uses."""

    def __init__(self, model):
        import sympy as sp
        z = list(model.x) + list(model.u)
        g = sp.Matrix([sp.sympify(e) for e in model.gnl])
        self.ns = len(model.gnl)
        self._v = sp.lambdify([z], g, "numpy")
        self._j = sp.lambdify([z], g.jacobian(z), "numpy")
        self._h = [sp.lambdify([z], sp.hessian(e, z), "numpy") for e in g]

    def val(self, z):
        return np.asarray(self._v(list(z)), dtype=np.float64).ravel()

    def jac(self, z):
        return np.asarray(self._j(list(z)), dtype=np.float64).reshape(self.ns, len(z))

    def hess(self, z):
        return np.array([np.asarray(h(list(z)), dtype=np.float64) for h in self._h])


class TrackingNlp:
    def __init__(self, pb, stage=None, gnl=None):
        self.pb = pb
        self.stage = stage if stage is not None else StageLib(pb.name)
        assert self.stage.nx == pb.nx and self.stage.nu == pb.nu
        self.lbg, self.ubg = pb.bounds()
        self.gnl = gnl
        if pb.ns and gnl is None:
            from tunempc_b200 import configs            # the model card's expressions (not the generated code)
            self.gnl = GnlFuns(configs.CONFIGS[pb.name]()["model"])
        self.nzm = pb.nx + pb.nu

    # parameter vector p = (x0, wref window, H window, q window)   (pmpc.py:186-208, 380-391)
    def _split(self, w):
        pb = self.pb
        Z = w[: pb.N * pb.nz].reshape(pb.N, pb.nz)
        return Z, Z[:, : pb.nx], Z[:, pb.nx: pb.nx + pb.nu], w[pb.N * pb.nz:]

    def _dZ(self, w, p):
        """(x,u,us)_k - reference: the tracking cost's argument (pmpc.py:305-313); the reference window has no usc entries"""
        pb = self.pb
        Z, _, _, _ = self._split(w)
        return Z[:, : pb.nzr] - p["wref"][: pb.N * pb.nz].reshape(pb.N, pb.nz)[:, : pb.nzr]

    def f(self, w, p):
        pb = self.pb
        dZ = self._dZ(w, p)
        J = float(sum(0.5 * dZ[k] @ p["H"][k] @ dZ[k] + p["q"][k] @ dZ[k] for k in range(pb.N)))  # mtools.py:54-55
        if pb.nsc:                                                                                # pmpc.py:338-339
            Z, _, _, _ = self._split(w)
            J += float(sum(pb.scost @ Z[k, pb.nzr:] for k in range(pb.N)))
        return J

    def jacf(self, w, p):
        pb = self.pb
        dZ = self._dZ(w, p)
        gr = np.zeros(pb.n_w)
        for k in range(pb.N):
            gr[pb.izr(k)] = 0.5 * (p["H"][k] + p["H"][k].T) @ dZ[k] + p["q"][k]
            if pb.nsc:
                gr[pb.iusc(k)] = pb.scost
        return gr

    def g(self, w, p, order=0):
        """constraint vector (pmpc.py:242-287); order>=1 also returns the dense Jacobian, order 2 the stage tensors"""
        pb = self.pb
        Z, X, U, xN = self._split(w)
        out = self.stage.F(X, U, order)
        xf = out if order == 0 else out[0]
        g = np.zeros(pb.n_g)
        g[pb.g_init()] = X[0] - p["x0"]
        Xn = np.vstack([X[1:], xN[None, :]])
        nzm = self.nzm
        for k in range(pb.N):
            g[pb.g_dyn(k)] = xf[k] - Xn[k]
            if pb.ns:                                                     # g_k = h_nl(x_k,u_k) - us_k (preprocessing.py:107-108)
                g[pb.g_g(k)] = self.gnl.val(Z[k, :nzm]) - Z[k, nzm: nzm + pb.ns]
            if pb.nh:
                g[pb.g_h(k)] = pb.C @ Z[k] + pb.c
        g[pb.g_term()] = pb.T @ (xN - p["wref"][pb.N * pb.nz:])
        if order == 0:
            return g
        S = out[1]
        J = np.zeros((pb.n_g, pb.n_w))
        J[pb.g_init(), pb.ix(0)] = np.eye(pb.nx)
        for k in range(pb.N):
            J[pb.g_dyn(k), k * pb.nz: k * pb.nz + nzm] = S[k]
            J[pb.g_dyn(k), pb.ix(k + 1)] = -np.eye(pb.nx)
            if pb.ns:
                J[pb.g_g(k), k * pb.nz: k * pb.nz + nzm] = self.gnl.jac(Z[k, :nzm])
                J[pb.g_g(k), pb.ius(k)] = -np.eye(pb.ns)
            if pb.nh:
                J[pb.g_h(k), pb.iz(k)] = pb.C
        J[pb.g_term(), pb.ix(pb.N)] = pb.T
        if order == 1:
            return g, J
        return g, J, out[2]

    def hess(self, w, p, lam, mode):
        """exact: hessian(f + lam'g) (sqp_method.py:90-96);  gauss_newton: blkdiag(H_k, 0_nx) (pmpc.py:327-333)"""
        pb = self.pb
        Hm = np.zeros((pb.n_w, pb.n_w))
        for k in range(pb.N):
            Hm[pb.izr(k), pb.izr(k)] = 0.5 * (p["H"][k] + p["H"][k].T)     # usc rows / columns stay zero (pmpc.py:327-333)
        if mode == "exact":
            _, _, T2 = self.g(w, p, order=2)
            Z, _, _, _ = self._split(w)
            for k in range(pb.N):
                zs = slice(k * pb.nz, k * pb.nz + self.nzm)
                Hm[zs, zs] += np.einsum("a,aij->ij", lam[pb.g_dyn(k)], T2[k])
                if pb.ns:
                    Hm[zs, zs] += np.einsum("a,aij->ij", lam[pb.g_g(k)], self.gnl.hess(Z[k, : self.nzm]))
        return Hm


class EconomicNlp(TrackingNlp):
    """economic MPC NLP (pmpc.py:97-107,173-183,299-301): same constraints, stage cost l(x_k,u_k) given as python callables
    (l, grad l, hess l) of z = (x,u); the Hessian is always exact (pmpc.py:101-104)."""

    def __init__(self, pb, cost_funs, stage=None):
        super().__init__(pb, stage)
        self.l_f, self.g_f, self.H_f = cost_funs

    def f(self, w, p):
        Z, _, _, _ = self._split(w)
        return float(sum(self.l_f(Z[k]) for k in range(self.pb.N)))

    def jacf(self, w, p):
        pb = self.pb
        Z, _, _, _ = self._split(w)
        gr = np.zeros(pb.n_w)
        for k in range(pb.N):
            gr[pb.iz(k)] = self.g_f(Z[k])
        return gr

    def hess(self, w, p, lam, mode):
        pb = self.pb
        Z, _, _, _ = self._split(w)
        Hm = np.zeros((pb.n_w, pb.n_w))
        _, _, T2 = self.g(w, p, order=2)
        for k in range(pb.N):
            Hk = np.asarray(self.H_f(Z[k]), dtype=np.float64)
            Hm[pb.iz(k), pb.iz(k)] = 0.5 * (Hk + Hk.T) + np.einsum("a,aij->ij", lam[pb.g_dyn(k)], T2[k])
        return Hm


# ------------------------------------------------------------------------------------------------------
#  Sqp  (tunempc/sqp_method.py)
# ------------------------------------------------------------------------------------------------------
class Sqp:
    def __init__(self, nlp, options=None, qp="auto"):
        self.nlp = nlp
        self.opts = {  # sqp_method.py:52-61
            "regularization": "reduced", "regularization_tol": 1e-8, "tol": 1e-6, "lam_tresh": 1e-8,
            "max_ls_iter": 300, "ls_step_factor": 0.8, "hessian_approximation": "exact", "max_iter": 2000,
        }
        for k, v in (options or {}).items():
            self.opts[k] = v
        if qp == "auto":
            qp = "qpoases" if qpoases_available() else "dense"
        self.qp = qp_qpoases if qp == "qpoases" else qp_dense
        self.stats = {}
        self.n_qp = 0
        self.n_reg = 0

    # sqp_method.py:223-238
    def _prefilter(self, lam):
        lam = np.array(lam, dtype=np.float64, copy=True)
        lam[np.abs(lam) < self.opts["lam_tresh"]] = 0.0
        return lam

    def _viol(self, g):  # sqp_method.py:253-256
        return float(np.linalg.norm(np.abs(np.minimum(g - self.nlp.lbg, 0.0) + np.maximum(g - self.nlp.ubg, 0.0)),
                                    np.inf))

    # sqp_method.py:405-425
    def _active_jac(self, J, lam):
        bounds = self.nlp.ubg - self.nlp.lbg
        eq_idx = [i for i, e in enumerate(bounds) if e == 0]
        as_idx = [i for i, e in enumerate(bounds) if e != 0 and lam[i] != 0]
        return J[eq_idx + as_idx, :], as_idx

    # sqp_method.py:327-403 ('reduced' branch)
    def _regularize(self, H, J, lam):
        tol = self.opts["regularization_tol"]
        Jact, _ = self._active_jac(J, lam)
        Z = null_space(Jact)
        Hr = Z.T @ H @ Z
        if Hr.shape[0] != 0:
            eva, evec = eig(Hr)
            regularize = min(eva.real) < tol
        else:
            regularize = False
        if regularize:
            self.n_reg += 1
            evmod = np.where(eva.real < tol, tol, eva)
            deva = evmod - eva
            dHr = evec @ np.diag(deva) @ np.linalg.inv(evec)
            H = H + Z @ dHr @ Z.T
            H = (H.real + H.real.T) / 2.0
        return H

    def _dual_infeas(self, w, p, lam, J=None):  # jlag_fun, sqp_method.py:246
        if J is None:
            _, J = self.nlp.g(w, p, order=1)
        return float(np.linalg.norm(self.nlp.jacf(w, p) + J.T @ lam, np.inf))

    def solve(self, w0, p0, lam_g_ip):
        o = self.opts
        nlp = self.nlp
        w0 = np.array(w0, dtype=np.float64, copy=True)
        lam = self._prefilter(lam_g_ip)                               # :142
        # k = 0 bookkeeping of __check_convergence (:248-261); its verdict is discarded (:145-146)
        g0, J = nlp.g(w0, p0, order=1)
        filt = [(nlp.f(w0, p0), self._viol(g0))]
        _, as_init = self._active_jac(J, lam)
        alpha = 0.0
        k = 0
        converged = False
        branches = {"gi": 0, "psd": 0, "held": 0, "qpoases": 0, "gn_resolve": 0}
        info = {}
        while not converged:                                          # :149
            g0, J = nlp.g(w0, p0, order=1)                            # :152
            H = nlp.hess(w0, p0, lam, o["hessian_approximation"])     # :330
            if o["regularization"] == "reduced":
                H = self._regularize(H, J, lam)                       # :155
            try:
                d, lam_new = self.qp(H, nlp.jacf(w0, p0), J, nlp.lbg - g0, nlp.ubg - g0, lam, info)   # :158-168
            except NonConvexQP:
                # qpOASES follows its homotopy through a QP that is not convex; the dense solver cannot.  Like the device
                # solver (DESIGN.md), re-solve this iteration with the Gauss-Newton Hessian (economic NLPs have none: raises
                # again).  Converged points stay those of the reference, the iteration path may not.
                branches["gn_resolve"] += 1
                H = nlp.hess(w0, p0, lam, "gauss_newton")
                d, lam_new = self.qp(H, nlp.jacf(w0, p0), J, nlp.lbg - g0, nlp.ubg - g0, lam, info)
            branches[info["branch"]] += 1
            self.n_qp += 1
            # line search (:289-325)
            alpha = 1.0
            wn = w0 + alpha * d
            fn, vn = nlp.f(wn, p0), self._viol(nlp.g(wn, p0))
            for _ in range(o["max_ls_iter"]):
                ndom = sum(1 for (F_, V_) in filt if (fn > F_) and (vn > V_))
                if ndom > 1:
                    alpha *= o["ls_step_factor"]
                    wn = w0 + alpha * d
                    fn, vn = nlp.f(wn, p0), self._viol(nlp.g(wn, p0))
                else:
                    break
            filt.append((fn, vn))                                     # :323
            w0 = w0 + alpha * d                                       # :174
            lam = lam_new                                             # :175 (full dual step)
            k += 1
            dual = self._dual_infeas(w0, p0, lam)                     # :246
            if filt[-1][1] < o["tol"] and dual < o["tol"]:            # :276-277
                converged = True
            elif k == o["max_iter"]:                                  # :281
                converged = True
        # postprocessing (:185-221)
        g0, J = nlp.g(w0, p0, order=1)
        H = nlp.hess(w0, p0, lam, o["hessian_approximation"])
        Jact, as_idx = self._active_jac(J, lam)
        Z = null_space(Jact)
        Hred = Z.T @ H @ Z
        min_eig = float(np.min(np.linalg.eigvals(Hred).real)) if Hred.shape[0] > 0 else np.inf
        status = 0
        if not (min_eig > o["regularization_tol"]):
            status = 3                                                # reference: AssertionError (:199-201)
        elif not (filt[-1][1] < o["tol"] and dual < o["tol"]):
            status = 1
        nAC = len([i for i in as_init if i not in as_idx]) + len([i for i in as_idx if i not in as_init])
        self.stats = {"x": w0, "lam_g": lam, "iter_count": k, "f": nlp.f(w0, p0), "nAC": nAC, "nAS": len(as_idx),
                      "status": status, "alpha": alpha, "min_eig": min_eig, "filter": np.array(filt),
                      "dual_infeas": dual, "as_idx": as_idx,
                      # QP solves per branch of qp_dense (or qpOASES); gn_resolve counts iterations re-solved with the
                      # Gauss-Newton Hessian, where the iteration path is no longer the reference's
                      "qp_branches": branches}
        return {"x": w0, "lam_g": lam, "S": {"H": H}}


# ------------------------------------------------------------------------------------------------------
#  Pmpc  (tunempc/pmpc.py) -- tracking/tuned type only
# ------------------------------------------------------------------------------------------------------
class Pmpc:
    def __init__(self, pb, tables=None, qp="auto", sqp_options=None, cost_funs=None):
        from tunempc_b200.problem import build_tables   # host-side table builder (restates pmpc.py:676-783)
        self.pb = pb
        self.tab = tables if tables is not None else build_tables(pb)
        if getattr(pb, "mpc_type", "tuned") == "economic":
            if cost_funs is None:
                raise ValueError("economic controller: pass cost_funs = (l, grad l, hess l)")
            self.nlp = EconomicNlp(pb, cost_funs)
        else:
            self.nlp = TrackingNlp(pb)
        so = {"hessian_approximation": "exact" if getattr(pb, "mpc_type", "tuned") == "economic" else pb.hessian_approximation,
              "max_iter": pb.max_iter, "tol": pb.tol}
        so.update(sqp_options or {})
        self.sqp = Sqp(self.nlp, so, qp=qp)
        self.reset()

    def reset(self):                                                  # pmpc.py:858-865, 930-942
        self.index = 0
        self.log = {k: [] for k in ("iter", "f", "status", "sol_x", "lam_g", "u0", "nACtot", "nAC", "nAS")}
        self.w0 = self.tab.ref[self.index].copy()
        self.lam_g0 = self.tab.ref_du[self.index].copy()

    def step(self, x0):                                               # pmpc.py:371-423
        pb = self.pb
        self.index = self.index % pb.p                                # :377
        idx = self.index
        p0 = {"x0": np.asarray(x0, dtype=np.float64).ravel(), "wref": self.tab.ref[idx],
              "H": self.tab.Href[idx], "q": self.tab.qref[idx]}       # :380-391
        sol = self.sqp.solve(self.w0, p0, self.lam_g0)                # :407
        self.w_sol = sol["x"]
        self.lam_g = sol["lam_g"]
        self.g_sol = self.nlp.g(sol["x"], p0)                         # :410
        st = self.sqp.stats
        # __detect_AC (:840-856): stage-0 active-set changes w.r.t. the reference multipliers
        nAC0 = 0
        if pb.nh:
            lo = self.lam_g[pb.g_h(0)]
            lr = self.tab.ref_du[idx][pb.g_h(0)]
            io = {i for i in range(pb.nh) if lo[i] != 0}
            ir = {i for i in range(pb.nh) if lr[i] != 0}
            nAC0 = len(io ^ ir)
        for key, val in (("iter", st["iter_count"]), ("f", st["f"]), ("status", st["status"]),
                         ("sol_x", self.w_sol), ("lam_g", self.lam_g), ("u0", self.w_sol[pb.iu(0)].copy()),
                         ("nACtot", st["nAC"]), ("nAC", nAC0), ("nAS", st["nAS"])):
            self.log[key].append(val)
        self.index += 1                                               # :415
        self.w0, self.lam_g0 = self._shift(self.w_sol, self.lam_g)    # :418-421
        return self.w_sol[pb.iu(0)].copy()

    def _shift(self, w, lam):                                         # pmpc.py:867-906
        pb = self.pb
        N = pb.N
        ws = np.zeros_like(w)
        ls = np.zeros_like(lam)
        ls[pb.g_init()] = lam[pb.g_dyn(0)]
        for i in range(N):
            ws[pb.ix(i)] = w[pb.ix(i + 1)]
            if i < N - 1:
                ws[pb.iu(i)] = w[pb.iu(i + 1)]
                ws[pb.ius(i)] = w[pb.ius(i + 1)]                          # :881-884
                ws[pb.iusc(i)] = w[pb.iusc(i + 1)]
                ls[pb.g_dyn(i)] = lam[pb.g_dyn(i + 1)]
                ls[pb.g_g(i)] = lam[pb.g_g(i + 1)]                        # :888-890
                if pb.nh:
                    ls[pb.g_h(i)] = lam[pb.g_h(i + 1)]
        ws[pb.ix(N)] = ws[pb.ix(N - 1)]
        ws[pb.iu(N - 1)] = ws[pb.iu(N - 2)]
        ws[pb.ius(N - 1)] = ws[pb.ius(N - 2)]                             # :895-898
        ws[pb.iusc(N - 1)] = ws[pb.iusc(N - 2)]
        ls[pb.g_dyn(N - 1)] = ls[pb.g_dyn(N - 2)]
        ls[pb.g_g(N - 1)] = ls[pb.g_g(N - 2)]
        if pb.nh:
            ls[pb.g_h(N - 1)] = ls[pb.g_h(N - 2)]
        ls[pb.g_term()] = lam[pb.g_term()]
        return ws, ls
