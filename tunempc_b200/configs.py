"""Model cards of the BASELINE.json configs, restated from the reference example scripts.

Every constant cites the reference line it comes from.  Each card returns the sympy ODE (`OdeModel`),
the economic stage cost l(x,u) as a sympy expression, the *linear* path constraints h(x,u) = C z + c >= 0
(all non-AWE configs have linear h, so `preprocessing.input_formatting` (`tunempc/preprocessing.py:78-118`)
would leave ns = 0), the OCP initial guess and the x0-perturbation scale of SURVEY.md section 8(d).
"""
from __future__ import annotations

import numpy as np
import sympy as sp

from .modelgen import OdeModel


def lq():
    """examples/convex_lqr.py:40-46 -- discrete LQ system, indefinite stage cost, steady state 0."""
    A = np.array([[-0.3319, 0.7595, 1.5399], [-0.3393, 0.1250, 0.4245], [-0.5090, 0.9388, 0.8864]])
    B = np.array([[0.1060], [-1.3835], [-0.1496]])
    Q = np.array([[-1.0029, -0.0896, 1.1050], [-0.0896, 1.6790, -0.5762], [1.1050, -0.5762, -0.4381]])
    R = np.array([[0.6192]])
    Nm = np.array([[-0.0420], [0.2112], [-0.2832]])
    x = sp.symbols("x0:3")
    u = sp.symbols("u0:1")
    z = sp.Matrix(list(x) + list(u))
    xdot = list(sp.Matrix(A) * sp.Matrix(x) + sp.Matrix(B) * sp.Matrix(u))
    Hm = np.block([[Q, Nm], [Nm.T, R]])
    cost = sp.Rational(1, 2) * (z.T * sp.Matrix(Hm) * z)[0, 0]
    model = OdeModel("lq", x, u, xdot, discrete=True, cost=cost)
    return dict(model=model, cost=cost, C=np.zeros((0, 4)), c=np.zeros(0),
                w_guess=np.zeros(4), period=1, A=A, B=B, Q=Q, R=R, Nmat=Nm,
                x0_scale=np.array([1.0, 1.0, 1.0]), N=10, term_idx=[0, 1, 2])


def cstr():
    """examples/cstr/cstr_model.py:34-168 -- CSTR, nx=4, nu=2, RK4 x 20 over 20 s, four input bounds."""
    k10, k20, k30 = 1.287e12, 1.287e12, 9.043e9           # :41-43
    E1, E2, E3 = -9758.3, -9758.3, -8560.0                # :44-46
    DH_AB, DH_BC, DH_AD = 4.2, -11.0, -41.85              # :47-49
    rho, Cp, kw, AR, VR = 0.9342, 3.01, 4032.0, 0.215, 10.0   # :50-54
    mK, CPK, cA0, theta0 = 5.0, 2.0, 5.10, 104.9          # :55-58
    rhoJ = 1e-1                                           # examples/cstr/main.py:57
    cA, cB, th, thK = sp.symbols("cA cB theta thetaK")
    Vd, QK = sp.symbols("Vdot QdotK")
    k1 = k10 * sp.exp(E1 / (th + 273.15))                 # :68-74
    k2 = k20 * sp.exp(E2 / (th + 273.15))
    k3 = k30 * sp.exp(E3 / (th + 273.15))
    xdot = [                                              # :82-91, divided by 3600 at :94
        (Vd * (cA0 - cA) - k1 * cA - k3 * cA * cA) / 3600,
        (-Vd * cB + k1 * cA - k2 * cB) / 3600,
        (Vd * (theta0 - th) - 1.0 / (rho * Cp) * (k1 * cA * DH_AB + k2 * cB * DH_BC + k3 * cA * cA * DH_AD)
         + kw * AR / (rho * Cp * VR) * (thK - th)) / 3600,
        (1.0 / (mK * CPK) * (QK + kw * AR * (th - thK))) / 3600,
    ]
    cost = 100 * (-cB / cA0 + rhoJ * (1e-4 * (Vd - 14.19) ** 2 + 1e-4 * (QK + 1113.5) ** 2))  # :117-129
    # h >= 0 (:154-159): Vdot-5, 35-Vdot, QdotK+9000, -QdotK
    C = np.zeros((4, 6))
    C[0, 4], C[1, 4], C[2, 5], C[3, 5] = 1.0, -1.0, 1.0, -1.0
    c = np.array([-5.0, 35.0, 9000.0, 0.0])
    model = OdeModel("cstr", (cA, cB, th, thK), (Vd, QK), xdot, rk_steps=20, tf=20.0, cost=cost)   # :62-64,97
    w_guess = np.array([2.1402, 1.0903, 114.191, 112.9066, 14.19, -1113.5])               # :168
    return dict(model=model, cost=cost, C=C, c=c, w_guess=w_guess, period=1, N=20,
                term_idx=[0, 1, 2, 3])


def unicycle():
    """examples/unicycle/main.py:40-129 -- periodic unicycle, nx=4, nu=1, RK4 x 50 over T/N, p=N=30."""
    rho_, v = 0.001, 1.0                                  # :46-47
    T, Np = 5.0, 30                                       # :87-88,97-99
    z_, y_, ez, ey = sp.symbols("z y ez ey")
    uu = sp.symbols("u")
    xdot = [                                              # :56-61
        v * ez,
        v * ey,
        -uu * ey - rho_ * ez * (ez ** 2 + ey ** 2 - 1),
        uu * ez - rho_ * ey * (ez ** 2 + ey ** 2 - 1),
    ]
    cost = uu ** 2 + z_ ** 2 + 5 * y_ ** 2                # :82
    model = OdeModel("unicycle", (z_, y_, ez, ey), (uu,), xdot, rk_steps=50, tf=T / Np, cost=cost)  # :67
    # analytic circular initial guess (:103-114)
    om = 2 * np.pi / T
    tg = np.arange(Np) * T / Np
    guess = np.stack([np.sin(om * tg) / om, -np.cos(om * tg) / om, np.cos(om * tg), np.sin(om * tg),
                      om * np.ones(Np)], axis=1)
    # terminal projection (examples/unicycle/main.py:124-129 selects x[0:3] = (z, y, ez)).  The OCP solution computed by
    # tuning.solve_periodic_ocp keeps the phase of the initial guess (ez = +-1, ey = 0 at k = 0, 15); there ez is the
    # radial direction of the invariant ez^2 + ey^2 = 1, which the input cannot move, so the reference's selection makes
    # the terminal constraint locally redundant and the SQP breaks down at those phases (the reference example runs with
    # ipopt_presolve=True, pmpc.py:394-404, unavailable here).  (z, y, ey) is the same projection a quarter turn away
    # and is well posed at every phase of this grid.
    return dict(model=model, cost=cost, C=np.zeros((0, 5)), c=np.zeros(0), w_guess=guess, period=Np, N=Np,
                term_idx=[0, 1, 3], x0_scale=np.array([0.5, 0.1, 0.0, 0.0]))                       # :172 disturbance sizes


def evaporation():
    """examples/evaporation_process/main.py:42-138 -- evaporation process, nx=2 (X2,P2), nu=2 (P100,F200), CasADi
    'collocation' integrator over tf = 1 (:103), five linear constraints of which three are pure state constraints."""
    a, b, c_, d, e, f_, g, h_ = 0.5616, 0.3126, 48.43, 0.507, 55.0, 0.1538, 90.0, 0.16      # :49-56
    M, Cc, UA2, Cp, lam, lams = 20.0, 4.0, 6.84, 0.07, 38.5, 36.6                              # :58-63
    F1, X1, F3, T1, T200 = 10.0, 5.0, 50.0, 40.0, 25.0                                         # :64-68
    X2, P2 = sp.symbols("X2 P2")
    P100, F200 = sp.symbols("P100 F200")
    T2 = a * P2 + b * X2 + c_                                                                 # :77-86
    T3 = d * P2 + e
    T100 = f_ * P100 + g
    UA1 = h_ * (F1 + F3)
    Q100 = UA1 * (T100 - T2)
    F100 = Q100 / lams
    Q200 = UA2 * (T3 - T200) / (1.0 + UA2 / (2.0 * Cp * F200))
    F5 = Q200 / lam
    F4 = (Q100 - F1 * Cp * (T2 - T1)) / lam
    F2 = F1 - F4
    xdot = [(F1 * X1 - F2 * X2) / M, (F4 - F5) / Cc]                                          # :96-99
    cost = 10.09 * (F2 + F3) + 600.0 * F100 + 0.6 * F200                                      # :121
    C = np.zeros((5, 4))                                                                      # :130-136
    C[0, 0], C[1, 1], C[2, 1], C[3, 2], C[4, 3] = 1.0, 1.0, -1.0, -1.0, -1.0
    c = np.array([-25.0, -40.0, 80.0, 400.0, 400.0])
    model = OdeModel("evaporation", (X2, P2), (P100, F200), xdot, rk_steps=20, tf=1.0, integrator="collocation", cost=cost)
    w_guess = np.array([25.0, 49.743, 191.713, 215.888])                                      # :155
    return dict(model=model, cost=cost, C=C, c=c, w_guess=w_guess, period=1, N=30, term_idx=[0, 1],
                conv_rho=1e-3)                                                                # :157 convexify(rho = 1e-3)


def chain():
    """SYNTHETIC (not in the reference): three masses on a line coupled by hardening springs, forces on the outer two.
    nx = 6, nu = 2 (nz = 8): exercises the generic-dimension paths (greedy direction groups in modelgen, the
    pair-per-thread linearisation when the warp-specialised kernel does not fit the register file)."""
    p = sp.symbols("p1:4")
    v = sp.symbols("v1:4")
    f = sp.symbols("f1 f3")
    k1, k3, dmp = 2.0, 0.8, 0.3
    spring = lambda dlt: k1 * dlt + k3 * dlt ** 3
    acc = [-spring(p[0]) + spring(p[1] - p[0]) - dmp * v[0] + f[0],
           -spring(p[1] - p[0]) + spring(p[2] - p[1]) - dmp * v[1],
           -spring(p[2] - p[1]) - dmp * v[2] + f[1]]
    xdot = [v[0], v[1], v[2]] + acc
    cost = (p[0] - 0.4) ** 2 + (p[1] - 0.7) ** 2 + 2 * (p[2] - 1.0) ** 2 + 0.1 * (v[0] ** 2 + v[1] ** 2 + v[2] ** 2) \
        + 0.05 * (f[0] ** 2 + f[1] ** 2)
    C = np.zeros((4, 8))
    C[0, 6], C[1, 6], C[2, 7], C[3, 7] = 1.0, -1.0, 1.0, -1.0
    c = np.array([1.0, 1.2, 1.0, 2.5])                                   # -1 <= f1 <= 1.2, -1 <= f3 <= 2.5
    model = OdeModel("chain", p + v, f, xdot, rk_steps=8, tf=0.4, cost=cost)
    return dict(model=model, cost=cost, C=C, c=c, w_guess=np.array([0.4, 0.7, 1.0, 0, 0, 0, 0.5, 1.0]), period=1, N=15,
                term_idx=[0, 1, 2, 3, 4, 5])


def dims9():
    """SYNTHETIC (not in the reference): stand-in with the DIMENSIONS of the AWE config (#5, SURVEY.md 8.0: nx = 9, nu = 3,
    14 path-constraint rows, N = 20, 7-row projected terminal constraint x[1:3], x[4:]); the reference's kite model is an
    opaque CasADi pickle.  Four masses with hardening springs, an actuator lag state, state-only, input-only and mixed
    constraint rows.  Exercises nz = 12: one warp-level QP per CTA (shared-memory fit), 280 inequality rows."""
    p = sp.symbols("p1:5")
    v = sp.symbols("v1:5")
    a = sp.symbols("a")
    u = sp.symbols("u1 u2 u3")
    k1, k3, dmp, tau = 1.5, 0.6, 0.25, 0.5
    spring = lambda dlt: k1 * dlt + k3 * dlt ** 3
    acc = [-spring(p[0]) + spring(p[1] - p[0]) - dmp * v[0] + u[0],
           -spring(p[1] - p[0]) + spring(p[2] - p[1]) - dmp * v[1] + a,
           -spring(p[2] - p[1]) + spring(p[3] - p[2]) - dmp * v[2],
           -spring(p[3] - p[2]) - dmp * v[3] + u[1] * (1 + 0.2 * p[3])]
    xdot = list(v) + acc + [(u[2] - a) / tau]
    cost = ((p[0] - 0.3) ** 2 + (p[1] - 0.6) ** 2 + (p[2] - 0.8) ** 2 + 2 * (p[3] - 1.1) ** 2
            + 0.1 * sum(vi ** 2 for vi in v) + 0.05 * a ** 2 + 0.05 * (u[0] ** 2 + u[1] ** 2) + 0.02 * u[2] ** 2)
    nz = 12
    rows = []
    def row(coefs, const):
        r = np.zeros(nz)
        for idx, val in coefs:
            r[idx] = val
        rows.append((r, const))
    for j, (lo, hi) in zip((9, 10, 11), ((-1.0, 1.0), (-1.0, 2.0), (-1.5, 1.5))):      # input bounds (6 rows)
        row([(j, 1.0)], -lo)
        row([(j, -1.0)], hi)
    row([(8, 1.0)], 1.2)                                                               # actuator state bounds (state only)
    row([(8, -1.0)], 1.2)
    for j, hi in zip((0, 1, 2), (0.9, 1.2, 1.4)):                                      # position upper bounds (state only)
        row([(j, -1.0)], hi)
    row([(9, -1.0), (0, -0.5)], 1.1)                                                   # mixed row: u1 + 0.5 p1 <= 1.1
    row([(7, 1.0)], 1.5)                                                               # |v4| <= 1.5
    row([(7, -1.0)], 1.5)
    C = np.array([r for r, _ in rows])
    cc = np.array([c0 for _, c0 in rows])
    model = OdeModel("dims9", p + v + (a,), u, xdot, rk_steps=10, tf=0.3, cost=cost)
    w_guess = np.array([0.3, 0.6, 0.8, 1.1, 0, 0, 0, 0, 0.3, 0.2, 0.8, 0.3])
    return dict(model=model, cost=cost, C=C, c=cc, w_guess=w_guess, period=1, N=20, term_idx=[1, 2, 4, 5, 6, 7, 8])


def awe9():
    """SYNTHETIC stand-in for config #5 (examples/awe_system: nx = 9, nu = 3, ns = 3, nsc = 3, 14 rows of h before the soft-
    constraint slacks, N = 20, p = 40, 7-row projected terminal constraint x[1:3], x[4:]; SURVEY.md 8.0 / App. B) -- the
    reference's kite model is an opaque CasADi pickle.  Dynamics of `dims9`; three NONLINEAR path constraints (one of them
    state-only) that `preprocessing.input_formatting` would slack into g = h_nl(x,u) - us = 0, us >= 0
    (tunempc/preprocessing.py:78-118); eleven linear rows; `add_mpc_slacks(..., 'active')` (preprocessing.py:120-155) softens
    the three rows that are active somewhere along the reference.  The periodic reference is a forced periodic response of
    the model (inputs riding two bounds and one nonlinear constraint), tracked with a user tuning -- create_mpc('tracking')."""
    card = dims9()
    m = card["model"]
    p, v, a, u = m.x[0:4], m.x[4:8], m.x[8], m.u
    gnl = [12.0 - p[3] ** 2 - 0.5 * v[3] ** 2,                 # state only  -> gnl_x_idx = [0] (pmpc.py:1107-1114)
           1.25 - u[0] * (1 + 0.3 * p[0]),
           3.0 - u[1] ** 2 - 0.5 * a ** 2]
    model = OdeModel("awe9", m.x, m.u, m.xdot, rk_steps=10, tf=0.3, cost=card["cost"], gnl=gnl, nsc=3)
    nzm, ns, nsc = 12, 3, 3
    nz = nzm + ns + nsc
    rows = []
    def row(coefs, const):
        r = np.zeros(nz)
        for idx, val in coefs:
            r[idx] = val
        rows.append((r, const))
    for j, (lo, hi) in zip((9, 10, 11), ((-1.0, 1.5), (-0.3, 2.0), (-1.5, 1.5))):      # input bounds (rows 0..5)
        row([(j, 1.0)], -lo)
        row([(j, -1.0)], hi)
    row([(8, 1.0)], 1.2)                                                               # actuator state bounds (rows 6, 7; state only)
    row([(8, -1.0)], 1.2)
    row([(9, -1.0), (0, -0.5)], 1.7)                                                   # mixed row 8: u1 + 0.5 p1 <= 1.7
    row([(7, 1.0)], 1.5)                                                               # |v4| <= 1.5 (rows 9, 10)
    row([(7, -1.0)], 1.5)
    for i in range(ns):                                                                # us >= 0 (rows 11..13; preprocessing.py:110-112)
        row([(nzm + i, 1.0)], 0.0)
    slacked = [7, 2, 12]                                                               # a <= 1.2, u2 >= -0.3, us_1 >= 0: active on the reference
    for j, i in enumerate(slacked):                                                    # h_i + usc_j >= 0 (preprocessing.py:140-150)
        rows[i][0][nzm + ns + j] = 1.0
    for j in range(nsc):                                                               # usc >= 0 (rows 14..16)
        row([(nzm + ns + j, 1.0)], 0.0)
    C = np.array([r for r, _ in rows])
    cc = np.array([c0 for _, c0 in rows])
    return dict(model=model, cost=card["cost"], C=C, c=cc, period=40, N=20, term_idx=[1, 2, 4, 5, 6, 7, 8], slacked=slacked,
                gnl_x_idx=[0], w_guess=card["w_guess"])


def awe9_problem(stage_F, N=None, hessian_approximation="exact", mpc_type="tuned"):
    """Reference trajectory, tuning and multipliers of the awe9 stand-in (see `awe9`): simulate the forced response until it is
    periodic, then pick multipliers on the active rows and the gradient q that makes the reference a KKT point.

    mpc_type='economic' mirrors `make_problem`: stage cost = the card's l(x,u) (+ scost'usc), H = q = 0, exact Hessian, the same
    lam_h_ref, lam_g_ref and scost, lam_dyn_ref = 0.  That is a problem of the shape of the paper's AWE economic MPC (nx 9, nu 3,
    ns 3, nsc 3, N 20, p 40, exact Hessian of a non-tracking cost).  It is not an economic optimum: the reference stays the
    forced periodic response, so the controller does not return u_ref at x_ref."""
    import sympy as sp
    from .problem import MpcProblem
    cfg = awe9()
    model = cfg["model"]
    nx, nu, ns, nsc, P = 9, 3, 3, 3, cfg["period"]
    nzm, nzr = nx + nu, nx + nu + ns
    z = list(model.x) + list(model.u)
    gf = sp.lambdify([z], sp.Matrix(model.gnl), "numpy")
    gj = sp.lambdify([z], sp.Matrix(model.gnl).jacobian(z), "numpy")
    # a+ = (1 - gam) a + gam u3 exactly (the actuator state is a decoupled linear lag)
    _, S0 = stage_F(np.zeros((1, nx)), np.zeros((1, nu)), 1)
    gam = S0[0][8, 11]
    x = np.array([0.3, 0.6, 0.8, 1.0, 0, 0, 0, 0, 0.3])
    ph = 2 * np.pi * np.arange(P) / P
    for per in range(80):
        X, U = [], []
        for k in range(P):
            u1 = min(0.75 + 0.6 * np.sin(ph[k]), 1.25 / (1 + 0.3 * x[0]))             # rides the nonlinear constraint n1
            u2 = max(0.4 * np.sin(ph[k] + 2.0), -0.3)                                  # rides its lower bound
            u3 = 0.45 + 1.0 * np.sin(ph[k] + 4.0)
            if (1 - gam) * x[8] + gam * u3 > 1.2:                                      # a rides its upper bound
                u3 = (1.2 - (1 - gam) * x[8]) / gam
            uk = np.array([u1, u2, u3])
            X.append(x.copy()); U.append(uk)
            x = stage_F(x[None, :], uk[None, :], 0)[0]
        if per > 20 and np.max(np.abs(x - X[0])) < 1e-13:
            break
    X, U = np.array(X), np.array(U)
    us = np.array([np.asarray(gf(list(np.concatenate([X[k], U[k]]))), dtype=np.float64).ravel() for k in range(P)])
    us[np.abs(us) < 1e-12] = 0.0
    wref = np.hstack([X, U, us])
    C, c = cfg["C"], cfg["c"]
    nh = C.shape[0]
    # active rows on the reference and their multipliers (CasADi sign: active lower bound -> negative)
    hval = np.array([C[:, :nzr] @ wref[k] + c for k in range(P)])
    act = np.abs(hval[:, : nh - nsc]) < 1e-9
    mu = {7: 0.5, 2: 0.3, 12: 0.4}
    lam_h = np.zeros((P, nh - nsc))
    for i, m_ in mu.items():
        lam_h[act[:, i], i] = -m_ * (1.0 + 0.25 * np.cos(ph[act[:, i]]))
    assert sorted(np.nonzero(act.any(axis=0))[0]) == sorted(cfg["slacked"]), np.nonzero(act.any(axis=0))[0]
    lam_g = np.zeros((P, ns))
    lam_g[:, 1] = lam_h[:, 12]                                # d/d us_1:  -lam_g + lam_(us>=0) = 0
    q = np.zeros((P, nzr))
    for k in range(P):
        Jg = np.asarray(gj(list(wref[k, :nzm])), dtype=np.float64).reshape(ns, nzm)
        q[k, :nzm] = -(Jg.T @ lam_g[k] + C[: nh - nsc, :nzm].T @ lam_h[k])
    scost = np.array([1e3 * np.max(-lam_h[:, i]) for i in cfg["slacked"]])            # preprocessing.py:145
    # tuning: positive definite, phase dependent
    d0 = np.array([2, 2, 2, 4, .5, .5, .5, .5, .2, .2, .2, .1, .05, .05, .05])
    vv = np.cos(0.7 * np.arange(nzr))
    H = np.array([(1 + 0.2 * np.sin(ph[k])) * np.diag(d0) + 0.02 * np.outer(vv, vv) for k in range(P)])
    xs, Ss = stage_F(X, U, 1)
    N = cfg["N"] if N is None else N
    pb = MpcProblem(name="awe9", nx=nx, nu=nu, N=N, p=P, wref=wref, H=H, q=q, C=C, c=c, lam_h_ref=lam_h,
                    lam_dyn_ref=np.zeros((P, nx)), term_idx=list(cfg["term_idx"]), S_A=np.array(Ss[:, :, :nx]),
                    S_B=np.array(Ss[:, :, nx:]), hessian_approximation=hessian_approximation, mpc_type="tuned",
                    ns=ns, nsc=nsc, scost=scost, lam_g_ref=lam_g, gnl_x_idx=list(cfg["gnl_x_idx"]))
    if mpc_type == "economic":
        pb.mpc_type = "economic"
        pb.hessian_approximation = "exact"
        pb.H = np.zeros_like(pb.H)
        pb.q = np.zeros_like(pb.q)
    info = {"cfg": cfg, "periodicity_error": float(np.max(np.abs(x - X[0]))), "active": act, "hval": hval}
    return pb, info


def dims9g():
    """SYNTHETIC: `dims9` with three NONLINEAR path constraints next to its 14 linear rows -- what `preprocessing.input_formatting`
    (tunempc/preprocessing.py:35-118) turns into slacks us, rows g = h_nl(x,u) - us = 0 and rows us >= 0.  The first one (state
    only) is active at the economic steady state.  Exercises `Tuner(...).solve_ocp().convexify().create_mpc('tuned')` with
    nonlinear rows (steady-state OCP, sensitivities and convexification in the slack form)."""
    import dataclasses
    card = dims9()
    m = card["model"]
    p, v, a, u = m.x[0:4], m.x[4:8], m.x[8], m.u
    gnl = (1.1 - p[3] ** 2 - 0.5 * v[3] ** 2, 0.5 - u[0] * (1 + 0.3 * p[0]), 0.5 - u[1] ** 2 - 0.5 * a ** 2)
    card["model"] = dataclasses.replace(m, name="dims9g", gnl=gnl, hess_nz=[])
    C, c = card["C"], card["c"]
    ns = len(gnl)
    card["C"] = np.block([[C, np.zeros((C.shape[0], ns))], [np.zeros((ns, C.shape[1])), np.eye(ns)]])
    card["c"] = np.concatenate([c, np.zeros(ns)])
    return card


def evaporation_sc1():
    """examples/evaporation_process with `create_mpc(..., opts={'slack_flag': 'active'})` (tuner.py:171-177): the one row that is
    active at the steady state (X2 >= 25) is softened -> the model library variant with nsc = 1"""
    from .constraints import soft_model
    card = evaporation()
    card["model"] = soft_model(card["model"], 1)
    return card


def sample_x0(name, pb, B, seed=0):
    """synthetic initial states of SURVEY.md section 8(d): the reference examples' own perturbation recipes, seeded"""
    rng = np.random.default_rng(seed)
    xs = pb.wref[0, :pb.nx]
    if name == "lq":
        return xs + rng.uniform(-1, 1, (B, pb.nx))
    if name == "cstr":
        alpha = rng.uniform(-0.1, 1.0, B)                       # examples/cstr/main.py:124
        X0 = np.tile(xs, (B, 1))
        X0[:, 0] += alpha * (1.0 - xs[0])                       # dx_diehl direction, examples/cstr/main.py:126-131
        X0[:, 1:] += 1e-2 * np.abs(xs[1:]) * rng.uniform(-1, 1, (B, pb.nx - 1))
        return X0
    if name in ("evaporation", "evaporation_sc1"):
        # X2 sits on its bound 25.0 -> perturb upward only; P2 +-1.0 (examples/evaporation_process/main.py:178-180)
        return xs + np.stack([0.5 * np.abs(rng.uniform(-1, 1, B)), 1.0 * rng.uniform(-1, 1, B)], axis=1)
    if name == "chain":
        return xs + np.array([0.5, 0.5, 0.5, 0.8, 0.8, 0.8]) * rng.uniform(-1, 1, (B, pb.nx))
    if name in ("dims9", "dims9g"):
        return xs + np.array([0.4] * 4 + [0.6] * 4 + [0.3]) * rng.uniform(-1, 1, (B, pb.nx))
    if name == "unicycle":
        return xs + np.array([0.5, 0.1, 0.0, 0.0]) * rng.uniform(-1, 1, (B, pb.nx))   # examples/unicycle/main.py:172
    if name == "awe9":
        return xs + np.array([0.15] * 4 + [0.2] * 4 + [0.1]) * rng.uniform(-1, 1, (B, pb.nx))
    raise KeyError(name)


CONFIGS = {"lq": lq, "cstr": cstr, "unicycle": unicycle, "evaporation": evaporation, "chain": chain, "dims9": dims9,
           "awe9": awe9, "evaporation_sc1": evaporation_sc1, "dims9g": dims9g}


def make_problem(name, stage_F, N=None, hessian_approximation="exact", mpc_type="tuned"):
    """Run the offline pipeline (tuning.py) for a config and return (MpcProblem, info).

    `stage_F(x, u, order)` evaluates the compiled model's one-interval map and derivatives on the host
    (product: `tunempc_b200.lib.ModelLib.stage_eval`; tests may pass the oracle's).  Mirrors what
    `Tuner(f,l,h,p).solve_ocp(w0); convexify(); create_mpc('tuned', N)` hands to `Pmpc` (tunempc/tuner.py:90-199).
    """
    from . import tuning
    from .problem import MpcProblem

    if name == "awe9":
        return awe9_problem(stage_F, N=N, hessian_approximation=hessian_approximation, mpc_type=mpc_type)
    cfg = CONFIGS[name]()
    model = cfg["model"]
    nx, nu = model.nx, model.nu
    N = cfg["N"] if N is None else N
    cost_funs = tuning.lambdify_cost(model, cfg["cost"])
    if cfg["period"] != 1:
        # periodic pipeline: Tuner(f, l, p=P).solve_ocp(w0); convexify(); create_mpc('tuned', N, opts={'p_operator': ...})
        # (examples/unicycle/main.py:95-142)
        if cfg["C"].shape[0]:
            raise NotImplementedError("periodic OCP with path constraints is not built yet")
        P = cfg["period"]
        z, lam_d, _ = tuning.solve_periodic_ocp(stage_F, cost_funs, cfg["w_guess"], nx)
        S = tuning.sensitivities_periodic(stage_F, cost_funs, z, lam_d, nx)
        Hc = tuning.convexify_periodic(S["A"], S["B"], S["H"])
        pb = MpcProblem(name=name, nx=nx, nu=nu, N=N, p=P, wref=z.copy(), H=np.array(Hc), q=np.array(S["q"]),
                        C=cfg["C"], c=cfg["c"], lam_h_ref=np.zeros((P, 0)), lam_dyn_ref=np.zeros((P, nx)),
                        term_idx=list(cfg["term_idx"]), S_A=np.array(S["A"]), S_B=np.array(S["B"]),
                        hessian_approximation=hessian_approximation)
        info = {"z_ocp": z, "lam_dyn_ocp": lam_d, "H_ocp": S["H"], "Hc": Hc, "cfg": cfg,
                "eig_H": np.array([np.linalg.eigvalsh(h) for h in S["H"]]),
                "eig_Hc": np.array([np.linalg.eigvalsh(h) for h in Hc])}
        if mpc_type == "economic":                                       # economic MPC on the periodic reference (pmpc.py:97-107,709-767)
            pb.mpc_type = "economic"
            pb.hessian_approximation = "exact"
            pb.lam_dyn_ref = np.array(lam_d).copy()
            pb.H = np.zeros_like(pb.H)
            pb.q = np.zeros_like(pb.q)
        return pb, info
    z, lam_d, lam_h = tuning.solve_steady_state(stage_F, cost_funs, cfg["C"], cfg["c"], cfg["w_guess"], nx)
    S = tuning.sensitivities(stage_F, cost_funs, cfg["C"], z, lam_d, lam_h, nx)
    Hc, dH = tuning.convexify_dare(S["A"][0], S["B"][0], S["H"][0], C_As=S["C_As"][0], scale=z)
    pb = MpcProblem(name=name, nx=nx, nu=nu, N=N, p=1, wref=z[None, :].copy(), H=Hc[None], q=S["q"][0][None, :],
                    C=cfg["C"], c=cfg["c"], lam_h_ref=lam_h[None, :], lam_dyn_ref=np.zeros((1, nx)),
                    term_idx=list(cfg["term_idx"]), S_A=np.array(S["A"]), S_B=np.array(S["B"]),
                    hessian_approximation=hessian_approximation)
    info = {"z_ss": z, "lam_dyn_ocp": lam_d, "lam_h_ocp": lam_h, "H_ocp": S["H"][0], "Hc": Hc,
            "eig_H": np.linalg.eigvalsh(S["H"][0]), "eig_Hc": np.linalg.eigvalsh(Hc), "cfg": cfg}
    if mpc_type == "economic":
        # create_mpc('economic') (tuner.py:180-182): cost = l, full OCP multipliers as dual reference, no tuning tables
        pb.mpc_type = "economic"
        pb.hessian_approximation = "exact"                               # pmpc.py:101-104
        pb.lam_dyn_ref = lam_d[None, :].copy()
        pb.H = np.zeros_like(pb.H)
        pb.q = np.zeros_like(pb.q)
    return pb, info
