"""CPU tests of the oracle (oracle/reference_port.py, oracle/stage.c) -- pins the checker itself.

The reference's own tests hold no value for Pmpc.step / Sqp.solve (SURVEY.md section 8(c)): the oracle is pinned by
an independent dense-KKT computation of the LQ feedback law, by finite differences, by KKT residuals, by two QP
solvers (the reference tree's qpOASES_e and a dense Goldfarb-Idnani), and by the committed golden outputs."""
import numpy as np
import pytest

from conftest import load_golden, load_problem

# LQ feedback gain of config #1 computed in the survey session from a dense KKT solve (SURVEY.md section 8(c))
G_LQ = np.array([-0.08241103740895, -0.188345092908991, 0.225692606094775])


@pytest.fixture(scope="module")
def rp(built):
    from oracle import reference_port
    return reference_port


def _dense_kkt_gain(pb):
    """u0 = G x0 from one dense KKT solve of the LQ tracking problem (independent of the SQP code)."""
    from tunempc_b200 import configs
    cfg = configs.lq()
    A, B = cfg["A"], cfg["B"]
    nx, nu, N = 3, 1, pb.N
    nz = nx + nu
    n = N * nz + nx
    H = np.zeros((n, n))
    for k in range(N):
        H[k * nz:(k + 1) * nz, k * nz:(k + 1) * nz] = pb.H[0]
    rows = []
    for k in range(N):
        r = np.zeros((nx, n))
        r[:, k * nz:k * nz + nx] = A
        r[:, k * nz + nx:(k + 1) * nz] = B
        r[:, (k + 1) * nz:(k + 1) * nz + nx] = -np.eye(nx)
        rows.append(r)
    r = np.zeros((nx, n)); r[:, N * nz:] = np.eye(nx); rows.append(r)          # terminal x_N = 0
    r0 = np.zeros((nx, n)); r0[:, :nx] = np.eye(nx)
    J = np.vstack([r0] + rows)
    m = J.shape[0]
    K = np.block([[H, J.T], [J, np.zeros((m, m))]])
    G = np.zeros((nu, nx))
    for i in range(nx):
        rhs = np.zeros(n + m); rhs[n + i] = 1.0
        G[:, i] = np.linalg.solve(K, rhs)[nx:nz]
    return G


def test_lq_gain_known_answer(rp):
    pb = load_problem("lq")
    G = _dense_kkt_gain(pb)
    assert np.allclose(G[0], G_LQ, atol=1e-10)
    ctrl = rp.Pmpc(pb)
    for x0 in (np.array([1.0, 0, 0]), np.array([0.3, -0.7, 0.2])):
        ctrl.reset()
        u = ctrl.step(x0)
        assert abs(u[0] - G_LQ @ x0) < 1e-10
        assert ctrl.log["iter"][-1] == 1 and ctrl.log["status"][-1] == 0      # LQ: one SQP iteration is exact


def test_lq_golden(rp):
    pb, gold = load_problem("lq"), load_golden("lq")
    assert np.allclose(gold["u0_t6"][:, 0], gold["X0"] @ G_LQ, atol=1e-9)


@pytest.mark.parametrize("name", ["lq", "cstr", "unicycle"])
def test_stage_derivatives_fd(rp, name):
    from tunempc_b200 import configs
    st = rp.StageLib(name)
    cfg = configs.CONFIGS[name]()
    rng = np.random.default_rng(3)
    wg = np.atleast_2d(cfg["w_guess"])[0]
    z = wg * (1 + 0.02 * rng.standard_normal(wg.shape)) + 0.01 * rng.standard_normal(wg.shape)
    x, u = z[:st.nx], z[st.nx:]
    xf, S, T = st.F(x, u, 2)
    for i in range(st.nz):
        h = 1e-6 * max(1.0, abs(z[i]))
        zp, zm = z.copy(), z.copy()
        zp[i] += h; zm[i] -= h
        fp, Sp, _ = st.F(zp[:st.nx], zp[st.nx:], 2)
        fm, Sm, _ = st.F(zm[:st.nx], zm[st.nx:], 2)
        assert np.allclose((fp[0] - fm[0]) / (2 * h), S[0][:, i], rtol=1e-6, atol=1e-8)
        assert np.allclose((Sp[0] - Sm[0]) / (2 * h), T[0][:, :, i], rtol=1e-5, atol=1e-7)
    assert np.allclose(T[0], np.transpose(T[0], (0, 2, 1)), atol=1e-12)


def test_stage_vs_sympy_rk4(rp):
    """generated C + C integrator against a numpy RK4 over sympy-lambdified f (independent code path)"""
    from tunempc_b200 import configs, modelgen
    cfg = configs.cstr()
    ff, _ = modelgen.lambdify_ode(cfg["model"])
    z = cfg["w_guess"].copy()
    x, u = z[:4].copy(), z[4:]
    h = cfg["model"].tf / cfg["model"].rk_steps
    f = lambda xx: np.array(ff(np.concatenate([xx, u]))).ravel()
    for _ in range(cfg["model"].rk_steps):
        k1 = f(x); k2 = f(x + h / 2 * k1); k3 = f(x + h / 2 * k2); k4 = f(x + h * k3)
        x = x + h / 6 * (k1 + 2 * k2 + 2 * k3 + k4)
    xf = rp.StageLib("cstr").F(z[:4], z[4:])
    assert np.allclose(xf[0], x, rtol=1e-12)
    assert np.max(np.abs(xf[0] - z[:4])) < 1e-4      # cstr_model.py:168 is a near-steady state (SURVEY 8(c) KAT 3)


def test_qp_solvers_agree(rp):
    if not rp.qpoases_available():
        pytest.skip("oracle/_ref not built")
    rng = np.random.default_rng(0)
    for trial in range(5):
        n, me, mi = 12, 4, 10
        M = rng.standard_normal((n, n)); H = M @ M.T + 0.1 * np.eye(n)
        g = rng.standard_normal(n)
        A = rng.standard_normal((me + mi, n))
        x_feas = rng.standard_normal(n)
        lba = A @ x_feas; uba = lba.copy()
        lba[me:] -= rng.uniform(0, 1, mi); uba[me:] = np.inf
        d1, l1 = rp.qp_qpoases(H, g, A, lba, uba)
        d2, l2 = rp.qp_dense(H, g, A, lba, uba)
        assert np.allclose(d1, d2, atol=1e-8) and np.allclose(l1, l2, atol=1e-7)
        assert np.linalg.norm(H @ d2 + g + A.T @ l2, np.inf) < 1e-9          # CasADi sign convention
        assert np.all(l2[me:] <= 1e-12)                                        # lower-active => negative
        assert set(np.nonzero(l1[me:])[0]) == set(np.nonzero(l2[me:])[0])


def test_qp_dense_semidefinite_known_answer(rp):
    """min 1/2 x^2 + 2 s  s.t.  y - x = 0, x + s >= 1, s >= 0 over (x, y, s): no curvature in y and s, so the reduced Hessian
    is only semidefinite.  Answer by hand: x = y = 1, s = 0; lam = (0, -1, -1) (lower-active => negative)."""
    H = np.diag([1.0, 0.0, 0.0])
    g = np.array([0.0, 0.0, 2.0])
    A = np.array([[-1.0, 1.0, 0.0], [1.0, 0.0, 1.0], [0.0, 0.0, 1.0]])
    lba, uba = np.array([0.0, 1.0, 0.0]), np.array([0.0, np.inf, np.inf])
    info = {}
    d, lam = rp.qp_dense(H, g, A, lba, uba, info=info)
    assert info["branch"] == "psd"
    assert np.allclose(d, [1.0, 1.0, 0.0], atol=1e-12) and np.allclose(lam, [0.0, -1.0, -1.0], atol=1e-12)


def test_qp_dense_held_rows_known_answer(rp):
    """min 1/2 (d1^2 - d2^2 + d3^2) + 2 d2  s.t.  d3 - d1 = 0, d2 >= 1, d1 + d2 >= -5: negative curvature in d2, so the QP is
    not convex on the null space of its equality row and is unbounded below.  With d2 >= 1 held (its multiplier in the hint)
    the local minimiser on that face is d = (0, 1, 0), lam = (0, -1, 0): f'(d2 = 1) = 1 > 0 keeps the row active."""
    H = np.diag([1.0, -1.0, 1.0])
    g = np.array([0.0, 2.0, 0.0])
    A = np.array([[-1.0, 0.0, 1.0], [0.0, 1.0, 0.0], [1.0, 1.0, 0.0]])
    lba, uba = np.array([0.0, 1.0, -5.0]), np.array([0.0, np.inf, np.inf])
    with pytest.raises(rp.NonConvexQP):
        rp.qp_dense(H, g, A, lba, uba)                                      # no held rows: no convex face to start from
    info = {}
    d, lam = rp.qp_dense(H, g, A, lba, uba, lam_hint=np.array([0.0, -0.5, 0.0]), info=info)
    assert info["branch"] == "held"
    assert np.allclose(d, [0.0, 1.0, 0.0], atol=1e-12) and np.allclose(lam, [0.0, -1.0, 0.0], atol=1e-12)


def test_qp_dense_rejects_saddle_point(rp):
    """min 1/2 (d1^2 - d2^2)  s.t.  d2 >= 0 with d2 >= 0 held: d = 0 is a KKT point (zero multiplier) but a saddle point --
    d2 > 0 decreases the objective -- and is not returned."""
    with pytest.raises(rp.NonConvexQP):
        rp.qp_dense(np.diag([1.0, -1.0]), np.zeros(2), np.array([[0.0, 1.0]]), np.array([0.0]), np.array([np.inf]),
                    lam_hint=np.array([-1.0]))


@pytest.mark.parametrize("name,idx,branch", [("evaporation_sc1", (0, 5, 11), "psd"), ("awe9", (0,), "psd"),
                                             ("cstr", (4, 5), "held")])
def test_dense_qp_branches_vs_qpoases_golden(rp, name, idx, branch):
    """The dense QP solver's semidefinite and held-row branches against the reference's qpOASES_e: the golden fixtures were
    computed by this oracle with qpOASES_e as its QP solver.  Soft-constrained evaporation and awe9 (slack columns without
    curvature) take the semidefinite branch in every QP; these CSTR instances reach QPs that are not convex on the null space of the
    equality rows.  Converged point, multipliers and active set match; the iteration count too wherever no iteration was
    re-solved with the Gauss-Newton Hessian."""
    pb, gold = load_problem(name), load_golden(name)
    oc = rp.Pmpc(pb, qp="dense")
    for b in idx:
        oc.reset()
        u = oc.step(gold["X0"][b])
        br = oc.sqp.stats["qp_branches"]
        assert br[branch] > 0 and oc.log["status"][-1] == 0, (b, br)
        assert np.max(np.abs(u - gold["u0_t6"][b]) / np.maximum(np.abs(gold["u0_t6"][b]), 1.0)) < 1e-7
        assert np.max(np.abs(oc.w_sol - gold["w_t6"][b]) / np.maximum(np.abs(gold["w_t6"][b]), 1.0)) < 1e-7
        assert np.max(np.abs(oc.lam_g - gold["lam_t6"][b]) / np.maximum(np.abs(gold["lam_t6"][b]), 1.0)) < 1e-5
        assert set(np.nonzero(oc.lam_g)[0]) == set(np.nonzero(gold["lam_t6"][b])[0]) and oc.log["nAS"][-1] == gold["nAS_t6"][b]
        if br["gn_resolve"] == 0:
            assert oc.log["iter"][-1] == gold["iter_t6"][b]


def test_cstr_reference_point_and_idempotence(rp):
    pb = load_problem("cstr")
    ctrl = rp.Pmpc(pb)
    u = ctrl.step(pb.wref[0, :4])                      # P1: step(x_ref) = u_ref
    assert np.allclose(u, pb.wref[0, 4:], rtol=1e-9) and ctrl.log["iter"][-1] == 1
    gold = load_golden("cstr")
    ctrl.reset(); u1 = ctrl.step(gold["X0"][3])
    ctrl.reset(); u2 = ctrl.step(gold["X0"][3])        # P5: reset-then-step is idempotent
    assert np.array_equal(u1, u2)
    assert np.allclose(u1, gold["u0_t6"][3], rtol=1e-9)
    # P4: KKT residuals of the converged point
    assert ctrl.sqp.stats["dual_infeas"] < 1e-6 and ctrl.sqp.stats["filter"][-1, 1] < 1e-6
    lam_h = np.array([ctrl.lam_g[pb.g_h(k)] for k in range(pb.N)])
    assert np.all(lam_h <= 0)
    gh = np.array([ctrl.g_sol[pb.g_h(k)] for k in range(pb.N)])
    assert gh.min() > -1e-6 and np.all(np.abs(gh[lam_h != 0]) < 1e-6)          # complementarity


def test_hessian_mode_independence(rp):
    """P3: the converged point does not depend on the Hessian approximation"""
    pb, gold = load_problem("cstr"), load_golden("cstr")
    a = rp.Pmpc(pb, sqp_options={"tol": 1e-9})
    b = rp.Pmpc(pb, sqp_options={"tol": 1e-9, "hessian_approximation": "gauss_newton", "max_iter": 400})
    x0 = gold["X0"][7]
    ua, ub = a.step(x0), b.step(x0)
    assert np.allclose(ua, ub, rtol=1e-7)
    assert np.allclose(a.w_sol, b.w_sol, rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("name", ["cstr", "evaporation", "cstr_economic"])
def test_oracle_solution_vs_independent_nlp_solver(rp, name):
    """Pin of the oracle's ANSWERS by an independent solver: the same NLP (tunempc/pmpc.py:162-369) handed to scipy's
    SLSQP -- a different algorithm (quasi-Newton SQP with its own least-squares QP) and different code -- started 1e-3
    away from the oracle's answer (from the reference SLSQP stalls on the evaporation problem); the local minimiser it
    converges to must be the oracle's point, to SLSQP's own accuracy.  (The iteration path of Sqp.solve is pinned by nothing but the
    restatement itself: 'parity unpinned', SURVEY.md 8(c).)"""
    import scipy.optimize as sopt
    from conftest import load_golden, load_problem
    pb, gold = load_problem(name), load_golden(name)
    cf = None
    if pb.mpc_type == "economic":
        from tunempc_b200 import configs, tuning
        card = configs.CONFIGS[pb.name]()
        cf = tuning.lambdify_cost(card["model"], card["cost"])
    oc = rp.Pmpc(pb, cost_funs=cf)
    nlp, tab = oc.nlp, oc.tab
    eq = np.where(nlp.ubg - nlp.lbg == 0)[0]
    iq = np.where((nlp.ubg - nlp.lbg != 0) & np.isfinite(nlp.lbg))[0]
    scale = np.maximum(np.abs(tab.ref[0]), 1.0)
    for b in (0, 3, 5):
        p0 = {"x0": gold["X0"][b], "wref": tab.ref[0], "H": tab.Href[0], "q": tab.qref[0]}
        cons = [{"type": "eq", "fun": lambda y: nlp.g(y * scale, p0)[eq], "jac": lambda y: nlp.g(y * scale, p0, order=1)[1][eq] * scale[None, :]},
                {"type": "ineq", "fun": lambda y: nlp.g(y * scale, p0)[iq], "jac": lambda y: nlp.g(y * scale, p0, order=1)[1][iq] * scale[None, :]}]
        res = sopt.minimize(lambda y: nlp.f(y * scale, p0), gold["w_t9"][b] / scale * (1 + 1e-3) + 1e-3,
                            jac=lambda y: nlp.jacf(y * scale, p0) * scale, constraints=cons, method="SLSQP",
                            options={"ftol": 1e-15, "maxiter": 400})
        w = res.x * scale
        assert np.abs(nlp.g(w, p0)[eq]).max() < 1e-5
        err = np.max(np.abs(w - gold["w_t9"][b]) / np.maximum(np.abs(gold["w_t9"][b]), 1.0))
        assert err < 1e-4, (name, b, err, res.message)                      # SLSQP's own accuracy
        assert abs(nlp.f(w, p0) - nlp.f(gold["w_t9"][b], p0)) < 1e-4 * max(1.0, abs(nlp.f(w, p0)))   # no better point nearby
