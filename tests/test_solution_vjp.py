"""Solution VJP G = v_u0' du0/dx0 + v_w' dw/dx0 (tm_solution_vjp) on the CPU twin: against the twin's feedback Jacobian, against
the forward and the adjoint form of an independent dense KKT solve with the oracle's NLP classes, against central differences of
twin solves, and the per-instance statuses."""
import copy

import numpy as np
import pytest

from conftest import load_golden, load_problem
from feedback_jacobian_support import active_set, twin_feedback_jacobian
from solution_vjp_support import FIXTURES, dense_kkt_adjoint, dense_kkt_dw_dx0, oracle_nlp, relerr, twin_solution_vjp

CONFIGS = FIXTURES + ["dims9g"]


def _twin(pb):
    from tunempc_b200.problem import build_tables
    from twin.twin import Twin
    return Twin(pb, build_tables(pb))


def _problem_states(name, B=8):
    if name == "dims9g":
        from economic_slack_support import economic_problem, initial_states
        pb, _, _ = economic_problem("dims9g")                         # writes gen/model_dims9g.h
        return pb, initial_states("dims9g", pb, B)
    return load_problem(name), load_golden(name)["X0"][:B]


def _solve(pb, X0, tol):
    tw = _twin(pb)
    X0 = np.atleast_2d(np.asarray(X0, dtype=np.float64))
    tw.reset(len(X0))
    return tw, tw.step(X0, tol=tol)


@pytest.mark.parametrize("name", CONFIGS)
def test_against_jacobian(built, name):
    """a cotangent on u0 alone: G = v' J with the twin's feedback Jacobian, to 1e-10, and the same jstatus"""
    pb, X0 = _problem_states(name)
    tw, o = _solve(pb, X0, 1e-10)
    J, js = twin_feedback_jacobian(tw, X0, o, tol=1e-10)
    v = np.random.default_rng(1).standard_normal((len(X0), pb.nu))
    G, gs = twin_solution_vjp(tw, o, v_u0=v, tol=1e-10)
    assert np.array_equal(gs, js), (gs, js)
    ok = js <= 1
    assert ok.sum() >= len(X0) // 2, js
    ref = np.einsum("bij,bi->bj", J, v)
    assert relerr(G[ok], ref[ok]) < 1e-10, relerr(G[ok], ref[ok])
    assert np.isnan(G[~ok]).all()


@pytest.mark.parametrize("name", FIXTURES)
def test_dense_kkt(built, name):
    """a cotangent on the whole w (and one on u0 with it): v' dw/dx0 from the dense forward solve (nx right-hand sides) and from
    the dense adjoint K [y; mu] = [v; 0], on every jstatus-0 instance, to 1e-8"""
    from tunempc_b200.problem import build_tables
    pb, X0 = _problem_states(name)
    tab = build_tables(pb)
    tw, o = _solve(pb, X0, 1e-10)
    rng = np.random.default_rng(2)
    vw = rng.standard_normal((len(X0), pb.n_w))
    vu = rng.standard_normal((len(X0), pb.nu))
    G, gs = twin_solution_vjp(tw, o, v_w=vw, tol=1e-10)
    G2, _ = twin_solution_vjp(tw, o, v_u0=vu, v_w=vw, tol=1e-10)
    nlp = oracle_nlp(pb)
    ok = np.nonzero(gs == 0)[0]
    assert len(ok) >= len(X0) // 2, gs
    for b in ok:
        D = dense_kkt_dw_dx0(nlp, pb, tab, X0[b], o["w"][b], o["lam"][b])
        fwd = vw[b] @ D
        adj = dense_kkt_adjoint(nlp, pb, tab, X0[b], o["w"][b], o["lam"][b], vw[b])
        assert relerr(adj, fwd) < 1e-8, (b, relerr(adj, fwd))
        assert relerr(G[b], fwd) < 1e-8, (name, b, relerr(G[b], fwd))
        assert relerr(G2[b], fwd + vu[b] @ D[pb.iu(0)]) < 1e-8, (name, b)


@pytest.mark.parametrize("name", ["cstr", "evaporation", "unicycle_economic"])
def test_finite_differences(built, name):
    """central differences of v' w*(x0) with twin solves at tol 1e-12, on the instances whose active set is the same at x0 +- h e_j"""
    pb = load_problem(name)
    X0 = load_golden(name)["X0"][:4]
    tw, o = _solve(pb, X0, 1e-12)
    B, nx, h = len(X0), pb.nx, 1e-5
    v = np.random.default_rng(3).standard_normal((B, pb.n_w))
    G, gs = twin_solution_vjp(tw, o, v_w=v, tol=1e-12)
    scale = np.maximum(np.abs(pb.wref[0, :nx]), 1.0)
    Xp = np.concatenate([X0 + h * scale[j] * np.eye(nx)[j] for j in range(nx)])
    Xm = np.concatenate([X0 - h * scale[j] * np.eye(nx)[j] for j in range(nx)])
    _, op = _solve(pb, Xp, 1e-12)
    _, om = _solve(pb, Xm, 1e-12)
    n = 0
    for j in range(nx):
        for b in range(B):
            s = j * B + b
            a0 = active_set(pb, o["lam"][b])
            if gs[b] != 0 or op["status"][s] or om["status"][s]:
                continue
            if not (np.array_equal(active_set(pb, op["lam"][s]), a0) and np.array_equal(active_set(pb, om["lam"][s]), a0)):
                continue
            fd = v[b] @ (op["w"][s] - om["w"][s]) / (2 * h * scale[j])
            assert abs(fd - G[b, j]) < 1e-6 * max(1.0, np.max(np.abs(G[b]))), (name, b, j, fd, G[b, j])
            n += 1
    assert n >= nx * B // 2


def test_input_bound_on_u0(built):
    """CSTR: a cotangent on an input whose bound is active at stage 0 gives G exactly zero"""
    pb = load_problem("cstr")
    X0 = load_golden("cstr")["X0"]
    tw, o = _solve(pb, X0, 1e-10)
    n = 0
    for b in range(len(X0)):
        l0 = o["lam"][b][pb.g_h(0)]
        for i in np.nonzero(l0)[0]:
            cols = np.nonzero(pb.C[i])[0]
            if len(cols) == 1 and pb.nx <= cols[0] < pb.nx + pb.nu:
                v = np.zeros((1, pb.nu))
                v[0, cols[0] - pb.nx] = 1.0
                sub = {k: o[k][b:b + 1] for k in ("w", "lam", "status")}
                G, gs = twin_solution_vjp(tw, sub, v_u0=v, tol=1e-10)
                if gs[0] == 0:
                    assert np.array_equal(G[0], np.zeros(pb.nx)), (b, i, G)
                    n += 1
    assert n > 0


def test_status_not_solved(built):
    """max_iter = 1: the steps do not converge, jstatus 2 and G NaN"""
    pb = copy.copy(load_problem("cstr"))
    pb.max_iter = 1
    X0 = load_golden("cstr")["X0"][:4]
    tw, o = _solve(pb, X0, 1e-10)
    G, gs = twin_solution_vjp(tw, o, v_u0=np.ones((4, pb.nu)), tol=1e-10)
    assert (o["status"] != 0).all() and (gs == 2).all() and np.isnan(G).all()


def test_status_weakly_active(built):
    """CSTR at the bisected point where the bound u_1 <= 35 becomes active at stage 0 (as in test_feedback_jacobian): jstatus 1
    on both sides of the switch, 0 further away, and G = v' J there"""
    pb = load_problem("cstr")
    xs = pb.wref[0, :pb.nx]
    x1 = load_golden("cstr")["X0"][0]
    row = pb.g_h(0).start + 1                                   # -u_1 + 35 >= 0

    def at(alpha):
        x = xs + alpha * (x1 - xs)
        tw, o = _solve(pb, x, 1e-10)
        assert o["status"][0] == 0
        return tw, o, x

    lo, hi = 0.0, 1.0
    while hi - lo > 1e-12:
        mid = 0.5 * (lo + hi)
        if at(mid)[1]["lam"][0][row] != 0:
            hi = mid
        else:
            lo = mid
    v = np.array([[0.3, -1.2]])
    for alpha, expect in ((lo, 1), (hi, 1), (lo - 1e-3, 0), (hi + 1e-3, 0)):
        tw, o, x = at(alpha)
        G, gs = twin_solution_vjp(tw, o, v_u0=v, tol=1e-10)
        J, js = twin_feedback_jacobian(tw, x, o, tol=1e-10)
        assert gs[0] == expect == js[0], (alpha, gs, js)
        assert relerr(G, np.einsum("bij,bi->bj", J, v)) < 1e-10


def test_cotangent_argument_check(built):
    pb = load_problem("lq")
    tw, o = _solve(pb, [[1.0, 0.0, 0.0]], 1e-8)
    with pytest.raises(ValueError):
        twin_solution_vjp(tw, o)
