"""Feedback Jacobian du0/dx0 (tm_feedback_jacobian) on the CPU twin: the LQ known answer, an independent dense KKT solve with the
oracle's NLP classes, finite differences of twin solves, a bound active on u_0, the tuned against the economic controller at the
reference (the first-order equivalence TuneMPC is built for, as a matrix), and the per-instance statuses."""
import copy

import numpy as np
import pytest

from conftest import load_golden, load_problem
from feedback_jacobian_support import FIXTURES, twin_feedback_jacobian, active_set, dense_kkt_jacobian, oracle_nlp, relerr

G_LQ = np.array([-0.08241103740895, -0.188345092908991, 0.225692606094775])   # tests/test_oracle.py (dense KKT of config #1)


def _twin(pb):
    from tunempc_b200.problem import build_tables
    from twin.twin import Twin
    return Twin(pb, build_tables(pb))


def _solve(pb, X0, tol):
    tw = _twin(pb)
    X0 = np.atleast_2d(np.asarray(X0, dtype=np.float64))
    tw.reset(len(X0))
    o = tw.step(X0, tol=tol)
    J, js = twin_feedback_jacobian(tw, X0, o, tol=tol)
    return J, js, o


def test_lq_known_answer(built):
    pb = load_problem("lq")
    J, js, o = _solve(pb, [[1.0, 0.0, 0.0], [0.3, -0.7, 0.2]], 1e-6)
    assert (o["status"] == 0).all() and (js == 0).all()
    assert np.max(np.abs(J[:, 0, :] - G_LQ)) < 1e-10


@pytest.mark.parametrize("name", FIXTURES)
def test_dense_kkt(built, name):
    """every jstatus-0 instance of the fixture states against the dense KKT Jacobian at the twin's solution, to 1e-8"""
    from tunempc_b200.problem import build_tables
    pb = load_problem(name)
    tab = build_tables(pb)
    X0 = load_golden(name)["X0"][:8]
    J, js, o = _solve(pb, X0, 1e-10)
    ok = np.nonzero(js == 0)[0]
    assert len(ok) >= len(X0) // 2, js
    assert set(js[o["status"] == 0]) <= {0, 1} and (js[o["status"] != 0] == 2).all()
    nlp = oracle_nlp(pb)
    for b in ok:
        Jd = dense_kkt_jacobian(nlp, pb, tab, X0[b], o["w"][b], o["lam"][b])
        assert relerr(J[b], Jd) < 1e-8, (name, b, relerr(J[b], Jd))


@pytest.mark.parametrize("name", ["cstr", "evaporation", "unicycle_economic"])
def test_finite_differences(built, name):
    """central differences of twin solves at tol 1e-12, on the instances whose active set is the same at x0 +- h e_j"""
    pb = load_problem(name)
    X0 = load_golden(name)["X0"][:4]
    J, js, o = _solve(pb, X0, 1e-12)
    nx, h = pb.nx, 1e-5
    scale = np.maximum(np.abs(pb.wref[0, :nx]), 1.0)
    Xp = np.concatenate([X0 + h * scale[j] * np.eye(nx)[j] for j in range(nx)])
    Xm = np.concatenate([X0 - h * scale[j] * np.eye(nx)[j] for j in range(nx)])
    _, _, op = _solve(pb, Xp, 1e-12)
    _, _, om = _solve(pb, Xm, 1e-12)
    B, n = len(X0), 0
    for j in range(nx):
        for b in range(B):
            s = j * B + b
            a0 = active_set(pb, o["lam"][b])
            if js[b] != 0 or op["status"][s] or om["status"][s]:
                continue
            if not (np.array_equal(active_set(pb, op["lam"][s]), a0) and np.array_equal(active_set(pb, om["lam"][s]), a0)):
                continue
            fd = (op["u0"][s] - om["u0"][s]) / (2 * h * scale[j])
            assert np.max(np.abs(fd - J[b][:, j])) < 1e-5 * max(1.0, np.max(np.abs(J[b]))), (name, b, j, fd, J[b][:, j])
            n += 1
    assert n >= nx * B // 2


def test_input_bound_on_u0(built):
    """CSTR: where an input bound (a row of C on one input) is active at stage 0, that input's row of J is exactly zero"""
    pb = load_problem("cstr")
    X0 = load_golden("cstr")["X0"]
    J, js, o = _solve(pb, X0, 1e-10)
    n = 0
    for b in range(len(X0)):
        l0 = o["lam"][b][pb.g_h(0)]
        for i in np.nonzero(l0)[0]:
            cols = np.nonzero(pb.C[i])[0]
            if len(cols) == 1 and pb.nx <= cols[0] < pb.nx + pb.nu and js[b] == 0:
                assert np.array_equal(J[b][cols[0] - pb.nx], np.zeros(pb.nx)), (b, i)
                assert np.abs(J[b]).max() > 0
                n += 1
    assert n > 0


@pytest.mark.parametrize("name", ["cstr", "evaporation"])
def test_tuned_vs_economic_fixtures(built, name):
    """paper eq. (6) as a matrix: J of the tuned and of the economic controller at x_ref.  Measured on the twin: 1.9e-14 (cstr)
    and 2.9e-15 (evaporation) relative to max |J|; the finite-difference slopes (test_gpu_parity.py) allow 1e-3"""
    pt, pe = load_problem(name), load_problem(name + "_economic")
    xs = pt.wref[0, :pt.nx]
    Jt, st, _ = _solve(pt, xs, 1e-10)
    Je, se, _ = _solve(pe, xs, 1e-10)
    assert st[0] == 0 and se[0] == 0
    assert np.max(np.abs(Jt - Je)) < 1e-10 * np.max(np.abs(Je))


@pytest.mark.parametrize("name,N,opts,rho", [("evaporation_sc1", 30, {"slack_flag": "active"}, 1e-3), ("dims9g", 20, {}, None)])
def test_tuned_vs_economic_tuner(built, name, N, opts, rho, capsys):
    """the same through the Tuner with soft constraints (evaporation_sc1) and slacked nonlinear rows (dims9g): 1e-3"""
    from economic_slack_support import economic_problem, tuner_problem
    pe, _, t = economic_problem(name)
    if rho is None:
        t.convexify()
    else:
        t.convexify(rho=rho)
    pt = tuner_problem(t, "tuned", N, opts)
    xs = pt.wref[0, :pt.nx]
    Jt, st, _ = _solve(pt, xs, 1e-10)
    Je, se, _ = _solve(pe, xs, 1e-10)
    assert st[0] in (0, 1) and se[0] in (0, 1), (st, se)
    err = np.max(np.abs(Jt - Je)) / np.max(np.abs(Je))
    with capsys.disabled():
        print("\n%s: |J_tuned - J_economic| / max|J_economic| = %.3e (jstatus %d / %d)" % (name, err, st[0], se[0]))
    assert err < 1e-3


def test_status_not_solved(built):
    """max_iter = 1: the steps do not converge, jstatus 2 and J NaN"""
    pb = copy.copy(load_problem("cstr"))
    pb.max_iter = 1
    J, js, o = _solve(pb, load_golden("cstr")["X0"][:4], 1e-10)
    assert (o["status"] != 0).all() and (js == 2).all() and np.isnan(J).all()


def test_status_weakly_active(built):
    """CSTR from x_ref towards a state whose solution holds the bound u_1 <= 35 at stage 0: at the point where that row becomes
    active (bisection in alpha to 1e-12) the Jacobian is flagged weakly active; on either side it is not"""
    pb = load_problem("cstr")
    xs = pb.wref[0, :pb.nx]
    x1 = load_golden("cstr")["X0"][0]
    row = pb.g_h(0).start + 1                                   # -u_1 + 35 >= 0

    def at(alpha):
        J, js, o = _solve(pb, xs + alpha * (x1 - xs), 1e-10)
        assert o["status"][0] == 0
        return o["lam"][0][row] != 0, int(js[0])

    lo, hi = 0.0, 1.0
    assert not at(lo)[0] and at(hi)[0]
    while hi - lo > 1e-12:
        mid = 0.5 * (lo + hi)
        if at(mid)[0]:
            hi = mid
        else:
            lo = mid
    assert at(lo)[1] == 1 and at(hi)[1] == 1
    assert at(lo - 1e-3)[1] == 0 and at(hi + 1e-3)[1] == 0
