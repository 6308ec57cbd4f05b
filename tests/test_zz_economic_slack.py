"""Economic MPC with slack variables on the GPU: the device against its CPU twin with every QP kernel, the device solutions as KKT
points of the oracle's NLP, the Tuner path, first-order equivalence of the tuned and the economic controller with slacks, and an
awe9 economic closed loop with the device plant step."""
import copy

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

NAMES = ["awe9", "evaporation_sc1", "dims9g"]


def _relerr(a, b):
    return np.max(np.abs(a - b) / np.maximum(np.abs(b), 1.0))


@pytest.fixture(scope="module")
def torch_mod(built):
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


@pytest.fixture(scope="module")
def problems(built):
    from economic_slack_support import economic_problem
    from tunempc_b200.lib import build_model_lib
    build_model_lib("dims9g")                                          # not among the prebuilt libraries
    return {n: economic_problem(n) for n in NAMES}


def _ctrl(pb, **kw):
    from tunempc_b200.pmpc import Pmpc
    pb = copy.copy(pb)
    for k, v in kw.items():
        setattr(pb, k, v)
    return Pmpc(pb, device=0)


@pytest.mark.parametrize("qpmode,q0min", [(None, None), ("t", None), ("w", None), (None, "2"), (None, "1000000")])
@pytest.mark.parametrize("name", NAMES)
def test_economic_slack_device_vs_twin(torch_mod, problems, name, qpmode, q0min, monkeypatch):
    """the default dispatch, each QP kernel forced (thread / warp per instance) and the shared-table first QP on and off, against
    the CPU twin of the same routines: status, iteration counts, nAS, active sets, u0 and w to 1e-8; every converged device solution
    is a KKT point of the oracle's economic NLP with slacks"""
    torch = torch_mod
    from economic_slack_support import EconomicSlackNlp, cost_funs, initial_states, kkt_error
    from tunempc_b200.problem import build_tables
    from twin.twin import Twin
    if qpmode is not None:
        monkeypatch.setenv("TMPC_QP_MODE", qpmode)
        monkeypatch.setenv("TMPC_QP_THREAD_MIN", "1")
    if q0min is not None:
        monkeypatch.setenv("TMPC_QP0_MIN", q0min)
    pb, cfg, _ = problems[name]
    tab = build_tables(pb)
    nlp = EconomicSlackNlp(pb, cost_funs(cfg))
    X0 = initial_states(name, pb)
    tw = Twin(pb, tab)
    for tol in (1e-6, 1e-9):
        tw.reset(len(X0))
        o = tw.step(X0, tol=tol, shared_first_qp=q0min == "2")
        ctrl = _ctrl(pb, tol=tol)
        U = ctrl.step(torch.tensor(X0, device="cuda:0")).cpu().numpy()
        st = ctrl.status.cpu().numpy()
        ok = st == 0
        # dims9g: x0 that make the hard nonlinear state row infeasible end as QP_Infeasible, or as Working_Set_Overflow where the
        # dual active set needs more than the default 32 rows first (DESIGN.md, tuner with nonlinear rows)
        assert np.array_equal(ok, o["status"] == 0) and set(st[~ok]) <= {2, 5}, (st, o["status"])
        assert ok.sum() >= (len(X0) * 2 // 3 if name == "dims9g" else len(X0))
        assert np.array_equal(ctrl.log["iter"][-1].cpu().numpy()[ok], o["iter"][ok])
        assert np.array_equal(ctrl.log["nAS"][-1].cpu().numpy()[ok], o["nAS"][ok])
        assert _relerr(U[ok], o["u0"][ok]) < 1e-8
        w, lam = ctrl.w_sol.cpu().numpy(), ctrl.lam_g.cpu().numpy()
        assert _relerr(w[ok], o["w"][ok]) < 1e-8
        for b in np.nonzero(ok)[0]:
            for k in range(pb.N):
                assert np.array_equal(lam[b][pb.g_h(k)] != 0, o["lam"][b][pb.g_h(k)] != 0), (b, k)
            assert kkt_error(nlp, pb, tab, X0[b], w[b], lam[b]) < tol, (tol, b)


def test_awe9_economic_closed_loop(torch_mod, problems):
    """awe9 economic (the shape of the paper's AWE EMPC) over the periodic reference with the device plant step, against the twin's
    closed loop with the oracle's model"""
    torch = torch_mod
    from oracle import reference_port as rp
    from tunempc_b200 import configs
    from tunempc_b200.problem import build_tables
    from twin.twin import Twin
    pb = problems["awe9"][0]
    X0 = configs.sample_x0("awe9", pb, 6, 5)
    tw = Twin(pb, build_tables(pb))
    tw.reset(len(X0))
    ctrl = _ctrl(pb)
    F = rp.StageLib("awe9").F
    X, x = torch.tensor(X0, device="cuda:0"), X0.copy()
    for s in range(8):
        U = ctrl.step(X)
        o = tw.step(x)
        assert (ctrl.status.cpu().numpy() == 0).all() and (o["status"] == 0).all(), s
        assert np.array_equal(ctrl.log["iter"][-1].cpu().numpy(), o["iter"]), s
        assert _relerr(U.cpu().numpy(), o["u0"]) < 1e-8, s
        X = ctrl.plant_step(X, U)
        x = F(x, o["u0"])
    assert _relerr(X.cpu().numpy(), x) < 1e-8


def test_tuner_economic_with_slacks_gpu(torch_mod, problems):
    """Tuner(...).create_mpc('economic', N[, opts={'slack_flag': 'active'}]).step(X0) on the GPU: the problem the host captured,
    status 0 on the soft-constraint states (some below the bound, absorbed by the slack), step(x_ref) = u_ref"""
    torch = torch_mod
    from economic_slack_support import initial_states
    from tunempc_b200.problem import build_tables
    for name, N, opts in (("evaporation_sc1", 30, {"slack_flag": "active"}), ("dims9g", 20, {})):
        pb0, _, t = problems[name]
        ctrl = t.create_mpc("economic", N, opts=opts)
        pb = ctrl.problem
        assert pb.name == pb0.name and pb.mpc_type == "economic"
        assert np.array_equal(build_tables(pb).ref_du, build_tables(pb0).ref_du)
        X0 = initial_states(name, pb)
        ctrl.step(torch.tensor(X0, device="cuda:0"))
        st = ctrl.status.cpu().numpy()
        assert (st == 0).all() if name == "evaporation_sc1" else set(st) <= {0, 2, 5}, st
        if name == "evaporation_sc1":
            below = X0[:, 0] < 25.0
            usc0 = ctrl.w_sol.cpu().numpy()[:, pb.iusc(0)][:, 0]
            assert np.allclose(usc0[below], 25.0 - X0[below, 0], atol=1e-8)
        ctrl.reset()
        U = ctrl.step(torch.tensor(pb.wref[0, :pb.nx][None, :], device="cuda:0")).cpu().numpy()
        atol = 1e-4 if name == "dims9g" else 1e-9                     # see tests/test_economic_slack.py (reference point)
        assert ctrl.status.cpu().numpy()[0] == 0 and np.allclose(U[0], pb.wref[0, pb.nx:pb.nx + pb.nu], rtol=0, atol=atol)


def _slopes(controllers, pt, dx, second_order=True):
    from tunempc_b200 import closed_loop_tools as clt
    xs = pt.wref[0, :pt.nx]
    alpha = np.array([0.0, 1e-3, 2e-3])
    lg = clt.check_equivalence(controllers, None, None, xs, dx, alpha)
    ut = lg["u"]["tuned"][:, 0].cpu().numpy()
    ue = lg["u"]["economic"][:, 0].cpu().numpy()
    st, se = (ut[1] - ut[0]) / alpha[1], (ue[1] - ue[0]) / alpha[1]
    assert np.max(np.abs(st - se)) < 1e-3 * np.max(np.abs(se)), (st, se)          # equal slopes; what remains is O(alpha)
    if second_order:
        d1 = np.max(np.abs((ut[1] - ut[0]) - (ue[1] - ue[0])))
        d2 = np.max(np.abs((ut[2] - ut[0]) - (ue[2] - ue[0])))
        assert 3.5 < d2 / d1 < 4.5, (d1, d2)                                     # the difference is second order in alpha


def test_first_order_equivalence_soft_constraints(torch_mod, problems):
    """closed_loop_tools.check_equivalence({'tuned', 'economic'}) with soft constraints (evaporation_sc1): equal feedback slopes
    du0/dalpha at the reference, the method and tolerance of test_gpu_parity.py::test_economic_controller"""
    t = problems["evaporation_sc1"][2]
    t.convexify(rho=1e-3)
    opts = {"slack_flag": "active"}
    ct = _ctrl(t.create_mpc("tuned", 30, opts=opts).problem, tol=1e-10)
    ce = _ctrl(t.create_mpc("economic", 30, opts=opts).problem, tol=1e-10)
    assert ct.problem.nsc == ce.problem.nsc == 1
    dx = np.zeros(2)
    dx[-1] = 1.0                                                                 # P2 (evaporation main.py:178-180)
    _slopes({"tuned": ct, "economic": ce}, ct.problem, dx)


def test_first_order_equivalence_nonlinear_rows(torch_mod, problems):
    """the same with slacked nonlinear path constraints (dims9g: the state-only nonlinear row active at the steady state): equal
    slopes.  The ratio of the differences at alpha = 2e-3 and 1e-3 was measured at 2.5 on a B200, not 4: the economic controller's
    3e-5 offset from u_ref at this steady state (tests/test_economic_slack.py) leaves a part that is not second order."""
    t = problems["dims9g"][2]
    t.convexify()
    ct = _ctrl(t.create_mpc("tuned", 20).problem, tol=1e-10)
    ce = _ctrl(t.create_mpc("economic", 20).problem, tol=1e-10)
    assert ct.problem.ns == ce.problem.ns == 3
    dx = np.zeros(9)
    dx[0] = 1.0
    _slopes({"tuned": ct, "economic": ce}, ct.problem, dx, second_order=False)
