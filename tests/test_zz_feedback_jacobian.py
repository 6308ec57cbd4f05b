"""Feedback Jacobian du0/dx0 on the GPU (tmpc_feedback_jacobian / Pmpc.feedback_jacobian): the device against the CPU twin on the
device's own solutions with every QP kernel dispatch, against the dense KKT Jacobian, the large seeded fixtures, tuned against
economic at the reference, the API errors, the asynchronous step, and the absence of side effects on the controller."""
import copy
import os

import numpy as np
import pytest

from conftest import load_golden, load_problem
from feedback_jacobian_support import FIXTURES, twin_feedback_jacobian, dense_kkt_jacobian, oracle_nlp, relerr

pytestmark = pytest.mark.gpu

CONFIGS = FIXTURES + ["dims9g"]


@pytest.fixture(scope="module")
def torch_mod(built):
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


@pytest.fixture(scope="module")
def dims9g(built):
    from economic_slack_support import economic_problem
    from tunempc_b200.lib import build_model_lib
    pb, _, _ = economic_problem("dims9g")                              # writes gen/model_dims9g.h
    build_model_lib("dims9g")                                          # not among the prebuilt libraries
    return pb


def _problem(name, dims9g):
    return dims9g if name == "dims9g" else load_problem(name)


def _states(name, pb):
    if name == "dims9g":
        from economic_slack_support import initial_states
        return initial_states("dims9g", pb, 8)
    return load_golden(name)["X0"][:8]


def _ctrl(pb, **kw):
    from tunempc_b200.pmpc import Pmpc
    pb = copy.copy(pb)
    for k, v in kw.items():
        setattr(pb, k, v)
    return Pmpc(pb, device=0)


def _twin_on(pb, X0, w, lam, st, tol):
    """the twin's Jacobian at the device's solutions (it linearises them again itself)"""
    from tunempc_b200.problem import build_tables
    from twin.twin import Twin
    tw = Twin(pb, build_tables(pb))
    return twin_feedback_jacobian(tw, X0, {"w": w, "lam": lam, "status": st}, tol=tol, phase=0)


@pytest.mark.parametrize("qpmode", [None, "t", "w"])
@pytest.mark.parametrize("name", CONFIGS)
def test_device_vs_twin(torch_mod, dims9g, name, qpmode, monkeypatch):
    """equal jstatus and J to 1e-8 against the twin on the same solutions, with the default dispatch and each kernel forced; the
    jstatus-0 instances also against the dense KKT Jacobian of the oracle's NLP"""
    torch = torch_mod
    from tunempc_b200.problem import build_tables
    if qpmode is not None:
        monkeypatch.setenv("TMPC_QP_MODE", qpmode)
        monkeypatch.setenv("TMPC_QP_THREAD_MIN", "1")
    pb = _problem(name, dims9g)
    X0 = _states(name, pb)
    tol = 1e-10
    ctrl = _ctrl(pb, tol=tol)
    ctrl.step(torch.tensor(X0, device="cuda:0"))
    J, js = ctrl.feedback_jacobian()
    assert J.shape == (len(X0), pb.nu, pb.nx) and J.is_cuda and js.is_cuda
    J, js = J.cpu().numpy(), js.cpu().numpy()
    st = ctrl.status.cpu().numpy()
    w, lam = ctrl.w_sol.cpu().numpy(), ctrl.lam_g.cpu().numpy()
    Jt, jst = _twin_on(pb, X0, w, lam, st, tol)
    assert np.array_equal(js, jst), (js, jst)
    assert (js[st != 0] == 2).all() and np.isnan(J[st != 0]).all()
    ok = js <= 1
    assert ok.sum() >= len(X0) // 2, (st, js)
    assert relerr(J[ok], Jt[ok]) < 1e-8
    if name == "dims9g":
        return                                           # the oracle NLP of dims9g needs the Tuner's cost; test_feedback_jacobian covers it
    nlp, tab = oracle_nlp(pb), build_tables(pb)
    for b in np.nonzero(js == 0)[0]:
        assert relerr(J[b], dense_kkt_jacobian(nlp, pb, tab, X0[b], w[b], lam[b])) < 1e-8, b


@pytest.mark.parametrize("name", ["cstr", "awe9"])
def test_large_fixture(torch_mod, name, capsys):
    """every instance of the large seeded fixture: the status histogram, and a prefix against the twin"""
    torch = torch_mod
    from tunempc_b200 import configs
    pb = load_problem(name)
    L = np.load(os.path.join(os.path.dirname(__file__), "golden", "large_%s.npz" % name))
    X0 = configs.sample_x0(name, pb, int(L["B"]), int(L["seed"]))
    ctrl = _ctrl(pb)
    ctrl.step(torch.tensor(X0, device="cuda:0"))
    J, js = ctrl.feedback_jacobian()
    J, js = J.cpu().numpy(), js.cpu().numpy()
    st = ctrl.status.cpu().numpy()
    hist = np.bincount(js, minlength=4)
    with capsys.disabled():
        print("\n%s B=%d jstatus histogram (ok, weak, not solved, singular): %s" % (name, len(X0), hist.tolist()))
    assert hist[0] >= len(X0) // 2 and (js[st != 0] == 2).all() and np.isfinite(J[js <= 1]).all()
    n = 64
    Jt, jst = _twin_on(pb, X0[:n], ctrl.w_sol.cpu().numpy()[:n], ctrl.lam_g.cpu().numpy()[:n], st[:n], pb.tol)
    assert np.array_equal(js[:n], jst)
    ok = jst <= 1
    assert relerr(J[:n][ok], Jt[ok]) < 1e-8


def test_tuned_vs_economic_gpu(torch_mod):
    """the tuned and the economic controller's Jacobians at x_ref on the device (CSTR; measured 1.9e-14 on the twin)"""
    torch = torch_mod
    pt, pe = load_problem("cstr"), load_problem("cstr_economic")
    xs = torch.tensor(pt.wref[0, :pt.nx][None, :], device="cuda:0")
    out = []
    for pb in (pt, pe):
        c = _ctrl(pb, tol=1e-10)
        c.step(xs)
        J, js = c.feedback_jacobian()
        assert js.cpu().numpy()[0] == 0
        out.append(J.cpu().numpy()[0])
    assert np.max(np.abs(out[0] - out[1])) < 1e-10 * np.max(np.abs(out[1]))


def test_api_errors(torch_mod):
    """before the first step, after reset, while a step is in flight, on a Gauss-Newton controller: RuntimeError; B = 0: empty"""
    torch = torch_mod
    pb = load_problem("cstr")
    X0 = torch.tensor(load_golden("cstr")["X0"][:4], device="cuda:0")
    ctrl = _ctrl(pb)
    with pytest.raises(RuntimeError, match="no step has finished"):
        ctrl.feedback_jacobian()
    ctrl.step(X0)
    J, js = ctrl.feedback_jacobian()
    assert J.shape == (4, pb.nu, pb.nx)
    ctrl.reset()
    with pytest.raises(RuntimeError, match="no step has finished"):
        ctrl.feedback_jacobian()
    ctrl.step_async(X0)
    with pytest.raises(RuntimeError, match="in flight"):
        ctrl.feedback_jacobian()
    ctrl.wait()
    ctrl.feedback_jacobian()
    gn = copy.copy(pb)
    gn.hessian_approximation = "gauss_newton"
    cg = _ctrl(gn)
    cg.step(X0)
    with pytest.raises(RuntimeError, match="exact Hessian"):
        cg.feedback_jacobian()
    c0 = _ctrl(pb)
    c0.step(np.zeros((0, pb.nx)))
    J0, js0 = c0.feedback_jacobian()
    assert J0.shape == (0, pb.nu, pb.nx) and js0.shape == (0,)
    # numpy and single-state steps: host arrays, (nu, nx) and an int
    cn = _ctrl(pb)
    Xn = load_golden("cstr")["X0"][:4]
    cn.step(Xn)
    Jn, jsn = cn.feedback_jacobian()
    assert isinstance(Jn, np.ndarray) and np.array_equal(Jn, J.cpu().numpy(), equal_nan=True)
    cn.reset()
    cn.step(Xn[0])
    J1, js1 = cn.feedback_jacobian()
    assert J1.shape == (pb.nu, pb.nx) and isinstance(js1, int)


def test_async_bitwise(torch_mod):
    """after step_async + wait the Jacobian is bitwise the synchronous one"""
    torch = torch_mod
    pb = load_problem("awe9")
    X0 = torch.tensor(load_golden("awe9")["X0"], device="cuda:0")
    a, s = _ctrl(pb), _ctrl(pb)
    for _ in range(2):
        a.step_async(X0)
        a.wait()
        s.step(X0)
        Ja, jsa = a.feedback_jacobian()
        Js, jss = s.feedback_jacobian()
        assert torch.equal(jsa, jss) and np.array_equal(Ja.cpu().numpy(), Js.cpu().numpy(), equal_nan=True)


@pytest.mark.parametrize("name", ["cstr", "awe9"])
def test_no_side_effects(torch_mod, name):
    """two controllers on the same three-step closed loop, one calling feedback_jacobian() after every step: u0, w, status,
    iterations and the log stay bitwise equal"""
    torch = torch_mod
    pb = load_problem(name)
    X = torch.tensor(load_golden(name)["X0"], device="cuda:0")
    a, b = _ctrl(pb), _ctrl(pb)
    for _ in range(3):
        Ua, Ub = a.step(X), b.step(X)
        a.feedback_jacobian()
        assert torch.equal(Ua, Ub) and torch.equal(a.w_sol, b.w_sol) and torch.equal(a.status, b.status)
        for key in ("iter", "f", "nAS", "nACtot", "nAC", "flags"):
            assert torch.equal(a.log[key][-1], b.log[key][-1]), key
        assert a.index == b.index
        X = a.plant_step(X, Ua)
        assert a.counters() == b.counters()
