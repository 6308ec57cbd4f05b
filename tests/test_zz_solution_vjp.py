"""Solution VJP and differentiable closed loop on the GPU (tmpc_solution_vjp / Pmpc.solution_vjp, tmpc_plant_jacobian,
tunempc_b200.autograd): the device against the CPU twin on the device's own solutions with every QP kernel dispatch and against
its own feedback Jacobian, stored solutions of earlier steps, the absence of side effects, autograd through one step and through
a closed loop against central differences, the plant Jacobian, the large seeded fixtures and the API errors."""
import copy
import os

import numpy as np
import pytest

from conftest import load_golden, load_problem
from solution_vjp_support import FIXTURES, relerr, twin_solution_vjp

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


def _problem(name, dims9g=None):
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


def _twin_on(pb, w, lam, st, tol, phase, v_u0=None, v_w=None):
    from tunempc_b200.problem import build_tables
    from twin.twin import Twin
    tw = Twin(pb, build_tables(pb))
    return twin_solution_vjp(tw, {"w": w, "lam": lam, "status": st}, v_u0=v_u0, v_w=v_w, tol=tol, phase=phase)


@pytest.mark.parametrize("qpmode", [None, "t", "w"])
@pytest.mark.parametrize("name", CONFIGS)
def test_device_vs_twin(torch_mod, dims9g, name, qpmode, monkeypatch):
    """explicit solutions with cotangents on u0 and w: equal jstatus and G to 1e-8 against the twin; the last step's own
    solutions (W == NULL) with a cotangent on u0: G = v' J with the device's feedback_jacobian() to 1e-10"""
    torch = torch_mod
    if qpmode is not None:
        monkeypatch.setenv("TMPC_QP_MODE", qpmode)
        monkeypatch.setenv("TMPC_QP_THREAD_MIN", "1")
    pb = _problem(name, dims9g)
    X0 = _states(name, pb)
    tol = 1e-10
    ctrl = _ctrl(pb, tol=tol)
    ctrl.step(torch.tensor(X0, device="cuda:0"))
    rng = np.random.default_rng(5)
    vu = torch.tensor(rng.standard_normal((len(X0), pb.nu)), device="cuda:0")
    vw = torch.tensor(rng.standard_normal((len(X0), pb.n_w)), device="cuda:0")
    G, js = ctrl.solution_vjp(v_u0=vu, v_w=vw, w=ctrl.w_sol, lam_g=ctrl.lam_g, status=ctrl.status, phase=ctrl.last_phase)
    assert G.shape == (len(X0), pb.nx) and G.is_cuda and js.is_cuda
    G, js = G.cpu().numpy(), js.cpu().numpy()
    st = ctrl.status.cpu().numpy()
    w, lam = ctrl.w_sol.cpu().numpy(), ctrl.lam_g.cpu().numpy()
    Gt, jst = _twin_on(pb, w, lam, st, tol, 0, vu.cpu().numpy(), vw.cpu().numpy())
    assert np.array_equal(js, jst), (js, jst)
    assert (js[st != 0] == 2).all() and np.isnan(G[st != 0]).all()
    ok = js <= 1
    assert ok.sum() >= len(X0) // 2, (st, js)
    assert relerr(G[ok], Gt[ok]) < 1e-8, relerr(G[ok], Gt[ok])
    J, jsj = ctrl.feedback_jacobian()
    G1, js1 = ctrl.solution_vjp(v_u0=vu)
    assert torch.equal(js1, jsj)
    ref = torch.einsum("bij,bi->bj", J, vu).cpu().numpy()
    G1 = G1.cpu().numpy()
    assert relerr(G1[ok], ref[ok]) < 1e-10, relerr(G1[ok], ref[ok])


@pytest.mark.parametrize("name", ["awe9", "unicycle_economic"])
def test_stored_solutions(torch_mod, name):
    """W == NULL equals the explicit call on the step's outputs; the VJP of step k computed after step k+3 from its saved
    solution (periodic problem: a different phase by then) equals the one computed right after step k"""
    torch = torch_mod
    pb = load_problem(name)
    X = torch.tensor(load_golden(name)["X0"][:8], device="cuda:0")
    ctrl = _ctrl(pb)
    rng = np.random.default_rng(6)
    vu = torch.tensor(rng.standard_normal((X.shape[0], pb.nu)), device="cuda:0")
    vw = torch.tensor(rng.standard_normal((X.shape[0], pb.n_w)), device="cuda:0")
    saved = []
    for k in range(5):
        U = ctrl.step(X)
        sol = dict(w=ctrl.w_sol, lam_g=ctrl.lam_g, status=ctrl.status, phase=ctrl.last_phase)
        assert sol["phase"] == k % pb.p
        Gs, jss = ctrl.solution_vjp(v_u0=vu, v_w=vw)
        Ge, jse = ctrl.solution_vjp(v_u0=vu, v_w=vw, **sol)
        assert torch.equal(jss, jse)
        ok = (jse <= 1).cpu().numpy()
        assert relerr(Gs.cpu().numpy()[ok], Ge.cpu().numpy()[ok]) < 1e-10
        saved.append((sol, Ge, jse))
        if k >= 3:
            sol0, G0, js0 = saved[k - 3]
            G3, js3 = ctrl.solution_vjp(v_u0=vu, v_w=vw, **sol0)
            assert torch.equal(js3, js0) and np.array_equal(G3.cpu().numpy(), G0.cpu().numpy(), equal_nan=True)
        X = ctrl.plant_step(X, U)


@pytest.mark.parametrize("name", ["cstr", "awe9"])
def test_no_side_effects(torch_mod, name):
    """two controllers on the same closed loop, one calling solution_vjp() (both forms) after every step: the Jacobian before
    and after is bitwise equal, and u0, w, status, the log, counters and timing stay as without the calls"""
    torch = torch_mod
    pb = load_problem(name)
    X = torch.tensor(load_golden(name)["X0"], device="cuda:0")
    a, b = _ctrl(pb), _ctrl(pb)
    vu = torch.ones((X.shape[0], pb.nu), dtype=torch.float64, device="cuda:0")
    for _ in range(3):
        Ua, Ub = a.step(X), b.step(X)
        assert torch.equal(Ua, Ub) and torch.equal(a.w_sol, b.w_sol) and torch.equal(a.status, b.status)
        J0, js0 = a.feedback_jacobian()
        cnt, tim = a.counters(), a.timing()
        a.solution_vjp(v_u0=vu)
        a.solution_vjp(v_u0=vu, v_w=a.w_sol, w=a.w_sol, lam_g=a.lam_g, status=a.status, phase=a.last_phase)
        J1, js1 = a.feedback_jacobian()
        assert torch.equal(js0, js1) and np.array_equal(J0.cpu().numpy(), J1.cpu().numpy(), equal_nan=True)
        assert a.counters() == cnt and a.timing() == tim
        for key in ("iter", "f", "nAS", "nACtot", "nAC", "flags"):
            assert torch.equal(a.log[key][-1], b.log[key][-1]), key
        assert a.index == b.index
        X = a.plant_step(X, Ua)
    assert torch.equal(a.step(X), b.step(X)) and torch.equal(a.w_sol, b.w_sol)


def _fd_ok(pb, lam0, lamp, lamm):
    from feedback_jacobian_support import active_set
    a0 = active_set(pb, lam0)
    return np.array_equal(active_set(pb, lamp), a0) and np.array_equal(active_set(pb, lamm), a0)


@pytest.mark.parametrize("name", ["cstr", "awe9"])
def test_autograd_mpc_step(torch_mod, name):
    """d/dX0 of sum(c * U0) + sum(d * W) through mpc_step against central differences of reset(); step(X0 +- h e_j) at tol
    1e-12, on the jstatus-0 instances whose active set is the same at both sides, to 1e-6 relative"""
    torch = torch_mod
    from tunempc_b200.autograd import mpc_step
    pb = load_problem(name)
    X0 = torch.tensor(load_golden(name)["X0"][:8], device="cuda:0")
    B, nx = X0.shape
    ctrl = _ctrl(pb, tol=1e-12)
    rng = np.random.default_rng(7)
    c = torch.tensor(rng.standard_normal((B, pb.nu)), device="cuda:0")
    d = torch.tensor(rng.standard_normal((B, pb.n_w)), device="cuda:0")

    def loss_rows(X):
        ctrl.reset()
        U = ctrl.step(X)
        return (c * U).sum(1) + (d * ctrl.w_sol).sum(1), ctrl.lam_g.cpu().numpy(), ctrl.status.cpu().numpy()

    ctrl.reset()
    X = X0.clone().requires_grad_()
    U, W = mpc_step(ctrl, X, outputs="u0,w")
    ((c * U).sum() + (d * W).sum()).backward()
    g = X.grad.cpu().numpy()
    _, js = ctrl.feedback_jacobian()
    js, lam0 = js.cpu().numpy(), ctrl.lam_g.cpu().numpy()
    h = 1e-5 * np.maximum(np.abs(pb.wref[0, :nx]), 1.0)
    n = 0
    for j in range(nx):
        e = torch.zeros(nx, dtype=torch.float64, device="cuda:0")
        e[j] = h[j]
        lp, lamp, sp = loss_rows(X0 + e)
        lm, lamm, sm = loss_rows(X0 - e)
        fd = ((lp - lm) / (2 * h[j])).cpu().numpy()
        for b in range(B):
            if js[b] != 0 or sp[b] or sm[b] or not _fd_ok(pb, lam0[b], lamp[b], lamm[b]):
                continue
            assert abs(fd[b] - g[b, j]) < 1e-6 * max(1.0, np.abs(g[b]).max()), (name, b, j, fd[b], g[b, j])
            n += 1
    assert n >= nx * B // 2, n


@pytest.mark.parametrize("name", ["cstr", "awe9"])
def test_closed_loop_backprop(torch_mod, name):
    """loss.backward() through a 5-step closed loop of mpc_step and plant_step (quadratic loss written in torch) against central
    differences of the whole rollout, over the instances whose jstatus stays 0 and, per direction, whose active sets along the
    rollout are those of the nominal rollout at both sides (else the difference spans a kink), to 1e-5 relative"""
    torch = torch_mod
    from tunempc_b200.autograd import mpc_step, plant_step
    pb = load_problem(name)
    X0 = torch.tensor(load_golden(name)["X0"][:8], device="cuda:0")
    B, nx = X0.shape
    ctrl = _ctrl(pb, tol=1e-12)
    xs = torch.tensor(pb.wref[0, :nx], device="cuda:0")
    sc = torch.tensor(np.maximum(np.abs(pb.wref[0, :nx]), 1.0), device="cuda:0")

    from feedback_jacobian_support import active_set

    def rollout(X, track=False):
        ctrl.reset()
        loss = torch.zeros(B, dtype=torch.float64, device="cuda:0")
        ok = np.ones(B, dtype=bool)
        act = []
        for _ in range(5):
            U = mpc_step(ctrl, X)
            if track:
                ok &= ctrl.feedback_jacobian()[1].cpu().numpy() == 0
            lam = ctrl.lam_g.cpu().numpy()
            act.append([active_set(pb, lam[b]) for b in range(B)])
            X = plant_step(ctrl, X, U)
            loss = loss + (((X - xs) / sc) ** 2).sum(1) + 1e-3 * (U ** 2).sum(1)
        return loss, ok, act

    def same(a1, a2, b):
        return all(np.array_equal(s1[b], s2[b]) for s1, s2 in zip(a1, a2))

    X = X0.clone().requires_grad_()
    loss, ok, act0 = rollout(X, track=True)
    loss.sum().backward()
    g = X.grad.cpu().numpy()
    assert np.isfinite(g[ok]).all() and ok.sum() >= B // 2, ok
    h = 1e-5 * sc.cpu().numpy()
    n = 0
    with torch.no_grad():
        for j in range(nx):
            e = torch.zeros(nx, dtype=torch.float64, device="cuda:0")
            e[j] = h[j]
            lp, _, ap = rollout(X0 + e)
            lm, _, am = rollout(X0 - e)
            fd = ((lp - lm) / (2 * h[j])).cpu().numpy()
            for b in np.nonzero(ok)[0]:
                if not (same(ap, act0, b) and same(am, act0, b)):
                    continue
                assert abs(fd[b] - g[b, j]) < 1e-5 * max(1.0, np.abs(g[b]).max()), (name, b, j, fd[b], g[b, j])
                n += 1
    assert n >= nx * ok.sum() // 2, n


@pytest.mark.parametrize("name", ["cstr", "lq", "evaporation"])
def test_plant_jacobian(torch_mod, name):
    """tmpc_plant_jacobian against the host stage evaluation (order 1) to 1e-13 -- RK4 (cstr), discrete (lq), collocation
    (evaporation) -- and plant_step's backward against central differences of plant_step"""
    torch = torch_mod
    from tunempc_b200.autograd import plant_step
    from tunempc_b200.lib import ModelLib
    pb = load_problem(name)
    ctrl = _ctrl(pb)
    X = torch.tensor(load_golden(name)["X0"][:8], device="cuda:0")
    U = torch.tensor(np.tile(pb.wref[0, pb.nx:pb.nx + pb.nu], (X.shape[0], 1)), device="cuda:0")
    U = U + 0.01 * torch.tensor(np.random.default_rng(8).standard_normal(U.shape), device="cuda:0") * U.abs().clamp(min=1.0)
    JF = ctrl.plant_jacobian(X, U).cpu().numpy()
    _, S = ModelLib(pb.name).stage_eval(X.cpu().numpy(), U.cpu().numpy(), 1)
    assert JF.shape == S.shape
    assert np.max(np.abs(JF - S)) <= 1e-13 * max(1.0, np.abs(S).max()), np.max(np.abs(JF - S))
    Xr, Ur = X.clone().requires_grad_(), U.clone().requires_grad_()
    v = torch.tensor(np.random.default_rng(9).standard_normal(X.shape), device="cuda:0")
    (v * plant_step(ctrl, Xr, Ur)).sum().backward()
    gz = torch.cat([Xr.grad, Ur.grad], 1).cpu().numpy()
    Z = torch.cat([X, U], 1)
    nz = Z.shape[1]
    for i in range(nz):
        hi = 1e-6 * max(1.0, float(Z[:, i].abs().max()))
        Zp, Zm = Z.clone(), Z.clone()
        Zp[:, i] += hi
        Zm[:, i] -= hi
        fp = (v * ctrl.plant_step(Zp[:, :pb.nx].contiguous(), Zp[:, pb.nx:].contiguous())).sum(1)
        fm = (v * ctrl.plant_step(Zm[:, :pb.nx].contiguous(), Zm[:, pb.nx:].contiguous())).sum(1)
        fd = ((fp - fm) / (2 * hi)).cpu().numpy()
        assert np.max(np.abs(fd - gz[:, i])) < 1e-6 * max(1.0, np.abs(gz).max()), (name, i)


@pytest.mark.parametrize("name", ["cstr", "awe9"])
def test_large_fixture(torch_mod, name, capsys):
    """every instance of the large seeded fixture: finite G and jstatus 0 for most, a prefix against the twin"""
    torch = torch_mod
    from tunempc_b200 import configs
    pb = load_problem(name)
    L = np.load(os.path.join(os.path.dirname(__file__), "golden", "large_%s.npz" % name))
    X0 = configs.sample_x0(name, pb, int(L["B"]), int(L["seed"]))
    ctrl = _ctrl(pb)
    ctrl.step(torch.tensor(X0, device="cuda:0"))
    rng = np.random.default_rng(10)
    vu = torch.tensor(rng.standard_normal((len(X0), pb.nu)), device="cuda:0")
    vw = torch.tensor(rng.standard_normal((len(X0), pb.n_w)), device="cuda:0")
    G, js = ctrl.solution_vjp(v_u0=vu, v_w=vw, w=ctrl.w_sol, lam_g=ctrl.lam_g, status=ctrl.status, phase=ctrl.last_phase)
    G, js = G.cpu().numpy(), js.cpu().numpy()
    st = ctrl.status.cpu().numpy()
    hist = np.bincount(js, minlength=4)
    with capsys.disabled():
        print("\n%s B=%d VJP jstatus histogram (ok, weak, not solved, singular): %s" % (name, len(X0), hist.tolist()))
    assert hist[0] >= len(X0) // 2 and (js[st != 0] == 2).all() and np.isfinite(G[js <= 1]).all()
    n = 64
    Gt, jst = _twin_on(pb, ctrl.w_sol.cpu().numpy()[:n], ctrl.lam_g.cpu().numpy()[:n], st[:n], pb.tol, 0,
                       vu.cpu().numpy()[:n], vw.cpu().numpy()[:n])
    assert np.array_equal(js[:n], jst)
    ok = jst <= 1
    assert relerr(G[:n][ok], Gt[ok]) < 1e-8


def test_api_errors(torch_mod):
    """Gauss-Newton handle, step in flight, W == NULL before a step, phase out of range, no cotangent: RuntimeError / ValueError;
    B = 0: empty; numpy in, numpy out; single-state step: (nx,) and an int"""
    torch = torch_mod
    pb = load_problem("cstr")
    X0 = torch.tensor(load_golden("cstr")["X0"][:4], device="cuda:0")
    vu = torch.ones((4, pb.nu), dtype=torch.float64, device="cuda:0")
    ctrl = _ctrl(pb)
    with pytest.raises(RuntimeError, match="no step has finished"):
        ctrl.solution_vjp(v_u0=vu)
    ctrl.step(X0)
    sol = dict(w=ctrl.w_sol, lam_g=ctrl.lam_g, status=ctrl.status)
    with pytest.raises(RuntimeError, match="both cotangents"):
        ctrl.solution_vjp()
    with pytest.raises(RuntimeError, match="phase"):
        ctrl.solution_vjp(v_u0=vu, phase=pb.p, **sol)
    with pytest.raises(RuntimeError, match="phase"):
        ctrl.solution_vjp(v_u0=vu, phase=-1, **sol)
    G, js = ctrl.solution_vjp(v_u0=vu, phase=0, **sol)
    ctrl.reset()
    with pytest.raises(RuntimeError, match="no step has finished"):
        ctrl.solution_vjp(v_u0=vu)
    G2, js2 = ctrl.solution_vjp(v_u0=vu, phase=0, **sol)                 # a stored solution needs no finished step
    assert torch.equal(js, js2) and np.array_equal(G.cpu().numpy(), G2.cpu().numpy(), equal_nan=True)
    ctrl.step_async(X0)
    with pytest.raises(RuntimeError, match="in flight"):
        ctrl.solution_vjp(v_u0=vu, phase=0, **sol)
    ctrl.wait()
    ctrl.solution_vjp(v_u0=vu)
    gn = copy.copy(pb)
    gn.hessian_approximation = "gauss_newton"
    cg = _ctrl(gn)
    cg.step(X0)
    with pytest.raises(RuntimeError, match="exact Hessian"):
        cg.solution_vjp(v_u0=vu)
    c0 = _ctrl(pb)
    c0.step(np.zeros((0, pb.nx)))
    G0, js0 = c0.solution_vjp(v_u0=np.zeros((0, pb.nu)))
    assert G0.shape == (0, pb.nx) and js0.shape == (0,)
    cn = _ctrl(pb)
    Xn = load_golden("cstr")["X0"][:4]
    cn.step(Xn)
    Gn, jsn = cn.solution_vjp(v_u0=np.ones((4, pb.nu)))
    assert isinstance(Gn, np.ndarray) and np.array_equal(Gn, G.cpu().numpy(), equal_nan=True)
    Gh, _ = cn.solution_vjp(v_u0=np.ones((4, pb.nu)), w=sol["w"].cpu().numpy(), lam_g=sol["lam_g"].cpu().numpy(),
                            status=sol["status"].cpu().numpy(), phase=0)
    assert isinstance(Gh, np.ndarray) and np.array_equal(Gh, Gn, equal_nan=True)
    cn.reset()
    cn.step(Xn[0])
    G1, js1 = cn.solution_vjp(v_u0=np.ones(pb.nu))
    assert G1.shape == (pb.nx,) and isinstance(js1, int)
