"""Tuner.create_mpc(..., opts={'slack_flag': 'active'}) end to end on the GPU (tunempc/tuner.py:171-177, preprocessing.py:120-155):
soft constraints through the user API, on the model-library variant evaporation_sc1, against the live oracle."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def test_tuner_soft_constraints_gpu(built):
    import torch
    from oracle import reference_port as rp
    from tunempc_b200 import configs
    from tunempc_b200.tuner import Tuner
    t = Tuner(configs.evaporation(), p=1)
    t.solve_ocp()
    t.convexify(rho=1e-3)
    ctrl = t.create_mpc("tuned", 30, opts={"slack_flag": "active"})
    pb = ctrl.problem
    assert pb.name == "evaporation_sc1" and pb.nsc == 1 and pb.nh == 6 and pb.scost[0] > 1e3
    xs = t.w_sol[0, :2]
    X0 = np.array([xs + [0.3, 0.5], [24.7, xs[1] - 0.4], [24.2, xs[1] + 0.2], xs + [0.05, -0.8]])
    U = ctrl.step(torch.tensor(X0, device="cuda:0")).cpu().numpy()
    assert (ctrl.status.cpu().numpy() == 0).all()
    w = ctrl.w_sol.cpu().numpy()
    assert np.isclose(w[1][pb.iusc(0)][0], 0.3, atol=1e-8) and np.isclose(w[2][pb.iusc(0)][0], 0.8, atol=1e-8)   # the slack absorbs x0 < bound
    oc = rp.Pmpc(pb)
    for b in range(4):
        oc.reset()
        uo = oc.step(X0[b])
        assert np.max(np.abs(U[b] - uo) / np.maximum(np.abs(uo), 1.0)) < 1e-6, b
        assert ctrl.log["iter"][-1].cpu().numpy()[b] == oc.log["iter"][-1]
        assert oc.sqp.stats["qp_branches"]["gn_resolve"] == 0            # the oracle followed the reference's path
    with pytest.raises(ValueError):
        t.create_mpc("tuned", 30, opts={"slack_flag": "some"})


def test_periodic_path_constraint_economic_gpu(built):
    """Tuner(p = 30) with a path constraint -> solve_ocp -> create_mpc('economic') on the GPU: closed loop against the live oracle"""
    import torch
    from oracle import reference_port as rp
    from tunempc_b200 import configs, tuning
    from tunempc_b200.tuner import Tuner
    card = configs.unicycle()
    C = np.zeros((1, 5))
    C[0, 0] = -1.0
    card["C"], card["c"] = C, np.array([0.7])
    t = Tuner(card, p=30)
    w = t.solve_ocp()
    ctrl = t.create_mpc("economic", 30)
    pb = ctrl.problem
    assert pb.mpc_type == "economic" and pb.p == 30 and pb.nh == 1 and np.abs(pb.lam_h_ref).max() > 1.0
    cf = tuning.lambdify_cost(card["model"], card["cost"])
    X0 = configs.sample_x0("unicycle", pb, 3, 5)
    X0[2] = w[0, :4]
    ocs = [rp.Pmpc(pb, cost_funs=cf) for _ in range(3)]
    X = torch.tensor(X0, device="cuda:0")
    xo = X0.copy()
    st = rp.StageLib("unicycle")
    for s in range(4):
        U = ctrl.step(X)
        uo = np.array([ocs[b].step(xo[b]) for b in range(3)])
        assert (ctrl.status.cpu().numpy() == 0).all()
        assert np.array_equal(ctrl.log["iter"][-1].cpu().numpy(), [ocs[b].log["iter"][-1] for b in range(3)])
        assert all(ocs[b].sqp.stats["qp_branches"]["gn_resolve"] == 0 for b in range(3))
        assert np.max(np.abs(U.cpu().numpy() - uo)) < 1e-8, s
        X = ctrl.plant_step(X, U)
        xo = st.F(xo, uo)
