"""Differentiable MPC step and plant step for torch autograd.

    from tunempc_b200.autograd import mpc_step, plant_step
    X = X0.requires_grad_()
    for _ in range(T):
        U = mpc_step(ctrl, X)                      # u0*(x), backward: tmpc_solution_vjp
        X = plant_step(ctrl, X, U)                 # F(x, u), backward: tmpc_plant_jacobian
    loss(X).backward()                             # dloss / dX0 through the closed loop

`mpc_step` solves with `ctrl.step` (the phase index advances as with any step) and keeps the step's solution, multipliers,
status and phase; its backward computes v' d(u0, w)/dx0 from that stored solution with one QP solve per instance
(Pmpc.solution_vjp), so it stays valid after later steps.  The derivative is the one of feedback_jacobian(): the active set
held.  Gradient rows of instances whose jstatus is 2 (the step did not converge) or 3 (singular) are NaN, as J is; rows with
jstatus 1 (a weakly active row) hold the derivative of the current active set.  The multipliers, constraint values and
statuses are not differentiable outputs.
"""
import torch


class _MpcStep(torch.autograd.Function):
    @staticmethod
    def forward(ctx, X0, ctrl, with_w):
        U0 = ctrl.step(X0.detach(), outputs="all")
        ctx.ctrl = ctrl
        ctx.phase = ctrl.last_phase
        ctx.save_for_backward(ctrl.w_sol, ctrl.lam_g, ctrl.status)
        if with_w:
            return U0, ctrl.w_sol
        return U0

    @staticmethod
    def backward(ctx, gU0, gW=None):
        W, LAM, st = ctx.saved_tensors
        G, _ = ctx.ctrl.solution_vjp(v_u0=gU0, v_w=gW, w=W, lam_g=LAM, status=st, phase=ctx.phase)
        return G, None, None


class _PlantStep(torch.autograd.Function):
    @staticmethod
    def forward(ctx, X, U, ctrl):
        ctx.ctrl = ctrl
        ctx.save_for_backward(X, U)
        return ctrl.plant_step(X.detach(), U.detach())

    @staticmethod
    def backward(ctx, g):
        X, U = ctx.saved_tensors
        JF = ctx.ctrl.plant_jacobian(X, U)                     # (B, nx, nx + nu)
        gxu = torch.bmm(g.unsqueeze(1), JF).squeeze(1)         # g' [A | B]
        nx = X.shape[1]
        return gxu[:, :nx], gxu[:, nx:], None


def mpc_step(ctrl, X0, outputs="u0"):
    """U0 = ctrl.step(X0) as a differentiable function of X0 (B, nx) float64 CUDA: outputs="u0" returns U0 (B, nu), "u0,w"
    returns (U0, W) with the whole primal solution W (B, n_w).  The controller needs the exact Hessian (or is economic)."""
    if outputs not in ("u0", "u0,w"):
        raise ValueError('outputs must be "u0" or "u0,w"')
    return _MpcStep.apply(X0, ctrl, outputs == "u0,w")


def plant_step(ctrl, X, U):
    """X+ = F(X, U) (Pmpc.plant_step) as a differentiable function of X (B, nx) and U (B, nu), float64 CUDA"""
    return _PlantStep.apply(X, U, ctrl)
