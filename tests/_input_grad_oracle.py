"""Input gradients dL/dx[:, :5] (S0, I0, R0, beta, gamma) of the oracle's rollout -- TEST INFRASTRUCTURE ONLY.

Built from oracle/gnode_oracle.py's encoder, right-hand side, Euler loop and decoder, unchanged:
  discrete  plain autograd through encode + euler_rollout + decode with x requiring grad;
  adjoint   torchdiffeq's adjoint recurrence (as gnode_oracle._AdjointRollout) extended by the bg block of the reference's
            ODE state: beta and gamma sit there (f reads them, ode_nn_ngraph_sim.py:60; d bg/dt = 0), so their adjoint
            builds up over the reverse sweep, g_beta += dt_i J_beta(y_i)^T a_i, and is returned as their gradient. The
            encoder's autograd then carries the final adjoint a_0 into x[:, 0:3].
"""
import torch

from oracle import gnode_oracle as orc


class _AdjointRolloutBG(torch.autograd.Function):
    """gnode_oracle._AdjointRollout with the adjoints of beta and gamma:
       a_{T-1} = g_{T-1};  for i=T-1..1:  (v_y, v_th, v_bg) = J(y_i)^T a_i ;
       a_{i-1} = a_i + dt_i v_y + g_{i-1};  g_th += dt_i v_th;  g_bg += dt_i v_bg."""

    @staticmethod
    def forward(ctx, y0, beta, gamma, W, b, coo, t):
        with torch.no_grad():
            traj = orc.euler_rollout(y0[0], y0[1], y0[2], beta, gamma, W, b, coo, t)
        ctx.coo, ctx.t = coo, t
        ctx.save_for_backward(traj, beta, gamma, W, b)
        return traj

    @staticmethod
    def backward(ctx, g):
        traj, beta, gamma, W, b = ctx.saved_tensors
        coo, t = ctx.coo, ctx.t
        a = g[-1].clone()
        gW, gb = torch.zeros_like(W), torch.zeros_like(b)
        gbeta, ggamma = torch.zeros_like(beta), torch.zeros_like(gamma)
        for i in range(len(t) - 1, 0, -1):
            with torch.enable_grad():
                y = traj[i].detach().requires_grad_(True)
                Wg, bg = W.detach().requires_grad_(True), b.detach().requires_grad_(True)
                be, ga = beta.detach().requires_grad_(True), gamma.detach().requires_grad_(True)
                f = torch.stack(orc.rhs(y[0], y[1], y[2], be, ga, Wg, bg, coo))
                vy, vW, vb, vbe, vga = torch.autograd.grad(f, (y, Wg, bg, be, ga), -a)
            dt = t[i - 1] - t[i]
            a = a + dt * vy
            gW, gb = gW + dt * vW, gb + dt * vb
            gbeta, ggamma = gbeta + dt * vbe, ggamma + dt * vga
            a = a + g[i - 1]
        return a, gbeta, ggamma, gW, gb, None, None


def loss_and_input_grads(x, params, coo, t, weight, grad_mode="adjoint"):
    """orc.loss_and_grads with x requiring grad: (loss, {key: dL/dparam}, dL/dx[:, :5]). A parameter that never enters
    the loss (linear.weight / bias of a one-point grid in discrete mode) gets a zero gradient."""
    x = x.detach().clone().requires_grad_(True)
    p = {k: v.detach().clone().requires_grad_(k in orc.GRAD_KEYS) for k, v in params.items()}
    S0, I0, R0, beta, gamma = orc.encode(x, p["linearS1.weight"], p["linearS1.bias"])
    W, b = p["odefunc.linear.weight"], p["odefunc.linear.bias"]
    if grad_mode == "adjoint":
        traj = _AdjointRolloutBG.apply(torch.stack((S0, I0, R0)), beta, gamma, W, b, coo, t)
    elif grad_mode == "discrete":
        traj = orc.euler_rollout(S0, I0, R0, beta, gamma, W, b, coo, t)
    else:
        raise ValueError(grad_mode)
    probs = orc.decode(traj[:, 0], traj[:, 1], traj[:, 2], p["linear3.weight"], p["linear3.bias"],
                       p["linearS2.weight"], p["linearS2.bias"])
    loss = weight(probs) if callable(weight) else (probs * weight).sum()
    loss.backward()
    grads = {k: p[k].grad.detach().clone() if p[k].grad is not None else torch.zeros_like(p[k]).detach()
             for k in orc.GRAD_KEYS}
    return loss.detach(), grads, x.grad[:, :5].detach().clone()
