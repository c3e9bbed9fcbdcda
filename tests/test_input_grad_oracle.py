"""CPU checks of the oracle's input gradients dL/dx[:, :5] (S0, I0, R0, beta, gamma), the yardstick of
tests/test_input_grad_gpu.py: the discrete gradient is plain autograd of the Euler loop and agrees with central
differences; the adjoint gradient is what the restated torchdiffeq adjoint returns for the reference's packed state
cat(S, I, R, bg), whose bg block carries beta and gamma."""
import torch
import torch.nn as nn

from _util import Golden
from _input_grad_oracle import loss_and_input_grads
from oracle import gnode_oracle as orc
from oracle.ref_harness import odeint_adjoint_restated


def karate_case(B=2, maxTime=3, deltaT=0.5, seed=21):
    A = Golden("sim_karate_b8").adjs[0]
    N = A.shape[0]
    params = {k: v.double() for k, v in orc.default_params(64, seed=seed).items()}
    x = torch.cat([orc.synthetic_trial(N, 64, 40 + b) for b in range(B)]).double()
    t = orc.time_grid(maxTime, deltaT)                        # T = 6
    w = torch.randn(len(t), B * N, 3, generator=torch.Generator().manual_seed(seed), dtype=torch.float64)
    return x, params, orc.batch_coo([A], [0] * B), t, w


def probe_loss(x, params, coo, t, w):
    return (orc.forward(x, params, coo, t) * w).sum()


def test_discrete_input_grads_are_autograd_and_match_central_differences():
    x, params, coo, t, w = karate_case()
    assert len(t) == 6
    _, _, gx = loss_and_input_grads(x, params, coo, t, w, "discrete")
    xr = x.clone().requires_grad_(True)
    probe_loss(xr, params, coo, t, w).backward()
    assert torch.equal(gx, xr.grad[:, :5])
    assert float(xr.grad[:, 5:].abs().max()) == 0.0
    scale = gx.abs().max(0).values                        # per column
    h = 1e-6
    gen = torch.Generator().manual_seed(5)
    rows = torch.randperm(x.size(0), generator=gen)[:6].tolist()
    with torch.no_grad():
        for r in rows:
            for c in range(5):
                xp, xm = x.clone(), x.clone()
                xp[r, c] += h
                xm[r, c] -= h
                fd = (probe_loss(xp, params, coo, t, w) - probe_loss(xm, params, coo, t, w)) / (2 * h)
                err = abs(float(fd) - float(gx[r, c])) / float(scale[c])
                assert err < 1e-6, (r, c, float(fd), float(gx[r, c]), err)


class PackedRhs(nn.Module):
    """f(t, y) on the reference's packed state y = cat(S, I, R, bg) [4M, H]: beta and gamma are read from the bg block
    (ode_nn_ngraph_sim.py:60), whose derivative is zero."""

    def __init__(self, W, b, coo, M):
        super().__init__()
        self.W, self.b = nn.Parameter(W.clone()), nn.Parameter(b.clone())
        self.coo, self.M = coo, M

    def forward(self, t, y):
        M = self.M
        bg = y[3 * M:]
        dS, dI, dR = orc.rhs(y[:M], y[M:2 * M], y[2 * M:3 * M], bg[:, 0], bg[:, 1], self.W, self.b, self.coo)
        return torch.cat((dS, dI, dR, torch.zeros_like(bg)))


def test_adjoint_input_grads_equal_restated_torchdiffeq():
    x, params, coo, t, w = karate_case()
    M = x.size(0)
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        _, _, gx = loss_and_input_grads(x, params, coo, t, w, "adjoint")
        xr = x.clone().requires_grad_(True)
        S0, I0, R0, _, _ = orc.encode(xr, params["linearS1.weight"], params["linearS1.bias"])
        y0 = torch.cat((S0, I0, R0, xr[:, 3:]))
        func = PackedRhs(params["odefunc.linear.weight"], params["odefunc.linear.bias"], coo, M)
        sol = odeint_adjoint_restated(func, y0, t, method="euler")
        probs = orc.decode(sol[:, :M], sol[:, M:2 * M], sol[:, 2 * M:3 * M], params["linear3.weight"],
                           params["linear3.bias"], params["linearS2.weight"], params["linearS2.bias"])
        (probs * w).sum().backward()
    finally:
        torch.set_default_dtype(prev)
    want = xr.grad[:, :5]
    scale = want.abs().max(0).values
    assert float(scale[3]) > 0 and float(scale[4]) > 0
    err = ((gx - want).abs().max(0).values / scale).max().item()
    assert err < 1e-12, err
    # the discrete and adjoint gradients are different quantities, but close on this short horizon
    _, _, gd = loss_and_input_grads(x, params, coo, t, w, "discrete")
    assert ((gd - gx).abs().max(0).values / scale).max().item() < 0.5


def test_parameter_gradients_unchanged_by_input_grads():
    x, params, coo, t, w = karate_case(B=1)
    for mode in ("adjoint", "discrete"):
        _, g0 = orc.loss_and_grads(x, params, coo, t, w, mode)
        _, g1, _ = loss_and_input_grads(x, params, coo, t, w, mode)
        for k in orc.GRAD_KEYS:
            assert torch.equal(g0[k], g1[k]), (mode, k)
