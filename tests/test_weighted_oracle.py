"""CPU checks of the oracle's weighted rollout at non-unit contact weights (tests/_edge_grad_oracle.py), the yardstick of
tests/test_weighted_gpu.py: dL/dw at random weights agrees with float64 central differences (discrete) and with the
restated torchdiffeq adjoint that carries w as an adjoint parameter (adjoint); every row's weighted edge gradients sum
to beta[r] dL/dbeta[r]. The last test shows from the oracle alone that the GPU bar fails a reverse sweep whose A^T
gather reads w_rc instead of w_cr (asymmetric weights on the symmetric karate graph, where the transposed pattern is the
forward one and only the weights' order can be wrong) or ignores the weights."""
import contextlib

import numpy as np
import pytest
import torch

import _graphs
from _edge_grad_oracle import edge_coo, forward_w, loss_and_edge_grads, row_sums, weighted
from _util import Golden
from oracle import gnode_oracle as orc
from oracle.ref_harness import odeint_adjoint_restated
from test_edge_grad_oracle import WeightedPackedRhs


def small_case(maxTime=3, deltaT=0.5, seed=21):
    """Two trials of a 40-node directed graph with a hub, float64, T = 6, weights in [0, 2) different per trial."""
    A = _graphs.random_directed(40, 3, 7)
    adjs, inst = [A], [0, 0]
    params = {k: v.double() for k, v in orc.default_params(64, seed=seed).items()}
    x = torch.cat([orc.synthetic_trial(40, 64, 40 + b) for b in range(2)]).double()
    t = orc.time_grid(maxTime, deltaT)
    c = torch.randn(len(t), 80, 3, generator=torch.Generator().manual_seed(seed), dtype=torch.float64)
    coo = edge_coo(adjs, inst)
    w = 2.0 * torch.rand(coo.shape[1], generator=torch.Generator().manual_seed(seed + 1), dtype=torch.float64)
    return x, params, coo, t, c, w


def test_discrete_weighted_grads_match_central_differences():
    x, params, coo, t, c, w = small_case()
    gw, gx = loss_and_edge_grads(x, params, coo, t, c, "discrete", w=w)
    scale = gw.abs().max().item()
    assert scale > 0
    loss = lambda wt, xt=x: (forward_w(xt, params, coo, t, wt) * c).sum()
    pick = torch.randperm(coo.shape[1], generator=torch.Generator().manual_seed(3))[:8].tolist()
    pick.append(int(np.flatnonzero(coo[0] == np.bincount(coo[0]).argmax())[0]))        # the longest row
    h = 1e-6
    with torch.no_grad():
        for e in pick:
            wp, wm = w.clone(), w.clone()
            wp[e] += h
            wm[e] -= h
            fd = (loss(wp) - loss(wm)) / (2 * h)
            assert abs(float(fd) - float(gw[e])) / scale < 1e-6, (e, float(fd), float(gw[e]))
        # and dL/dbeta of one row at these weights
        r = int(coo[0][pick[-1]])
        xp, xm = x.clone(), x.clone()
        xp[r, 3] += h
        xm[r, 3] -= h
        fd = (loss(w, xp) - loss(w, xm)) / (2 * h)
        assert abs(float(fd) - float(gx[r, 3])) <= 1e-6 * gx[:, 3].abs().max().item()


def test_adjoint_weighted_grads_equal_restated_torchdiffeq():
    x, params, coo, t, c, w = small_case()
    M = x.size(0)
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        gw, _ = loss_and_edge_grads(x, params, coo, t, c, "adjoint", w=w)
        S0, I0, R0, _, _ = orc.encode(x, params["linearS1.weight"], params["linearS1.bias"])
        func = WeightedPackedRhs(params["odefunc.linear.weight"], params["odefunc.linear.bias"], coo, M)
        with torch.no_grad():
            func.w.copy_(w)
        sol = odeint_adjoint_restated(func, torch.cat((S0, I0, R0, x[:, 3:])), t, method="euler")
        probs = orc.decode(sol[:, :M], sol[:, M:2 * M], sol[:, 2 * M:3 * M], params["linear3.weight"],
                           params["linear3.bias"], params["linearS2.weight"], params["linearS2.bias"])
        (probs * c).sum().backward()
    finally:
        torch.set_default_dtype(prev)
    want = func.w.grad
    scale = want.abs().max().item()
    assert scale > 0 and (gw - want).abs().max().item() / scale < 1e-12


@pytest.mark.parametrize("mode", ["adjoint", "discrete"])
def test_weighted_row_sums_are_beta_times_dbeta(mode):
    """sum_c w_rc dL/dw_rc = beta[r] dL/dbeta[r]: AI is linear in the row's weights and enters only as beta AI."""
    x, params, coo, t, c, w = small_case()
    gw, gx = loss_and_edge_grads(x, params, coo, t, c, mode, w=w)
    want = x[:, 3] * gx[:, 3]
    scale = want.abs().max().item()
    assert scale > 0
    assert (row_sums(gw * w, coo, x.size(0)) - want).abs().max().item() / scale < 1e-12


@contextlib.contextmanager
def mistaken_transpose(w, w_back):
    """The weighted neighbour sum whose backward to I' uses w_back in place of w: gI'[c] = sum over entries (r, c) of
    w_back[e] G[r] -- what a sweep computes whose A^T gather reads the weights in the wrong order (w_back = w of the
    mirrored entry) or not at all (w_back = 1). The gradient with respect to w itself is left intact."""
    class NS(torch.autograd.Function):
        @staticmethod
        def forward(ctx, Ip, wt, idx):
            ctx.save_for_backward(Ip, idx)
            out = torch.zeros(Ip.size(), dtype=Ip.dtype)
            return out.scatter_add_(0, idx[0].unsqueeze(1).repeat(1, Ip.size(1)), Ip[idx[1]] * wt.unsqueeze(1))

        @staticmethod
        def backward(ctx, g):
            Ip, idx = ctx.saved_tensors
            gIp = torch.zeros_like(Ip).index_add_(0, idx[1], g[idx[0]] * w_back.unsqueeze(1))
            return gIp, (g[idx[0]] * Ip[idx[1]]).sum(1), None

    plain = orc.neighbour_sum
    orc.neighbour_sum = lambda Ip, coo: NS.apply(Ip, w, coo if torch.is_tensor(coo) else torch.from_numpy(coo))
    try:
        yield
    finally:
        orc.neighbour_sum = plain


def grads64(x, params, coo, t, c, w, w_back=None):
    """(linear.weight gradient, dL/dx[:, :5]) of the discrete rollout, float64."""
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        xx = x.double().clone().requires_grad_(True)
        p = {k: v.double().clone().requires_grad_(k in orc.GRAD_KEYS) for k, v in params.items()}
        ctxm = mistaken_transpose(w, w_back) if w_back is not None else weighted(w)
        with ctxm:
            probs = orc.forward(xx, p, coo, t)
        (probs * c.double()).sum().backward()
        return p["odefunc.linear.weight"].grad.clone(), xx.grad[:, :5].clone()
    finally:
        torch.set_default_dtype(prev)


def test_gpu_bar_fails_transpose_gather_in_forward_order_or_unweighted():
    """karate x 2 (symmetric pattern), asymmetric weights in [0, 2): a sweep gathering sum_c w_rc G[c] instead of
    sum_c w_cr G[c], or sum_c G[c], misses the GPU bar max(1e-3, 2 x the fp32 oracle's error) on linear.weight and on
    every dL/dx column that the neighbour sum reaches (measured factors printed; asserted: 10x)."""
    A = Golden("sim_karate_b8").adjs[0]
    assert (A != A.T).nnz == 0
    adjs, inst = [A], [0, 0]
    x = torch.cat([orc.synthetic_trial(A.shape[0], 64, 700 + b) for b in range(2)])
    params = orc.default_params(64, seed=31)
    t = orc.time_grid(5, 0.5)
    coo = edge_coo(adjs, inst)
    M = x.size(0)
    c = torch.randn(len(t), M, 3, generator=torch.Generator().manual_seed(9))
    w = 2.0 * torch.rand(coo.shape[1], generator=torch.Generator().manual_seed(4), dtype=torch.float64)
    key = coo[0] * M + coo[1]
    mirror = np.searchsorted(key, coo[1] * M + coo[0])                 # entry (c, r) of every entry (r, c)
    assert np.array_equal(key[mirror], coo[1] * M + coo[0])
    assert (w - w[mirror]).abs().max() > 0.5                            # the weights are far from symmetric
    gl64, gx64 = grads64(x, params, coo, t, c, w)
    gl, gx = grads64(x, params, coo, t, c, w, w_back=w)                 # the helper with the right order is the oracle
    assert torch.allclose(gl, gl64, rtol=0, atol=1e-12 * gl64.abs().max().item())
    # the fp32 oracle's own error sets the bar, as in the GPU tests
    xx = x.clone().requires_grad_(True)
    p = {k: v.clone().requires_grad_(k in orc.GRAD_KEYS) for k, v in params.items()}
    with weighted(w.float()):
        (orc.forward(xx, p, coo, t) * c).sum().backward()
    rel = lambda a, b: (a.double() - b).abs().max().item() / b.abs().max().item()
    cols = [0, 1, 3, 4]                                                 # R0 does not enter the rollout's I' chain
    bar_l = max(1e-3, 2 * rel(p["odefunc.linear.weight"].grad, gl64))
    bar_x = [max(1e-3, 2 * rel(xx.grad[:, j], gx64[:, j])) for j in cols]
    for what, w_back in (("forward order", w[mirror]), ("unweighted", torch.ones_like(w))):
        gl, gx = grads64(x, params, coo, t, c, w, w_back=w_back)
        f_l = rel(gl, gl64) / bar_l
        f_x = [rel(gx[:, j], gx64[:, j]) / b for j, b in zip(cols, bar_x)]
        print("karate, transpose gather %s: misses the bar by %.0fx on linear.weight, %s on dL/dx columns %s"
              % (what, f_l, ["%.0fx" % v for v in f_x], cols))
        assert f_l >= 10 and min(f_x) >= 10, (what, f_l, f_x)
