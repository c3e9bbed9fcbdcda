"""Edge gradients dL/dw of the oracle's rollout -- TEST INFRASTRUCTURE ONLY.

The forward is the reference's binary adjacency. The edge gradient is that of the weighted extension of the neighbour
sum, AI[r] = sum over stored (r, c) of w_rc I'[c], taken at w = 1. It is built from oracle/gnode_oracle.py's rhs, Euler
loop, encoder and decoder, unchanged: only orc.neighbour_sum is swapped for the weighted sum while a rollout runs.
  discrete  plain autograd through encode + euler_rollout + decode with w requiring grad;
  adjoint   torchdiffeq's adjoint recurrence (as tests/_input_grad_oracle._AdjointRolloutBG) with w as one more adjoint
            parameter: g_w += dt_i J_w(y_i)^T a_i.
Edges are numbered as the library numbers them (edge_coo): instance after instance, inside an instance row by row with
ascending columns.
"""
import contextlib

import numpy as np
import torch

from oracle import gnode_oracle as orc

_plain_neighbour_sum = orc.neighbour_sum


def edge_coo(adjs, inst):
    """(2, nnz) int64 row-major COO of the block-diagonal batch, every row's columns ascending: the order of the
    library's edge vector (DeviceGraph.edges() per instance, instance after instance)."""
    rows, cols, r0 = [], [], 0
    for g in inst:
        A = adjs[g].tocsr()
        n = A.shape[0]
        r = np.repeat(np.arange(n, dtype=np.int64), np.diff(A.indptr))
        c = np.asarray(A.indices[:A.indptr[-1]], dtype=np.int64)
        o = np.lexsort((c, r))
        rows.append(r[o] + r0)
        cols.append(c[o] + r0)
        r0 += n
    return np.vstack((np.concatenate(rows), np.concatenate(cols)))


def edge_offsets(adjs, inst):
    return np.concatenate(([0], np.cumsum([adjs[g].nnz for g in inst]))).astype(np.int64)


@contextlib.contextmanager
def weighted(w):
    """orc.rhs with AI[r] = sum_e w_e I'[col_e] over the COO it is given (w = 1 is the binary sum, bit for bit)."""
    def ns(Ip, coo):
        H = Ip.size(1)
        idx = coo if torch.is_tensor(coo) else torch.from_numpy(coo)
        out = torch.zeros(Ip.size(), dtype=Ip.dtype)
        return out.scatter_add_(0, idx[0, :].unsqueeze(1).repeat(1, H), Ip[idx[1, :]] * w.unsqueeze(1))
    orc.neighbour_sum = ns
    try:
        yield
    finally:
        orc.neighbour_sum = _plain_neighbour_sum


class _AdjointRolloutW(torch.autograd.Function):
    """torchdiffeq's adjoint recurrence with the adjoints of beta, gamma and the edge weights w:
       a_{T-1} = g_{T-1};  for i=T-1..1:  (v_y, v_th, v_bg, v_w) = J(y_i)^T a_i ;
       a_{i-1} = a_i + dt_i v_y + g_{i-1};  g_th += dt_i v_th;  g_bg += dt_i v_bg;  g_w += dt_i v_w."""

    @staticmethod
    def forward(ctx, y0, beta, gamma, W, b, w, coo, t):
        with torch.no_grad(), weighted(w):
            traj = orc.euler_rollout(y0[0], y0[1], y0[2], beta, gamma, W, b, coo, t)
        ctx.coo, ctx.t = coo, t
        ctx.save_for_backward(traj, beta, gamma, W, b, w)
        return traj

    @staticmethod
    def backward(ctx, g):
        traj, beta, gamma, W, b, w = ctx.saved_tensors
        coo, t = ctx.coo, ctx.t
        a = g[-1].clone()
        gW, gb = torch.zeros_like(W), torch.zeros_like(b)
        gbeta, ggamma, gw = torch.zeros_like(beta), torch.zeros_like(gamma), torch.zeros_like(w)
        for i in range(len(t) - 1, 0, -1):
            with torch.enable_grad():
                y = traj[i].detach().requires_grad_(True)
                Wg, bg = W.detach().requires_grad_(True), b.detach().requires_grad_(True)
                be, ga = beta.detach().requires_grad_(True), gamma.detach().requires_grad_(True)
                wg = w.detach().requires_grad_(True)
                with weighted(wg):
                    f = torch.stack(orc.rhs(y[0], y[1], y[2], be, ga, Wg, bg, coo))
                vy, vW, vb, vbe, vga, vw = torch.autograd.grad(f, (y, Wg, bg, be, ga, wg), -a, allow_unused=True)
            dt = t[i - 1] - t[i]
            a = a + dt * vy
            gW, gb = gW + dt * vW, gb + dt * vb
            gbeta, ggamma = gbeta + dt * vbe, ggamma + dt * vga
            if vw is not None:                             # (an edgeless batch: w enters nothing)
                gw = gw + dt * vw
            a = a + g[i - 1]
        return a, gbeta, ggamma, gW, gb, gw, None, None


def forward_w(x, params, coo, t, w):
    """orc.forward with the weighted neighbour sum (probabilities [T, M, 3])."""
    with weighted(w):
        return orc.forward(x, params, coo, t)


def loss_and_edge_grads(x, params, coo, t, weight, grad_mode="adjoint", w=None):
    """(dL/dw [nnz], dL/dx[:, :5]) of L = weight(probs) or sum(weight * probs), at w = 1 unless w is given. coo from
    edge_coo (or any COO whose entries w numbers)."""
    x = x.detach().clone().requires_grad_(True)
    p = {k: v.detach().clone().requires_grad_(k in orc.GRAD_KEYS) for k, v in params.items()}
    nnz = coo.shape[1]
    w = (torch.ones(nnz, dtype=x.dtype) if w is None else w.detach().clone()).requires_grad_(True)
    S0, I0, R0, beta, gamma = orc.encode(x, p["linearS1.weight"], p["linearS1.bias"])
    W, b = p["odefunc.linear.weight"], p["odefunc.linear.bias"]
    if grad_mode == "adjoint":
        traj = _AdjointRolloutW.apply(torch.stack((S0, I0, R0)), beta, gamma, W, b, w, coo, t)
    elif grad_mode == "discrete":
        with weighted(w):
            traj = orc.euler_rollout(S0, I0, R0, beta, gamma, W, b, coo, t)
    else:
        raise ValueError(grad_mode)
    probs = orc.decode(traj[:, 0], traj[:, 1], traj[:, 2], p["linear3.weight"], p["linear3.bias"],
                       p["linearS2.weight"], p["linearS2.bias"])
    loss = weight(probs) if callable(weight) else (probs * weight).sum()
    loss.backward()
    gw = w.grad.detach().clone() if w.grad is not None else torch.zeros_like(w).detach()
    return gw, x.grad[:, :5].detach().clone()


def row_sums(gw, coo, M):
    """sum over each row's stored entries of dL/dw (float64)."""
    return torch.zeros(M, dtype=torch.float64).index_add_(0, torch.from_numpy(np.asarray(coo[0])), gw.double())


def per_instance_rel_err(got, want, offsets):
    """[n_inst] max |got - want| / max |want| over each instance's slice of the edge vector (nan: empty slice or zero
    scale)."""
    got, want = got.double(), want.double()
    out = []
    for e0, e1 in zip(offsets[:-1], offsets[1:]):
        scale = want[e0:e1].abs().max().item() if e1 > e0 else 0.0
        out.append((got[e0:e1] - want[e0:e1]).abs().max().item() / scale if scale > 0 else float("nan"))
    return np.asarray(out)


# -------------------------------------------------------------------------------------------------- shared cases
MAXTIME, DELTAT, PARAM_SEED = 5, 0.5, 31           # T = 10, as tests/test_graph_structure_gpu.py


def directed_case():
    """(adjs, inst, x [M, 3+64]): two trials of tests/_graphs.directed(); trial 0 seeds the in-hub and a sink, trial 1
    the out-hub (A and A^T differ most there)."""
    import _graphs
    A = _graphs.directed()
    sizes = [A.shape[0]] * 2
    seeds = [[_graphs.IN_HUB, int(_graphs.SINKS[0])], [_graphs.OUT_HUB, 123]]
    x = torch.from_numpy(_graphs.dense_x(sizes, seeds, [0.3, 0.15], [0.2, 0.35]))
    return [A], [0, 0], x


def oracle_pair(x, params, coo, t, cot32, mode, weight=None):
    """((gw64, gx64), (gw32, gx32)): the float64 oracle and the fp32 oracle's own result (the bar's yardstick). cot32:
    the dense cotangent [T, M, 3] (float32), or None with `weight` a loss of probs (sparse cotangent)."""
    out32 = loss_and_edge_grads(x, params, coo, t, weight if cot32 is None else cot32, mode)
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        p64 = {k: v.double() for k, v in params.items()}
        out64 = loss_and_edge_grads(x.double(), p64, coo, t, weight if cot32 is None else cot32.double(), mode)
    finally:
        torch.set_default_dtype(prev)
    return out64, out32
