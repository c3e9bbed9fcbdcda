"""GN-ODE rollout oracle -- TEST INFRASTRUCTURE ONLY.

A CPU (torch) restatement of the reference's rollout hot path.  It exists to
CHECK the CUDA product path; nothing under ``gn-ode-sir_b200/`` may import it.
Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline /
``--impl reference`` legs call into this file.

Parity status: the reference ships NO test, golden vector or known-answer for
this path (SURVEY.md section 4), so this oracle is pinned the other way the
task allows: against outputs of the reference's own classes executed in the
build container (``oracle/ref_harness.py`` + ``tests/golden/make_golden.py``;
``tests/test_oracle_vs_reference.py`` and ``tests/test_oracle_golden.py``
check the committed fixtures bit for bit).  The torchdiffeq boundary itself
(un-vendored ``torchdiffeq==0.2.2``, requirements.txt:59) is restated from the
published algorithm and is "parity unpinned" by any reference-held test.

Reference lines followed (all under /root/reference):
  encoder      ode_nn_ngraph_sim.py:149-156   ode_nn_ngraphs.py:125-131
  state pack   ode_nn_ngraph_sim.py:168       ode_nn_ngraphs.py:137
  Euler loop   torchdiffeq FixedGridODESolver.integrate / Euler._step_func
  rhs f(t,y)   ode_nn_ngraph_sim.py:58-96     ode_nn_ngraphs.py:54-83
  decoder      ode_nn_ngraph_sim.py:170-188   ode_nn_ngraphs.py:138-152
  adjoint bwd  torchdiffeq OdeintAdjointMethod.backward (see ref_harness.py)

Conventions: M rows = concatenation of "instances" (one graph + one trial
each); every instance is a contiguous row range; the adjacency of the batch is
the block diagonal of the instances' adjacencies (binary weights, every stored
entry counts once -- the reference ignores ``A.data`` and uses only the COO
pattern, ode_nn_ngraph_sim.py:69-73).
"""
from collections import OrderedDict

import numpy as np
import scipy.sparse
import torch
import torch.nn.functional as F

PARAM_SHAPES = OrderedDict([
    # state_dict key                 shape as a function of H
    ("odefunc.ln.weight", lambda H: (H,)),      # unused LayerNorm (ode_nn_ngraph_sim.py:47)
    ("odefunc.ln.bias", lambda H: (H,)),
    ("odefunc.linear.weight", lambda H: (H, H)),  # :48
    ("odefunc.linear.bias", lambda H: (H,)),
    ("linearS1.weight", lambda H: (H, 1)),      # :123
    ("linearS1.bias", lambda H: (H,)),
    ("ln.weight", lambda H: (H,)),              # unused LayerNorm (:124)
    ("ln.bias", lambda H: (H,)),
    ("linear3.weight", lambda H: (4, H)),       # :126
    ("linear3.bias", lambda H: (4,)),
    ("linearS2.weight", lambda H: (1, 4)),      # :131
    ("linearS2.bias", lambda H: (1,)),
])


def time_grid(maxTime, deltaT):
    """integration_time of ODEBlock.__init__ (ode_nn_ngraph_sim.py:110), float64."""
    return torch.from_numpy(np.arange(0, maxTime, deltaT))


def batch_coo(adjs, instance_graph):
    """Row-major COO (row, col) of the block-diagonal batch adjacency.

    adjs: list of scipy sparse matrices; instance_graph: graph index per instance.
    Follows scipy.sparse.block_diag + bdiag.row/bdiag.col at
    ode_nn_ngraph_sim.py:68-70 / ode_nn_ngraphs.py:65-70 (entry order of each
    block is its COO order, i.e. row-major for the CSR the reference holds).
    """
    blocks = [adjs[g] for g in instance_graph]
    bd = scipy.sparse.block_diag(blocks)
    return np.vstack((bd.row, bd.col)).astype(np.int64)


def neighbour_sum(Ip, coo):
    """AI[r,:] = sum over stored (r,c) of Ip[c,:] via gather + scatter_add_
    (ode_nn_ngraph_sim.py:73). On CPU scatter_add_ accumulates in index order,
    i.e. ascending column per row."""
    H = Ip.size(1)
    idx = coo if torch.is_tensor(coo) else torch.from_numpy(coo)
    out = torch.zeros(Ip.size(), dtype=Ip.dtype)
    return out.scatter_add_(0, idx[0, :].unsqueeze(1).repeat(1, H), Ip[idx[1, :]])


def rhs(S, I, R, beta, gamma, W, b, coo):
    """f(t, y) of ODEfunc.forward. Returns (dS, dI, dR); d(beta/gamma block) = 0.

    The transformed R' = sigmoid(linear(R)) is computed-and-dropped by the
    reference (:62-66 computes it, :75-77 never uses it); it is kept here only
    so that the one batched Linear call sees the same [3M,H] operand.
    """
    M = S.size(0)
    Z = torch.sigmoid(F.linear(torch.cat((S, I, R)), W, b))
    Sp, Ip = Z[:M], Z[M:2 * M]
    AI = neighbour_sum(Ip, coo)
    dS = -beta.unsqueeze(-1) * torch.multiply(AI, Sp)
    dI = -dS - gamma.unsqueeze(-1) * Ip
    dR = gamma.unsqueeze(-1) * Ip
    return dS, dI, dR


def encode(x, w1, b1):
    """x: [M, 3+H]. Returns S0, I0, R0 ([M,H] each), beta [M], gamma [M]."""
    enc = lambda c: torch.relu(F.linear(c.unsqueeze(-1), w1, b1))
    return enc(x[:, 0]), enc(x[:, 1]), enc(x[:, 2]), x[:, 3], x[:, 4]


def decode(S, I, R, W3, b3, W2, b2):
    """[..., M, H] x3 -> probabilities [..., M, 3] (softmax over {S,I,R})."""
    dec = lambda C: F.linear(torch.relu(F.linear(C, W3, b3)), W2, b2)
    return torch.softmax(torch.cat((dec(S), dec(I), dec(R)), -1), dim=-1)


def euler_rollout(S, I, R, beta, gamma, W, b, coo, t, rebuild_index=None):
    """Fixed-grid Euler over the grid t (float64 tensor). Returns traj [T,3,M,H].

    rebuild_index: optional callable returning a fresh COO each step -- used by
    the CPU baseline timing to reproduce the reference's per-step host-side
    block_diag rebuild (ode_nn_ngraph_sim.py:68-71).
    """
    states = [torch.stack((S, I, R))]
    for k in range(len(t) - 1):
        dt = t[k + 1] - t[k]                 # 0-dim float64: does not promote fp32
        if rebuild_index is not None:
            coo = rebuild_index()
        dS, dI, dR = rhs(S, I, R, beta, gamma, W, b, coo)
        S, I, R = S + dt * dS, I + dt * dI, R + dt * dR
        states.append(torch.stack((S, I, R)))
    return torch.stack(states)


def _p(params, key):
    return params[key]


def forward(x, params, coo, t, return_traj=False, rebuild_index=None):
    """ODEBlock.forward. x: [M, 3+H]; params: state_dict-style mapping.
    Returns probs [T, M, 3] (columns S, I, R) and optionally traj [T,3,M,H]."""
    S0, I0, R0, beta, gamma = encode(x, _p(params, "linearS1.weight"), _p(params, "linearS1.bias"))
    traj = euler_rollout(S0, I0, R0, beta, gamma,
                         _p(params, "odefunc.linear.weight"), _p(params, "odefunc.linear.bias"),
                         coo, t, rebuild_index=rebuild_index)
    probs = decode(traj[:, 0], traj[:, 1], traj[:, 2],
                   _p(params, "linear3.weight"), _p(params, "linear3.bias"),
                   _p(params, "linearS2.weight"), _p(params, "linearS2.bias"))
    return (probs, traj) if return_traj else probs


def neighbour_sum_chunked(Ip, rowptr, colidx, rows_per_chunk=1 << 17):
    """neighbour_sum for graphs whose [nnz, H] gather + repeated int64 index (ode_nn_ngraph_sim.py:73) does not fit
    host memory (BA N=2M: 30 GB): the same gather + scatter_add_ over consecutive row ranges of the row-major COO.
    scatter_add_ on CPU accumulates every output row in index order, so cutting the COO between rows leaves each row's
    sum bitwise unchanged (tests/test_oracle_golden.py::test_streaming_forward_is_bitwise_forward)."""
    H = Ip.size(1)
    M = Ip.size(0)
    out = torch.zeros(Ip.size(), dtype=Ip.dtype)
    rp = torch.as_tensor(rowptr, dtype=torch.int64)
    ci = torch.as_tensor(colidx, dtype=torch.int64)
    for r0 in range(0, M, rows_per_chunk):
        r1 = min(M, r0 + rows_per_chunk)
        e0, e1 = int(rp[r0]), int(rp[r1])
        if e1 == e0:
            continue
        rows = torch.repeat_interleave(torch.arange(r0, r1), rp[r0 + 1:r1 + 1] - rp[r0:r1]) - r0
        out[r0:r1].scatter_add_(0, rows.unsqueeze(1).repeat(1, H), Ip[ci[e0:e1]])
    return out


def forward_streaming(x, params, A, t, out_steps=None):
    """forward() for ONE instance of a graph too large for the [T,3,M,H] trajectory and the [nnz,H] gather: the same
    operations in the same order (encode, rhs with the chunked neighbour sum, Euler update, decode), keeping only the
    current state; probabilities of the grid points in out_steps (default: all). A: scipy CSR with sorted indices."""
    A = scipy.sparse.csr_matrix(A)
    A.sort_indices()
    S, I, R, beta, gamma = encode(x, _p(params, "linearS1.weight"), _p(params, "linearS1.bias"))
    W, b = _p(params, "odefunc.linear.weight"), _p(params, "odefunc.linear.bias")
    dec = lambda S_, I_, R_: decode(S_, I_, R_, _p(params, "linear3.weight"), _p(params, "linear3.bias"),
                                    _p(params, "linearS2.weight"), _p(params, "linearS2.bias"))
    keep = set(range(len(t))) if out_steps is None else set(int(k) for k in out_steps)
    out = []
    M = S.size(0)
    for k in range(len(t)):
        if k in keep:
            out.append(dec(S, I, R))
        if k + 1 == len(t):
            break
        dt = t[k + 1] - t[k]
        Z = torch.sigmoid(F.linear(torch.cat((S, I, R)), W, b))
        Sp, Ip = Z[:M], Z[M:2 * M]
        AI = neighbour_sum_chunked(Ip, A.indptr, A.indices)
        dS = -beta.unsqueeze(-1) * torch.multiply(AI, Sp)
        dI = -dS - gamma.unsqueeze(-1) * Ip
        dR = gamma.unsqueeze(-1) * Ip
        S, I, R = S + dt * dS, I + dt * dI, R + dt * dR
    return torch.stack(out)


# --------------------------------------------------------------------------
# gradients
# --------------------------------------------------------------------------
GRAD_KEYS = ("odefunc.linear.weight", "odefunc.linear.bias", "linearS1.weight",
             "linearS1.bias", "linear3.weight", "linear3.bias",
             "linearS2.weight", "linearS2.bias")


class _AdjointRollout(torch.autograd.Function):
    """torchdiffeq's adjoint recurrence specialised to this rhs (SURVEY 3C):
       a_{T-1} = g_{T-1};  for i=T-1..1:  (v_y, v_th) = J(y_i)^T a_i ;
       a_{i-1} = a_i + dt_i v_y + g_{i-1};  g_th += dt_i v_th."""

    @staticmethod
    def forward(ctx, y0, beta, gamma, W, b, coo, t):
        with torch.no_grad():
            traj = euler_rollout(y0[0], y0[1], y0[2], beta, gamma, W, b, coo, t)
        ctx.coo, ctx.t = coo, t
        ctx.save_for_backward(traj, beta, gamma, W, b)
        return traj

    @staticmethod
    def backward(ctx, g):
        traj, beta, gamma, W, b = ctx.saved_tensors
        coo, t = ctx.coo, ctx.t
        a = g[-1].clone()
        gW, gb = torch.zeros_like(W), torch.zeros_like(b)
        for i in range(len(t) - 1, 0, -1):
            with torch.enable_grad():
                y = traj[i].detach().requires_grad_(True)
                Wg, bg = W.detach().requires_grad_(True), b.detach().requires_grad_(True)
                f = torch.stack(rhs(y[0], y[1], y[2], beta, gamma, Wg, bg, coo))
                vy, vW, vb = torch.autograd.grad(f, (y, Wg, bg), -a)
            dt = t[i - 1] - t[i]
            a = a + dt * vy
            gW, gb = gW + dt * vW, gb + dt * vb
            a = a + g[i - 1]
        return a, None, None, gW, gb, None, None


def loss_and_grads(x, params, coo, t, weight, grad_mode="adjoint"):
    """Scalar probe loss  L = sum(weight * probs)  and dL/dparams.

    grad_mode "adjoint" reproduces what loss.backward() yields in the
    reference (torchdiffeq adjoint); "discrete" is exact back-propagation
    through the Euler loop. Returns (loss, {key: grad}).
    """
    p = {k: v.detach().clone().requires_grad_(k in GRAD_KEYS) for k, v in params.items()}
    S0, I0, R0, beta, gamma = encode(x, p["linearS1.weight"], p["linearS1.bias"])
    W, b = p["odefunc.linear.weight"], p["odefunc.linear.bias"]
    if grad_mode == "adjoint":
        traj = _AdjointRollout.apply(torch.stack((S0, I0, R0)), beta, gamma, W, b, coo, t)
    elif grad_mode == "discrete":
        traj = euler_rollout(S0, I0, R0, beta, gamma, W, b, coo, t)
    else:
        raise ValueError(grad_mode)
    probs = decode(traj[:, 0], traj[:, 1], traj[:, 2], p["linear3.weight"], p["linear3.bias"],
                   p["linearS2.weight"], p["linearS2.bias"])
    loss = weight(probs) if callable(weight) else (probs * weight).sum()
    loss.backward()
    return loss.detach(), {k: p[k].grad.detach().clone() for k in GRAD_KEYS}


def unit_time_rows(maxTime, deltaT):
    """Rows get_sir_t_nodes_torch copies out of a [T, nodes] trajectory: int(i/deltaT), i = 0..maxTime-1
    (/root/reference/ode_nn.py:249-261, count=False branch)."""
    return [int(i / deltaT) for i in range(int(maxTime))]


def train_loss(probs, y, maxTime, deltaT):
    """The loss of the reference's train()/test() (/root/reference/ode_nn_ngraph_sim.py:230-234,
    ode_nn_ngraphs.py:212-216): the S, I, R predictions at the unit-time rows, stacked on the last axis and
    transposed to [M, maxTime, 3], against the labels y.view(-1, maxTime, 3) (float64), nn.L1Loss (mean) on
    [:, 1:, :]. The float32 prediction is promoted to float64 by the subtraction, as in the reference."""
    rows = torch.tensor(unit_time_rows(maxTime, deltaT))
    pred = probs.index_select(0, rows).transpose(0, 1)                    # [M, maxTime, 3]
    target = y.reshape(-1, y.size(-2), y.size(-1))
    return torch.nn.functional.l1_loss(pred[:, 1:, :], target[:, 1:, :]) if pred.dtype == target.dtype \
        else (pred[:, 1:, :] - target[:, 1:, :]).abs().mean()


def train_loss_and_grads(x, params, coo, t, y, maxTime, deltaT, grad_mode="adjoint"):
    """One train() mini-batch of the reference: (loss, {key: grad})."""
    return loss_and_grads(x, params, coo, t, lambda probs: train_loss(probs, y, maxTime, deltaT), grad_mode)


# --------------------------------------------------------------------------
# deterministic synthetic inputs shared by tests, smoke() and bench.py
# (SURVEY.md section 8d; monitorer-sim.py:116-119 for the trial distribution)
# --------------------------------------------------------------------------
def default_params(H, seed=0, dtype=torch.float32):
    """nn.Linear / nn.LayerNorm default initialisation in the construction
    order of the reference (ODEfunc first, then ODEBlock; ode_nn_ngraph_sim.py:437-438)."""
    gen_state = torch.random.get_rng_state()
    torch.manual_seed(seed)
    import torch.nn as nn
    of_ln, of_lin = nn.LayerNorm(H), nn.Linear(H, H)
    s1, ln, l3, s2 = nn.Linear(1, H), nn.LayerNorm(H), nn.Linear(H, 4), nn.Linear(4, 1)
    torch.random.set_rng_state(gen_state)
    sd = OrderedDict([
        ("odefunc.ln.weight", of_ln.weight), ("odefunc.ln.bias", of_ln.bias),
        ("odefunc.linear.weight", of_lin.weight), ("odefunc.linear.bias", of_lin.bias),
        ("linearS1.weight", s1.weight), ("linearS1.bias", s1.bias),
        ("ln.weight", ln.weight), ("ln.bias", ln.bias),
        ("linear3.weight", l3.weight), ("linear3.bias", l3.bias),
        ("linearS2.weight", s2.weight), ("linearS2.bias", s2.bias)])
    return OrderedDict((k, v.detach().to(dtype).clone()) for k, v in sd.items())


def synthetic_trial(n_nodes, H, trial_id, graph_marker=0.0, n_seeds=2, dtype=torch.float32):
    """One [N, 3+H] input block as main() builds it (ode_nn_ngraph_sim.py:371-390,
    ode_nn_ngraphs.py:332-348): columns S0 | I0 | R0 | beta gamma marker 0..."""
    rng = np.random.RandomState(1000 + trial_id)
    seeds = rng.choice(n_nodes, n_seeds, replace=False)
    beta, gamma = rng.uniform(0.1, 0.5), rng.uniform(0.1, 0.5)
    x = torch.zeros(n_nodes, 3 + H, dtype=dtype)
    x[seeds, 1] = 1.0
    x[:, 0] = 1.0 - x[:, 1]
    x[:, 3], x[:, 4] = beta, gamma
    if graph_marker:
        x[0, 5] = graph_marker
    return x


# --------------------------------------------------------------------------
# Monte-Carlo SIR labels: the process of /root/reference/ode_nn.py:30-88 (sir_torch), all simulations advanced
# together with numpy (checker of the CUDA label generator; statistical comparison only -- the random streams differ)
# --------------------------------------------------------------------------
def mc_sir_counts(A, seed_set, beta, gamma, sims, T, rng):
    """Returns counts [3, T, n] (S, I, R) over `sims` simulations; t = 0 rows hold the 0/1 initial state, as the
    reference assigns them (ode_nn.py:54-55). Per step (ode_nn.py:57-76): every edge from a node infected at the start
    of the step to a susceptible node transmits with probability beta; every such infected node recovers with
    probability gamma."""
    import numpy as np
    A = A.tocoo()
    src, dst = A.row, A.col
    keep = src != dst
    src, dst = src[keep], dst[keep]
    n = A.shape[0]
    I = np.zeros((sims, n), dtype=bool)
    I[:, list(seed_set)] = True
    S = ~I
    R = np.zeros_like(I)
    counts = np.zeros((3, T, n))
    counts[0, 0], counts[1, 0] = S[0], I[0]
    for t in range(1, T):
        hit = I[:, src] & S[:, dst] & (rng.random_sample((sims, len(src))) < beta)
        newly = np.zeros((sims, n), dtype=bool)
        rows, cols = np.nonzero(hit)
        newly[rows, dst[cols]] = True
        rec = I & (rng.random_sample((sims, n)) < gamma)
        R |= rec
        I = (I | newly) & ~rec
        S &= ~newly
        counts[0, t], counts[1, t], counts[2, t] = S.sum(0), I.sum(0), R.sum(0)
    return counts
