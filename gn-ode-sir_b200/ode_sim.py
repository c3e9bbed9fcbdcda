"""Drop-in ``ODEfunc`` / ``ODEBlock`` for the single-graph / many-trials script.

Same constructors, ``forward`` signatures, parameter names / shapes / default
initialisation order as /root/reference/ode_nn_ngraph_sim.py:37-96 (ODEfunc) and
:99-188 (ODEBlock), so ``ode_nn_ngraph_sim.py``'s ``train`` / ``test`` / ``main``
(and therefore ``monitorer-sim.py``) run unchanged and ``state_dict``s interchange.
The arithmetic runs in hand-written sm_100a kernels behind the C ABI.
"""
import numpy as np
import torch
import torch.nn as nn

from . import rollout as _ro
from .graph import BatchCache, DeviceGraph


class ODEfunc(nn.Module):
    """Right-hand side holder: owns ``linear`` (H->H) and the unused ``ln``."""

    def __init__(self, A, beta, gamma, hidden1, device):
        super().__init__()
        _ro.check_hidden(hidden1)
        self.hidden1 = hidden1
        self.A = A
        self.beta = beta
        self.gamma = gamma
        # construction order == reference (LayerNorm draws no random numbers, Linear does)
        self.ln = nn.LayerNorm(hidden1)
        self.linear = nn.Linear(hidden1, hidden1)
        self.relu = nn.ReLU()
        self.sigmoid = nn.Sigmoid()
        self.dropout = nn.Dropout(0.1)
        self._graph = None
        self._batches = BatchCache()

    # -- device graph management ------------------------------------------
    def device_graph(self):
        if self._graph is None:
            self._graph = DeviceGraph(self.A)
        return self._graph

    def batch_for(self, n_trials):
        g = self.device_graph()
        return self._batches.get([g] * n_trials)

    def forward(self, t, x):
        """f(t, y) on the packed state y = cat(S, I, R, bg) of shape [4M, H]
        (ode_nn_ngraph_sim.py:58-96). Inference-only entry: ODEBlock.forward runs the
        whole rollout in one fused call and never comes through here."""
        M = x.size(0) // 4
        N = self.device_graph().n
        batch = self.batch_for(M // N)
        h = x.size(1)
        y = x[:3 * M].view(3, M, h)
        bg = x[3 * M:]
        W, b = _ro.pad_linear(self.linear.weight, self.linear.bias)
        dy = _ro.odefunc_eval(_ro.pad_channels(y), bg[:, 0], bg[:, 1], batch, [W, b] + [b] * 6)[..., :h]
        return torch.cat((dy.reshape(3 * M, -1), torch.zeros_like(bg)))


class ODEBlock(nn.Module):
    """Encoder -> fixed-grid Euler rollout -> decoder -> softmax, one fused rollout."""

    grad_mode = "adjoint"      # what the reference trains with (torchdiffeq odeint_adjoint)

    def __init__(self, maxTime, deltaT, n_nodes, indices, hidden1, odefunc, device):
        super().__init__()
        self.maxTime = maxTime
        self.deltaT = deltaT
        self.device = device
        self.integration_time = torch.from_numpy(np.arange(0, self.maxTime, self.deltaT)).to(device)
        self.odefunc = odefunc
        self.n_nodes = n_nodes
        self.indices = torch.tensor(indices, requires_grad=False)
        self.hidden1 = hidden1
        self.linearS1 = nn.Linear(1, hidden1)
        self.ln = nn.LayerNorm(hidden1)
        self.linear3 = nn.Linear(hidden1, 4)
        self.relu3 = nn.ReLU()
        self.linearS2 = nn.Linear(4, 1)
        self.softmax = nn.Softmax(dim=2)
        self.relu = nn.ReLU()
        self.dropout = nn.Dropout(0.2)
        self._dt = _ro.dt_array(self.integration_time)

    def _params(self):
        return _ro.padded_params(self.odefunc.linear.weight, self.odefunc.linear.bias, self.linearS1.weight,
                                 self.linearS1.bias, self.linear3.weight, self.linear3.bias, self.linearS2.weight,
                                 self.linearS2.bias)

    def _finish(self, probs):
        # adjoint parameters that never enter f get ZERO gradients in the reference (torchdiffeq
        # returns zeros for unused adjoint params): keep Adam's view of odefunc.ln identical
        if probs.requires_grad:
            probs = probs + 0.0 * (self.odefunc.ln.weight.sum() + self.odefunc.ln.bias.sum())
        return probs

    def rollout_probs(self, x, out_steps=None):
        """x [B, N, 3+H] -> probabilities [T (or len(out_steps)), B*N, 3] in one tensor."""
        x = x.view(-1, x.size(-1))                     # [B*N, 3+H]
        n_trials = x.size(0) // self.odefunc.device_graph().n
        batch = self.odefunc.batch_for(n_trials)
        return self._finish(_ro.rollout(x, batch, self._dt, self._params(), self.grad_mode, out_steps))

    def forward(self, x):
        S, I, R = self.rollout_probs(x).chunk(3, dim=-1)               # each [T, M, 1]
        return S, I, R

    def forward_trials(self, seeds, beta, gamma, out_steps=None, probs_out=None, workspace=None):
        """The same rollout from compact trial descriptors (N4): seeds[i] = node ids infected at t = 0 in trial i,
        beta[i], gamma[i] -- instead of the dense [N, 3+H] block per trial main() builds (ode_nn_ngraph_sim.py:371-390).
        Returns (S, I, R), each [T (or len(out_steps)), B*N, 1]. beta / gamma given as tensors that require grad receive
        dL/dbeta[i], dL/dgamma[i] (calibration of a trial through the trained model)."""
        is_set = isinstance(seeds, _ro.TrialSet)                      # a prepared (device-resident) descriptor set
        batch = self.odefunc.batch_for(seeds.n_inst if is_set else len(seeds))
        dev = self.linearS1.weight.device
        trials = seeds if is_set else _ro.TrialSet(seeds, beta, gamma, batch.sizes, dev)
        probs = self._finish(_ro.rollout_trials(batch, trials, self._dt, self._params(), self.grad_mode, out_steps,
                                                probs_out, workspace, *((None, None) if is_set else (beta, gamma))))
        return probs.chunk(3, dim=-1)
