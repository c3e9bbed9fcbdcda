"""Drop-in ``ODEfunc`` / ``ODEBlock`` for the multi-graph script.

Mirrors /root/reference/ode_nn_ngraphs.py:37-83 (ODEfunc) and :86-152 (ODEBlock):
the state is the ragged concatenation of instances along the node axis and every
instance names its graph through the marker ``x[first row of instance, 5]`` =
graph index + 1 (ode_nn_ngraphs.py:55,65-67,333).
"""
import numpy as np
import torch
import torch.nn as nn

from . import rollout as _ro
from .graph import BatchCache, DeviceGraph


class ODEfunc(nn.Module):
    def __init__(self, A_list, hidden1, device):
        super().__init__()
        _ro.check_hidden(hidden1, need_marker=True)
        self.hidden1 = hidden1
        self.A_list = A_list
        self.ln = nn.LayerNorm(hidden1)
        self.linear = nn.Linear(hidden1, hidden1)
        self.relu = nn.ReLU()
        self.sigmoid = nn.Sigmoid()
        self._graphs = None
        self._batches = BatchCache()
        self._marker_cache = {}

    def device_graphs(self):
        if self._graphs is None:
            self._graphs = [DeviceGraph(A) for A in self.A_list]
        return self._graphs

    def batch_from_instances(self, graph_ids):
        """Batch of the instances graph_ids[i] (0-based indices into A_list): no device read."""
        graphs = self.device_graphs()
        return self._batches.get([graphs[int(g)] for g in graph_ids])

    def batch_from_markers(self, marker_col):
        """marker_col: x[:, 5] (device or host). Non-zero entries open an instance. A device column costs one
        device -> host copy (a stream sync): the result is remembered per (storage, version) of the input tensor, so a
        loader batch that stays on the device resolves its instances once, not once per forward (the reference's
        torch.nonzero(x[3,:,2]) at ode_nn_ngraphs.py:55 runs at every Euler step)."""
        key = (marker_col.data_ptr(), marker_col.numel(), marker_col.stride(0), marker_col._version, str(marker_col.device))
        hit = self._marker_cache.get(key)
        if hit is not None:
            return hit
        batch = self._batch_from_marker_values(marker_col.detach().to("cpu", torch.float32).numpy())
        if len(self._marker_cache) >= 256:
            self._marker_cache.clear()
        self._marker_cache[key] = batch
        return batch

    def _batch_from_marker_values(self, mk):
        starts = np.flatnonzero(mk)
        gids = mk[starts].astype(np.int64) - 1
        graphs = self.device_graphs()
        if len(starts) == 0 or starts[0] != 0:
            raise RuntimeError("the first row of the batch must carry a graph marker (ode_nn_ngraphs.py:333)")
        sizes = np.diff(np.append(starts, len(mk)))
        for s, g in zip(sizes, gids):
            if g < 0 or g >= len(graphs) or graphs[g].n != s:
                raise RuntimeError("instance of %d rows does not match graph %d" % (s, g))
        return self._batches.get([graphs[g] for g in gids])

    def forward(self, t, x):
        """f(t, y) on the stacked state [4, sum N, H] (ode_nn_ngraphs.py:54-83); inference-only."""
        batch = self.batch_from_markers(x[3, :, 2])
        h = x.size(2)
        W, b = _ro.pad_linear(self.linear.weight, self.linear.bias)
        dy = _ro.odefunc_eval(_ro.pad_channels(x[:3]), x[3, :, 0], x[3, :, 1], batch, [W, b] + [b] * 6)[..., :h]
        return torch.cat((dy, torch.zeros_like(x[3:])))


class ODEBlock(nn.Module):
    grad_mode = "adjoint"

    def __init__(self, maxTime, deltaT, hidden1, odefunc, device):
        super().__init__()
        self.maxTime = maxTime
        self.deltaT = deltaT
        self.device = device
        self.integration_time = torch.from_numpy(np.arange(0, self.maxTime, self.deltaT)).to(device)
        self.odefunc = odefunc
        self.hidden1 = hidden1
        self.linearS1 = nn.Linear(1, hidden1)
        self.ln = nn.LayerNorm(hidden1)
        self.linear3 = nn.Linear(hidden1, 4)
        self.relu3 = nn.ReLU()
        self.linearS2 = nn.Linear(4, 1)
        self.softmax = nn.Softmax(dim=2)
        self.relu = nn.ReLU()
        self._dt = _ro.dt_array(self.integration_time)

    def _params(self):
        return _ro.padded_params(self.odefunc.linear.weight, self.odefunc.linear.bias, self.linearS1.weight,
                                 self.linearS1.bias, self.linear3.weight, self.linear3.bias, self.linearS2.weight,
                                 self.linearS2.bias)

    def _finish(self, probs):
        if probs.requires_grad:
            probs = probs + 0.0 * (self.odefunc.ln.weight.sum() + self.odefunc.ln.bias.sum())
        return probs

    def rollout_probs(self, x, out_steps=None, instances=None, *, edge_weight=None, contact_weight=None):
        """x [sum N, 3+H] -> probabilities [T (or len(out_steps)), sum N, 3]. `instances` (graph index per instance)
        spares the marker column's device read when the caller knows its batch. edge_weight: all-ones CUDA tensor of the
        batch's nnz (instance after instance, each in its graph's DeviceGraph.edges() order); when it requires grad it
        receives dL/dw of every stored adjacency entry. contact_weight: the weights the neighbour sum runs with, same
        layout, any finite values; when it requires grad it receives dL/dw at those weights."""
        batch = self.odefunc.batch_from_instances(instances) if instances is not None \
            else self.odefunc.batch_from_markers(x[:, 5])
        if batch.M != x.size(0):
            raise RuntimeError("batch of %d rows for an input of %d rows" % (batch.M, x.size(0)))
        return self._finish(_ro.rollout(x, batch, self._dt, self._params(), self.grad_mode, out_steps, edge_weight,
                                        contact_weight))

    def forward(self, x, instances=None, *, edge_weight=None, contact_weight=None):
        S, I, R = self.rollout_probs(x, instances=instances, edge_weight=edge_weight,
                                    contact_weight=contact_weight).chunk(3, dim=-1)
        return S, I, R

    def forward_trials(self, instances, seeds, beta, gamma, out_steps=None, *, edge_weight=None, contact_weight=None):
        """Rollout from compact descriptors (N4): instance i runs on graph instances[i] with seeds[i], beta[i], gamma[i]
        (replaces the dense per-instance blocks of ode_nn_ngraphs.py:326-345). Returns (S, I, R). beta / gamma given as
        tensors that require grad receive dL/dbeta[i], dL/dgamma[i]; edge_weight and contact_weight as in rollout_probs."""
        batch = self.odefunc.batch_from_instances(instances)
        trials = _ro.TrialSet(seeds, beta, gamma, batch.sizes, self.linearS1.weight.device)
        probs = self._finish(_ro.rollout_trials(batch, trials, self._dt, self._params(), self.grad_mode, out_steps,
                                                beta=beta, gamma=gamma, edge_weight=edge_weight,
                                                contact_weight=contact_weight))
        return probs.chunk(3, dim=-1)
