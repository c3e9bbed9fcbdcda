"""torch.autograd.Function around the C-ABI rollout (forward + reverse sweep).

PyTorch is plumbing here: it owns device memory, the stream and autograd's graph;
all arithmetic of the path runs in libgnode_b200.so.
"""
import ctypes
import os

import numpy as np
import torch

from . import _lib

H = _lib.GNODE_H
# training keeps I'_k and A I'_k of every Euler step beside the trajectory (5 instead of 3 state planes per grid point)
# so that the reverse sweep gathers once per step; False = trajectory only (less memory, two gathers per reverse step)
AUX_STORAGE = os.environ.get("GNODE_AUX_STORAGE", "1") != "0"
PARAM_ORDER = tuple(k for k, _ in _lib.GRAD_LAYOUT)


def check_hidden(hidden1, need_marker=False):
    """Hidden widths up to 64 run on the 64-wide kernels (narrower ones zero-padded, see padded_params); wider ones
    are not supported."""
    lo = 3 if need_marker else 2            # the input block carries beta, gamma (and the graph marker) in its bg columns
    if not (lo <= int(hidden1) <= H):
        raise NotImplementedError("the B200 kernels support hidden widths %d..%d (got %d)" % (lo, H, hidden1))


def pad_linear(W, b):
    h = W.size(0)
    if h == H:
        return W, b
    return torch.nn.functional.pad(W, (0, H - h, 0, H - h)), torch.nn.functional.pad(b, (0, H - h))


def pad_channels(y):
    h = y.size(-1)
    return y if h == H else torch.nn.functional.pad(y, (0, H - h))


def padded_params(lin_w, lin_b, s1_w, s1_b, l3_w, l3_b, s2_w, s2_b):
    """Parameters in PARAM_ORDER, embedded into the 64-wide kernels when hidden < 64: the extra channels start at
    relu(0 * c + 0) = 0, evolve on their own (sigmoid(0) = 0.5 feeds only themselves: the padded rows AND columns of
    linear.weight are zero) and are ignored by the decoder (zero linear3 columns), so the real channels compute exactly
    the hidden-wide model; autograd slices the gradients back through the pads."""
    h = lin_w.size(0)
    if h == H:
        return [lin_w, lin_b, s1_w, s1_b, l3_w, l3_b, s2_w, s2_b]
    pad = torch.nn.functional.pad
    W, b = pad_linear(lin_w, lin_b)
    return [W, b, pad(s1_w, (0, 0, 0, H - h)), pad(s1_b, (0, H - h)), pad(l3_w, (0, H - h)), l3_b, s2_w, s2_b]


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def _stream(device=None):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _steps_arg(out_steps, T):
    """out_steps (None | sequence of grid indices) -> (int32 array or None, ctypes pointer or None, n_out)."""
    if out_steps is None:
        return None, None, T
    arr = np.ascontiguousarray(np.asarray(out_steps, dtype=np.int32))
    if arr.ndim != 1 or len(arr) == 0 or np.any(np.diff(arr) <= 0) or arr[0] < 0 or arr[-1] >= T:
        raise ValueError("out_steps must be strictly ascending grid indices in [0, %d), got %r" % (T, out_steps))
    return arr, arr.ctypes.data_as(_lib.c_int32_p), len(arr)


def unit_time_steps(maxTime, deltaT):
    """Grid indices int(i/deltaT), i = 0..maxTime-1: the rows get_sir_t_nodes_torch picks (ode_nn.py:249-261)."""
    return np.asarray([int(i / deltaT) for i in range(int(maxTime))], dtype=np.int32)


def _params_struct(tensors):
    return _lib.GnodeParams(*[t.data_ptr() for t in tensors])


def _check_cuda_f32(t, name):
    if not t.is_cuda:
        raise RuntimeError("%s must be a CUDA tensor: the GN-ODE rollout has no CPU path (got %s)" % (name, t.device))
    if t.dtype != torch.float32:
        raise RuntimeError("%s must be float32 (got %s)" % (name, t.dtype))


def dt_array(integration_time):
    """dt_k = float32(t_{k+1} - t_k) computed in float64 like torchdiffeq's fixed grid."""
    t = np.asarray(integration_time.detach().cpu().numpy() if torch.is_tensor(integration_time)
                   else integration_time, dtype=np.float64)
    return np.ascontiguousarray((t[1:] - t[:-1]).astype(np.float32))


class _Rollout(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, batch, dt, grad_mode, want_grad, out_steps, *params):
        L = _lib.lib()
        M, T = batch.M, len(dt) + 1
        steps, steps_p, n_out = _steps_arg(out_steps, T)
        _check_cuda_f32(x, "x")
        if x.dim() != 2 or x.size(0) != M or x.size(1) < 5 or x.stride(1) != 1:
            raise RuntimeError("x must be [M=%d, >=5] with unit column stride, got %r" % (M, tuple(x.shape)))
        ps = []
        for k, p in zip(PARAM_ORDER, params):
            _check_cuda_f32(p, k)
            ps.append(p.detach().contiguous())
        # grad mode is always off inside forward(): the caller's grad mode arrives as `want_grad`
        need_grad = bool(want_grad) and (ctx.needs_input_grad[0] or any(ctx.needs_input_grad[6:]))
        with torch.cuda.device(x.device):
            traj = torch.empty((T, 3, M, H), dtype=torch.float32, device=x.device) if need_grad else None
            probs = torch.empty((n_out, M, 3), dtype=torch.float32, device=x.device)
            ws_bytes = int(L.gnode_rollout_workspace_bytes(batch.handle, 1 if need_grad else 0))
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
            pstruct = _params_struct(ps)
            # training: I'_k and A I'_k of every step are kept for the reverse sweep (one neighbour gather per reverse
            # step instead of two, no recomputed I'); AUX_STORAGE = False restores the trajectory-only sweep
            aux, filled = None, ctypes.c_int32(0)
            if need_grad and AUX_STORAGE and T > 1:
                try:
                    aux = torch.empty(int(L.gnode_rollout_aux_bytes(batch.handle, T)) // 4, dtype=torch.float32, device=x.device)
                except torch.cuda.OutOfMemoryError:          # 2/3 of the trajectory's size on top of it: optional
                    aux = None
            _lib.check(L.gnode_rollout_forward_aux(batch.handle, _ptr(x), x.stride(0), ctypes.byref(pstruct), T,
                                                   dt.ctypes.data_as(_lib.c_float_p), steps_p, n_out,
                                                   _ptr(traj) if need_grad else None,
                                                   _ptr(aux) if aux is not None else None, ctypes.byref(filled),
                                                   _ptr(probs), _ptr(ws), ws_bytes,
                                                   _stream(x.device)), "gnode_rollout_forward_aux")
        if need_grad:
            ctx.save_for_backward(x, traj, *ps)
            ctx.batch, ctx.dt, ctx.grad_mode, ctx.steps = batch, dt, grad_mode, steps
            ctx.aux = aux if filled.value == 1 else None
            ctx.wgrad = any(ctx.needs_input_grad[6:])       # False: input gradients only (no weight-gradient phase)
        return probs

    @staticmethod
    def backward(ctx, grad_probs):
        L = _lib.lib()
        x, traj, *ps = ctx.saved_tensors
        batch, dt = ctx.batch, ctx.dt
        T = len(dt) + 1
        grad_probs = grad_probs.contiguous()
        _check_cuda_f32(grad_probs, "grad_probs")
        steps = ctx.steps
        steps_p = steps.ctypes.data_as(_lib.c_int32_p) if steps is not None else None
        with torch.cuda.device(x.device):
            grads = torch.empty(_lib.GRAD_COUNT, dtype=torch.float32, device=x.device) if ctx.wgrad else None
            # dL/dx: columns 0..4 written by the sweep, the others (graph marker, unused bg channels) carry no gradient
            grad_x = torch.zeros(tuple(x.shape), dtype=torch.float32, device=x.device) if ctx.needs_input_grad[0] else None
            ws_bytes = int(L.gnode_backward_workspace_bytes(batch.handle))
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
            pstruct = _params_struct(ps)
            mode = {"adjoint": _lib.GRAD_ADJOINT, "discrete": _lib.GRAD_DISCRETE}[ctx.grad_mode]
            _lib.check(L.gnode_rollout_backward_input(batch.handle, _ptr(x), x.stride(0), ctypes.byref(pstruct), T,
                                                      dt.ctypes.data_as(_lib.c_float_p), _ptr(traj),
                                                      _ptr(ctx.aux) if ctx.aux is not None else None, _ptr(grad_probs),
                                                      steps_p, len(steps) if steps is not None else 0, mode,
                                                      _ptr(grads) if grads is not None else None,
                                                      _ptr(grad_x) if grad_x is not None else None,
                                                      grad_x.stride(0) if grad_x is not None else 0,
                                                      _ptr(ws), ws_bytes, _stream(x.device)),
                       "gnode_rollout_backward_input")
        out, off = [], 0
        for i, (k, shape) in enumerate(_lib.GRAD_LAYOUT):
            n = int(np.prod(shape))
            out.append(grads[off:off + n].view(shape) if ctx.needs_input_grad[6 + i] else None)
            off += n
        return (grad_x, None, None, None, None, None, *out)


def rollout(x, batch, dt, params, grad_mode="adjoint", out_steps=None):
    """x [M, >=5] -> probabilities [T, M, 3] (or [len(out_steps), M, 3]: only those grid points are decoded and
    stored); params in PARAM_ORDER (state_dict names). Differentiable with respect to the parameters and to x (columns
    S0, I0, R0, beta, gamma; the other columns get zero gradients)."""
    if grad_mode not in ("adjoint", "discrete"):
        raise ValueError("grad_mode must be 'adjoint' or 'discrete'")
    want_grad = torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in params))
    return _Rollout.apply(x, batch, dt, grad_mode, want_grad, out_steps, *params)


class TrialSet:
    """Compact trial descriptors of one batch (N4): per instance the seed list (instance-local node ids), beta and
    gamma -- what main() expands into a dense [N, 3+H] block per trial on the host (ode_nn_ngraph_sim.py:371-390).
    A few KB per batch instead of 268 B per row. device=None keeps the set in pinned host memory (a dataset of
    batches that a streaming loop copies into a device-resident set with copy_from). beta and gamma may be sequences or
    torch tensors; the set keeps detached copies (gradients reach them through rollout_trials' beta / gamma)."""

    def __init__(self, seeds, beta, gamma, sizes, device=None):
        if not (len(seeds) == len(beta) == len(gamma) == len(sizes)):
            raise ValueError("seeds, beta, gamma and sizes must have one entry per instance")
        ptr = np.zeros(len(seeds) + 1, dtype=np.int32)
        flat = []
        for i, (sd, n) in enumerate(zip(seeds, sizes)):
            sd = np.asarray(sd, dtype=np.int64).reshape(-1)
            if len(sd) and (sd.min() < 0 or sd.max() >= n):
                raise ValueError("instance %d: seed %d outside [0, %d)" % (i, int(sd.max() if sd.max() >= n else sd.min()), n))
            flat.append(sd.astype(np.int32))
            ptr[i + 1] = ptr[i] + len(sd)
        self.n_inst = len(seeds)
        hi = torch.from_numpy(np.concatenate([ptr] + flat))
        host = lambda v: v.detach().to("cpu", torch.float32).numpy() if torch.is_tensor(v) else v
        hf = torch.from_numpy(np.concatenate([np.asarray(host(beta), dtype=np.float32).reshape(-1),
                                              np.asarray(host(gamma), dtype=np.float32).reshape(-1)]))
        if torch.cuda.is_available():
            hi, hf = hi.pin_memory(), hf.pin_memory()
        self._host = (hi, hf)
        if device is None:
            self._bind(hi, hf)
        else:
            self._bind(hi.to(device, non_blocking=True), hf.to(device, non_blocking=True))

    def _bind(self, ti, tf):
        self._i, self._f = ti, tf
        self.seed_ptr, self.seeds = ti[:self.n_inst + 1], ti[self.n_inst + 1:]
        self.beta, self.gamma = tf[:self.n_inst], tf[self.n_inst:]
        self.h2d_bytes = ti.numel() * 4 + tf.numel() * 4

    def to(self, device):
        """A copy of this set on `device` (two small asynchronous copies from pinned memory)."""
        out = object.__new__(TrialSet)
        out.n_inst, out._host = self.n_inst, self._host
        out._bind(self._i.to(device, non_blocking=True), self._f.to(device, non_blocking=True))
        return out

    def copy_from(self, other, non_blocking=True):
        """Overwrite this (device) set with another set of the same shape (e.g. the next batch of a pinned dataset)."""
        if other._i.shape != self._i.shape or other._f.shape != self._f.shape:
            raise ValueError("trial sets differ in shape")
        self._i.copy_(other._i, non_blocking=non_blocking)
        self._f.copy_(other._f, non_blocking=non_blocking)
        return self


def expand_trials(batch, trials, ldx=_lib.GNODE_TRIAL_LDX):
    """TrialSet -> x [M, ldx] with the five live columns S0 I0 R0 beta gamma (the rest is uninitialised and never read)."""
    L = _lib.lib()
    if trials.n_inst != len(batch.sizes):
        raise ValueError("%d trial descriptors for a batch of %d instances" % (trials.n_inst, len(batch.sizes)))
    dev = trials.beta.device
    with torch.cuda.device(dev):
        x = torch.empty((batch.M, ldx), dtype=torch.float32, device=dev)
        _lib.check(L.gnode_expand_trials(batch.handle, _ptr(trials.seeds) if trials.seeds.numel() else _ptr(trials.seed_ptr),
                                         _ptr(trials.seed_ptr), _ptr(trials.beta), _ptr(trials.gamma), _ptr(x), ldx,
                                         _stream(dev)), "gnode_expand_trials")
    return x


class _ExpandTrials(torch.autograd.Function):
    """expand_trials as a function of the descriptors' beta and gamma: dL/dbeta[i] and dL/dgamma[i] are the sums of
    dL/dx[:, 3] and dL/dx[:, 4] over the rows of instance i (gnode_trials_grad, fixed summation order)."""

    @staticmethod
    def forward(ctx, beta, gamma, batch, trials):
        ctx.batch = batch
        ctx.meta = [(t.shape, t.dtype, t.device) for t in (beta, gamma)]
        return expand_trials(batch, trials)

    @staticmethod
    def backward(ctx, gx):
        L = _lib.lib()
        gx = gx.contiguous()
        n = len(ctx.batch.sizes)
        with torch.cuda.device(gx.device):
            gbg = torch.empty((2, n), dtype=torch.float32, device=gx.device)
            _lib.check(L.gnode_trials_grad(ctx.batch.handle, _ptr(gx), gx.stride(0), _ptr(gbg[0]), _ptr(gbg[1]),
                                           _stream(gx.device)), "gnode_trials_grad")
        out = [g.reshape(shape).to(device=dev, dtype=dtype) for g, (shape, dtype, dev) in zip(gbg, ctx.meta)]
        return out[0], out[1], None, None


def rollout_trials(batch, trials, dt, params, grad_mode="adjoint", out_steps=None, probs_out=None, workspace=None,
                   beta=None, gamma=None):
    """Rollout straight from compact trial descriptors. Without gradients: ONE C-ABI call (expansion into the
    workspace + rollout), optionally into caller-owned `probs_out` / `workspace` buffers (streaming loops reuse them).
    With gradients: the compact x is kept for the reverse sweep. `beta` / `gamma`: the tensors the set was made from;
    when one of them requires grad, it receives dL/dbeta[i] (dL/dgamma[i]) per instance. Seed sets are discrete and
    have no gradient."""
    want_x = torch.is_grad_enabled() and any(torch.is_tensor(v) and v.requires_grad for v in (beta, gamma))
    want_grad = want_x or (torch.is_grad_enabled() and any(p.requires_grad for p in params))
    if want_grad:
        if want_x:
            bt = beta if torch.is_tensor(beta) else trials.beta
            gt = gamma if torch.is_tensor(gamma) else trials.gamma
            if bt.numel() != trials.n_inst or gt.numel() != trials.n_inst:
                raise ValueError("beta and gamma must hold one value per instance (%d)" % trials.n_inst)
            x = _ExpandTrials.apply(bt, gt, batch, trials)
        else:
            x = expand_trials(batch, trials)
        return rollout(x, batch, dt, params, grad_mode, out_steps)
    L = _lib.lib()
    if trials.n_inst != len(batch.sizes):
        raise ValueError("%d trial descriptors for a batch of %d instances" % (trials.n_inst, len(batch.sizes)))
    dev = trials.beta.device
    T = len(dt) + 1
    steps, steps_p, n_out = _steps_arg(out_steps, T)
    ps = []
    for k, p in zip(PARAM_ORDER, params):
        _check_cuda_f32(p, k)
        ps.append(p.detach().contiguous())
    with torch.cuda.device(dev):
        ws_bytes = int(L.gnode_rollout_trials_workspace_bytes(batch.handle, 0))
        if workspace is None:
            workspace = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        elif workspace.numel() < ws_bytes:
            raise ValueError("workspace too small: %d < %d bytes" % (workspace.numel(), ws_bytes))
        if probs_out is None:
            probs_out = torch.empty((n_out, batch.M, 3), dtype=torch.float32, device=dev)
        elif tuple(probs_out.shape) != (n_out, batch.M, 3) or not probs_out.is_contiguous():
            raise ValueError("probs_out must be a contiguous [%d, %d, 3] tensor" % (n_out, batch.M))
        pstruct = _params_struct(ps)
        _lib.check(L.gnode_rollout_forward_trials(batch.handle, _ptr(trials.seeds) if trials.seeds.numel() else _ptr(trials.seed_ptr),
                                                  _ptr(trials.seed_ptr), _ptr(trials.beta), _ptr(trials.gamma),
                                                  ctypes.byref(pstruct), T, dt.ctypes.data_as(_lib.c_float_p), steps_p, n_out,
                                                  None, _ptr(probs_out), _ptr(workspace), workspace.numel(), _stream(dev)),
                   "gnode_rollout_forward_trials")
    return probs_out


class _L1Subsampled(torch.autograd.Function):
    @staticmethod
    def forward(ctx, probs, labels, skip, scale):
        L = _lib.lib()
        _check_cuda_f32(probs, "probs")
        if labels.dtype != torch.float64 or not labels.is_cuda:
            raise RuntimeError("labels must be a float64 CUDA tensor [M, n_out, 3] (the reference's label dtype)")
        n_out, M = probs.size(0), probs.size(1)
        labels = labels.reshape(-1, labels.size(-2), labels.size(-1)).contiguous()
        if tuple(labels.shape) != (M, n_out, 3):
            raise RuntimeError("labels %r do not match probs %r" % (tuple(labels.shape), tuple(probs.shape)))
        probs = probs.contiguous()
        need = ctx.needs_input_grad[0]
        with torch.cuda.device(probs.device):
            loss = torch.empty((), dtype=torch.float64, device=probs.device)
            grad = torch.empty_like(probs) if need else None
            scratch = torch.empty(int(L.gnode_l1_scratch_bytes()), dtype=torch.uint8, device=probs.device)
            _lib.check(L.gnode_l1_loss_grad(_ptr(probs), _ptr(labels), M, n_out, int(skip), float(scale), _ptr(loss),
                                            _ptr(grad) if need else None, _ptr(scratch), _stream(probs.device)),
                       "gnode_l1_loss_grad")
        if need:
            ctx.save_for_backward(grad)
        return loss

    @staticmethod
    def backward(ctx, g):
        (grad,) = ctx.saved_tensors
        return grad * g.to(grad.dtype), None, None, None


def l1_subsampled(probs, labels, skip=1, scale=1.0):
    """Mean |probs[t, m, c] - labels[m, t, c]| over t >= skip (float64, like the reference's promoted nn.L1Loss on
    [:, 1:, :]) with the cotangent written in the same pass. probs [n_out, M, 3] fp32, labels [M, n_out, 3] fp64.
    `scale` multiplies the cotangent only (data-parallel shards pass their share of the global item count)."""
    return _L1Subsampled.apply(probs, labels, skip, scale)


def odefunc_eval(y, beta, gamma, batch, params):
    """One f(t, y): y [3, M, H] -> [3, M, H] (dS, dI, dR). Not differentiable."""
    L = _lib.lib()
    for t, n in ((y, "y"), (beta, "beta"), (gamma, "gamma")):
        _check_cuda_f32(t, n)
    y, beta, gamma = y.contiguous(), beta.contiguous(), gamma.contiguous()
    ps = [p.detach().contiguous() for p in params]
    dy = torch.empty_like(y)
    scratch = torch.empty((batch.M, H), dtype=torch.float32, device=y.device)
    pstruct = _params_struct(ps)
    _lib.check(L.gnode_odefunc_eval(batch.handle, _ptr(y), _ptr(beta), _ptr(gamma), ctypes.byref(pstruct),
                                    _ptr(dy), _ptr(scratch), _stream()), "gnode_odefunc_eval")
    return dy


def aggregate(v, batch, transpose=False):
    """out[r] = sum of v over the neighbours of r. v: [M, H]."""
    L = _lib.lib()
    _check_cuda_f32(v, "v")
    v = v.contiguous()
    out = torch.empty_like(v)
    _lib.check(L.gnode_aggregate(batch.handle, _ptr(v), _ptr(out), 1 if transpose else 0, _stream()),
               "gnode_aggregate")
    return out
