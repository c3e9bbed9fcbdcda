"""Graph structure the golden fixtures never reach (tests/_graphs.py): a directed graph, where A and its transpose differ,
a graph without edges, a symmetric graph with one entry removed, and a batch of one-node, small directed, symmetric and
edgeless instances with an instance boundary at every offset inside a tile.

On a symmetric pattern the transpose CSR is A itself (gnode_graph_create aliases the two), so only these graphs check
that the reverse sweep gathers A^T gAI over the transpose (bwd_gz_kernel), that the transpose is uploaded separately,
and that the input gradients resting on it are right. The forward, the reverse sweep, the descriptor path and the
Monte-Carlo kernel are compared with the float64 oracle (orc.loss_and_grads, tests/_input_grad_oracle.py) and the
numpy process. The CPU tests at the end prove from the oracle alone that the GPU tests would fail if the reverse sweep
gathered over A instead of A^T, or if the Monte-Carlo process spread infection against the edge direction."""
import ctypes
import functools

import numpy as np
import pytest
import torch

import _graphs
from _input_grad_oracle import loss_and_input_grads
from oracle import gnode_oracle as orc

DEV = "cuda:0"
H = 64
MAXTIME, DELTAT = 5, 0.5                     # T = 10
PARAM_SEED = 31
PARAM_ORDER = ("odefunc.linear.weight", "odefunc.linear.bias", "linearS1.weight", "linearS1.bias",
               "linear3.weight", "linear3.bias", "linearS2.weight", "linearS2.bias")
STEP_KERNELS = {5: "stream", 6: "stream-barrier", 7: "stream-3xtf32", 3: "dual", 0: "generic"}
gpu = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------------------- inputs
@functools.lru_cache(maxsize=None)
def case(name):
    """(graphs, inst, seeds, beta, gamma): distinct graphs, graph of every instance, per-instance descriptors."""
    if name == "directed":                   # trial 0 seeds the in-hub and a sink: A and A^T differ most there
        return ([_graphs.directed()], [0, 0], [[_graphs.IN_HUB, int(_graphs.SINKS[0])], [_graphs.OUT_HUB, 123]],
                [0.3, 0.15], [0.2, 0.35])
    if name == "directed-probe":             # trial 0 of "directed" alone
        g, _, s, b, c = case("directed")
        return g, [0], s[:1], b[:1], c[:1]
    if name == "nearly_symmetric":
        graphs, inst = [_graphs.nearly_symmetric()], [0, 0]
    elif name == "edgeless":
        graphs, inst = [_graphs.edgeless()], [0, 0]
    elif name == "mixed":
        graphs, inst = _graphs.mixed()
    else:
        raise KeyError(name)
    seeds, beta, gamma = _graphs.trial_inputs([graphs[i].shape[0] for i in inst], seed=5)
    return graphs, inst, seeds, beta, gamma


def sizes_of(name):
    graphs, inst = case(name)[:2]
    return [graphs[i].shape[0] for i in inst]


def x_of(name):
    graphs, inst, seeds, beta, gamma = case(name)
    return torch.from_numpy(_graphs.dense_x(sizes_of(name), seeds, beta, gamma, H))


def coo_of(name):
    graphs, inst = case(name)[:2]
    return orc.batch_coo(graphs, inst)


def params():
    return orc.default_params(H, seed=PARAM_SEED)


def time_grid():
    return orc.time_grid(MAXTIME, DELTAT)


def unit_steps():
    return np.asarray(orc.unit_time_rows(MAXTIME, DELTAT), dtype=np.int32)


def cotangent(name, cot):
    """dense: w [T, M, 3] of L = sum(w * probs); sparse: labels y [M, maxTime, 3] of the L1 training loss at the unit-time
    grid points."""
    M = sum(sizes_of(name))
    if cot == "dense":
        return torch.randn(len(time_grid()), M, 3, generator=torch.Generator().manual_seed(9))
    return torch.rand(M, len(unit_steps()), 3, generator=torch.Generator().manual_seed(2), dtype=torch.float64)


def out_degree_zero_rows(name):
    """Rows whose CSR row of A is empty: A I' = 0 there, so dL/dbeta of the row is exactly 0."""
    graphs, inst = case(name)[:2]
    return np.concatenate([r + np.flatnonzero(np.diff(graphs[i].indptr) == 0)
                           for r, i in zip(_graphs.instance_rows(sizes_of(name)), inst)])


# ---------------------------------------------------------------------------------------------------------- oracle
_neighbour_sum = orc.neighbour_sum


class _GatherOverA(torch.autograd.Function):
    """The oracle's neighbour sum with a WRONG backward: A g instead of A^T g (what bwd_gz_kernel would compute if it
    read the CSR of A instead of its transpose)."""

    @staticmethod
    def forward(ctx, Ip, coo):
        ctx.coo = coo
        return _neighbour_sum(Ip, coo)

    @staticmethod
    def backward(ctx, g):
        return _neighbour_sum(g, ctx.coo), None


def _wrong_neighbour_sum(Ip, coo):
    return _GatherOverA.apply(Ip, coo)


@functools.lru_cache(maxsize=None)
def oracle(name, mode, cot, dtype="float32", gather_over_a=False):
    """({key: dL/dparam}, dL/dx[:, :5]) of the oracle in float32 or float64."""
    x, p, t = x_of(name), params(), time_grid()
    c = cotangent(name, cot)
    prev = torch.get_default_dtype()
    if dtype == "float64":
        torch.set_default_dtype(torch.float64)
        x, p = x.double(), {k: v.double() for k, v in p.items()}
        if cot == "dense":
            c = c.double()
    weight = c if cot == "dense" else (lambda probs: orc.train_loss(probs, c, MAXTIME, DELTAT))
    if gather_over_a:
        orc.neighbour_sum = _wrong_neighbour_sum
    try:
        _, grads, gx = loss_and_input_grads(x, p, coo_of(name), t, weight, mode)
    finally:
        orc.neighbour_sum = _neighbour_sum
        torch.set_default_dtype(prev)
    return grads, gx


def rel_err_params(got, want64):
    """{key: scale-relative max error}; the scale of a tensor is max |want|, and at least 1 for linearS2.bias, whose true
    gradient is exactly zero (softmax is shift invariant)."""
    out = {}
    for k in orc.GRAD_KEYS:
        scale = max(want64[k].abs().max().item(), 1.0 if k == "linearS2.bias" else 0.0)
        out[k] = (got[k].double() - want64[k]).abs().max().item() / scale
    return out


def rel_err_columns(got, want64):
    out = []
    for c in range(5):
        scale = want64[:, c].abs().max().item()
        out.append((got[:, c].double() - want64[:, c]).abs().max().item() / scale if scale > 0 else 0.0)
    return out


def bars(name, mode, cot):
    """The suite's bar per parameter tensor and per input column: max(1e-3, 2 x the fp32 oracle's error)."""
    want = oracle(name, mode, cot, "float64")
    ref = oracle(name, mode, cot, "float32")
    pb = {k: max(1e-3, 2.0 * e) for k, e in rel_err_params(ref[0], want[0]).items()}
    cb = [max(1e-3, 2.0 * e) for e in rel_err_columns(ref[1], want[1])]
    return pb, cb


def assert_grads_close(what, got_params, got_x, name, mode, cot):
    want_p, want_x = oracle(name, mode, cot, "float64")
    pb, cb = bars(name, mode, cot)
    if got_params is not None:
        for k, e in rel_err_params(got_params, want_p).items():
            print("%s %s: %.3e (bar %.3e)" % (what, k, e, pb[k]))
            assert e <= pb[k], (what, k, e, pb[k])
    for c, (e, col) in enumerate(zip(rel_err_columns(got_x, want_x), ("S0", "I0", "R0", "beta", "gamma"))):
        if want_x[:, c].abs().max().item() == 0.0:
            assert float(got_x[:, c].abs().max()) == 0.0, (what, col)
            continue
        print("%s dL/d%s: %.3e (bar %.3e)" % (what, col, e, cb[c]))
        assert e <= cb[c], (what, col, e, cb[c])


# ---------------------------------------------------------------------------------------------------------- catalogue
def test_directed_graph_is_asymmetric_with_hubs_in_both_directions():
    A = _graphs.directed()
    AT = A.T.tocsr()
    deg, deg_t = np.diff(A.indptr), np.diff(AT.indptr)
    assert (A != AT).nnz > 0 and A.has_sorted_indices
    assert deg.max() > 1536 and int(deg.argmax()) == _graphs.OUT_HUB          # beyond the staged CSR slice
    assert deg_t.max() > 1024 and int(deg_t.argmax()) == _graphs.IN_HUB       # a long row of A^T only
    assert deg_t[_graphs.OUT_HUB] < 32 and deg[_graphs.IN_HUB] < 32
    t = _graphs.OUT_HUB // _graphs.TILE                                     # the out-hub is alone in its tile
    assert np.sort(deg[t * _graphs.TILE:(t + 1) * _graphs.TILE])[-2] <= 512
    assert deg[_graphs.SINKS].max() == 0 and deg_t[_graphs.SINKS].min() > 0
    assert deg_t[_graphs.SOURCES].max() == 0 and deg[_graphs.SOURCES].min() > 0
    assert all(A[v, v] == 1 for v in _graphs.SELF_LOOPS)
    assert all(A[u, v] == 1 and A[v, u] == 1 for u, v in _graphs.MUTUAL)


def test_mixed_batch_has_a_boundary_at_every_tile_offset():
    graphs, inst = _graphs.mixed()
    sizes = [graphs[i].shape[0] for i in inst]
    assert inst.count(0) == 200 and sizes[inst.index(5)] == 300 and graphs[5].nnz == 0
    assert sorted(graphs[i].shape[0] for i in (1, 2, 3)) == [127, 128, 129]
    assert all((graphs[i] != graphs[i].T).nnz > 0 for i in (1, 2, 3))
    assert (graphs[4] != graphs[4].T).nnz == 0
    assert set((_graphs.instance_rows(sizes) % _graphs.TILE).tolist()) == set(range(_graphs.TILE))


def test_nearly_symmetric_differs_from_its_transpose_in_one_entry():
    A = _graphs.nearly_symmetric()
    assert (A != A.T).nnz == 2 and A.nnz % 2 == 1


# ---------------------------------------------------------------------------------------------------------- GPU helpers
@pytest.fixture(scope="module")
def gn():
    import gn_ode_sir_b200 as g
    g.build_library()
    return g


@pytest.fixture(scope="module")
def lib(gn):
    from gn_ode_sir_b200 import _lib
    return _lib


@pytest.fixture(scope="module")
def batches(gn):
    cache = {}

    def get(name):
        if name not in cache:
            graphs, inst = case(name)[:2]
            dg = [gn.DeviceGraph(A) for A in graphs]
            cache[name] = (dg, gn.DeviceBatch([dg[i] for i in inst]))
        return cache[name][1]
    return get


class switches:
    """Sets process-wide kernel switches for a block and restores every one of them (and AUX_STORAGE) on exit."""
    NAMES = ("step_kernel", "variant", "persistent", "hub_relay", "bwd_kernel", "r_state")

    def __init__(self, gn, lib, **kw):
        self.gn, self.lib, self.kw = gn, lib, kw

    def __enter__(self):
        L = self.lib.lib()
        self.prev = {n: getattr(L, "gnode_get_" + n)() for n in self.NAMES}
        self.prev_aux = self.gn.rollout.AUX_STORAGE
        return self

    def set(self, **kw):
        L = self.lib.lib()
        for n, v in kw.items():
            if n == "aux":
                self.gn.rollout.AUX_STORAGE = v
            else:
                self.lib.check(getattr(L, "gnode_set_" + n)(v), "gnode_set_" + n)
        return self

    def __exit__(self, *exc):
        L = self.lib.lib()
        for n, v in self.prev.items():
            getattr(L, "gnode_set_" + n)(v)
        self.gn.rollout.AUX_STORAGE = self.prev_aux
        return False


def dev_params(requires_grad=False):
    p = params()
    return [p[k].to(DEV).requires_grad_(requires_grad) for k in PARAM_ORDER]


def infer(gn, batch, x):
    with torch.no_grad():
        out = gn.rollout.rollout(x.to(DEV), batch, gn.rollout.dt_array(time_grid()), dev_params())
    torch.cuda.synchronize()
    return out.cpu()


def train_forward(gn, batch, x):
    out = gn.rollout.rollout(x.to(DEV), batch, gn.rollout.dt_array(time_grid()), dev_params(True))
    return out.detach().cpu()


@functools.lru_cache(maxsize=None)
def oracle_probs(name):
    return orc.forward(x_of(name), params(), coo_of(name), time_grid())


def cuda_grads(gn, batch, x, mode, cot, c, frozen):
    """(dL/dx, {key: dL/dparam} or None) of one backward through rollout()."""
    ps = dev_params(not frozen)
    xin = x.to(DEV).clone().requires_grad_(True)
    dt = gn.rollout.dt_array(time_grid())
    if cot == "dense":
        loss = (gn.rollout.rollout(xin, batch, dt, ps, grad_mode=mode) * c.to(DEV)).sum()
    else:
        probs = gn.rollout.rollout(xin, batch, dt, ps, grad_mode=mode, out_steps=unit_steps())
        loss = gn.rollout.l1_subsampled(probs, c.to(DEV), skip=1)
    loss.backward()
    torch.cuda.synchronize()
    if frozen:
        assert all(p.grad is None for p in ps)
        return xin.grad.cpu(), None
    return xin.grad.cpu(), {k: p.grad.cpu() for k, p in zip(PARAM_ORDER, ps)}


# ---------------------------------------------------------------------------------------------------------- forward
@gpu
def test_graph_info_reports_symmetry(gn, batches):
    """gnode_graph_info: directed and nearly-symmetric patterns are not symmetric (their transpose is uploaded
    separately and the transposed aggregation equals the oracle's sum over A^T bitwise); edgeless and one-node graphs
    are."""
    for name in ("directed", "nearly_symmetric"):
        batch = batches(name)
        A = case(name)[0][0]
        assert not batch.graphs[0].symmetric
        assert batch.graphs[0].max_degree == int(np.diff(A.indptr).max())
        v = torch.rand(batch.M, H, generator=torch.Generator().manual_seed(3))
        assert torch.equal(gn.rollout.aggregate(v.to(DEV), batch).cpu(), orc.neighbour_sum(v, coo_of(name)))
        cooT = orc.batch_coo([A.T.tocsr()], [0, 0])
        assert torch.equal(gn.rollout.aggregate(v.to(DEV), batch, transpose=True).cpu(), orc.neighbour_sum(v, cooT))
    assert batches("directed").graphs[0].max_degree > 1536
    mixed, inst = batches("mixed"), case("mixed")[1]
    assert [mixed.graphs[inst.index(i)].symmetric for i in range(6)] == [True, False, False, False, True, True]
    assert batches("edgeless").graphs[0].symmetric and batches("edgeless").graphs[0].max_degree == 0


@gpu
@pytest.mark.parametrize("persistent", [0, 1], ids=["launch-per-step", "cooperative"])
@pytest.mark.parametrize("kernel", list(STEP_KERNELS), ids=list(STEP_KERNELS.values()))
@pytest.mark.parametrize("name", ["directed", "mixed"])
def test_step_kernels_against_oracle(gn, lib, batches, name, kernel, persistent):
    """Every step kernel (the generic one with the FFMA transform), both launch structures, inference and training
    forward, against the oracle's fp32 probabilities (bar 1e-5, as for the strict goldens)."""
    want = oracle_probs(name)
    with switches(gn, lib) as s:
        s.set(step_kernel=kernel, persistent=persistent)
        if kernel == 0:
            s.set(variant=0)
        inf = infer(gn, batches(name), x_of(name))
        trn = train_forward(gn, batches(name), x_of(name))
    for what, got in (("inference", inf), ("training", trn)):
        err = (got - want).abs().max().item()
        print("%s kernel %d persistent %d %s: %.3e" % (name, kernel, persistent, what, err))
        assert err < 1e-5, (what, err)
    assert (inf.sum(-1) - 1).abs().max().item() < 1e-6


@gpu
@pytest.mark.parametrize("persistent", [0, 1], ids=["launch-per-step", "cooperative"])
@pytest.mark.parametrize("name", ["directed", "mixed"])
def test_bitwise_promises_hold(gn, lib, batches, name, persistent):
    """Kernels 5, 6 and 3 issue the same operations: bitwise equal in inference and training forward. The hub relay is
    bitwise the serial walk (directed: the out-hub's tile takes the relay)."""
    batch, x = batches(name), x_of(name)
    out = {}
    with switches(gn, lib) as s:
        s.set(persistent=persistent)
        for k in (5, 6, 3):
            s.set(step_kernel=k)
            out[k] = (infer(gn, batch, x), train_forward(gn, batch, x))
        for k in (5, 3):
            s.set(step_kernel=k, hub_relay=0)
            serial = infer(gn, batch, x)
            s.set(hub_relay=1)
            assert torch.equal(serial, out[k][0]), (k, (serial - out[k][0]).abs().max().item())
    for k in (6, 3):
        assert torch.equal(out[k][0], out[5][0]), ("inference", k)
        assert torch.equal(out[k][1], out[5][1]), ("training", k)


@gpu
@pytest.mark.parametrize("name", ["directed", "mixed"])
def test_descriptor_rollout_is_bitwise_the_dense_input(gn, lib, batches, name):
    """rollout_trials from compact descriptors, one launch per step: step 0 is fused with the encoder and reads the seed
    bits of every row's CSR neighbours (directed: trial 0 seeds the in-hub and a sink, which many rows point at but whose
    own rows are short or empty). Bitwise the dense-input rollout."""
    graphs, inst, seeds, beta, gamma = case(name)
    batch = batches(name)
    dt = gn.rollout.dt_array(time_grid())
    trials = gn.rollout.TrialSet(seeds, beta, gamma, batch.sizes, DEV)
    with switches(gn, lib) as s:
        s.set(persistent=0)
        with torch.no_grad():
            compact = gn.rollout.rollout_trials(batch, trials, dt, dev_params()).cpu()
        dense = infer(gn, batch, x_of(name))
    assert torch.equal(compact, dense), (compact - dense).abs().max().item()
    assert (dense - oracle_probs(name)).abs().max().item() < 1e-5


@gpu
def test_r_state_modes_on_directed(gn, lib, batches):
    """Inference with the R plane (0) and from the conserved sum (1): both within 1e-5 of the oracle, 2e-6 of each other,
    and the decoded encoder state at t = 0 is the same."""
    want = oracle_probs("directed")
    out = {}
    with switches(gn, lib) as s:
        for mode in (0, 1):
            s.set(r_state=mode)
            out[mode] = infer(gn, batches("directed"), x_of("directed"))
            err = (out[mode] - want).abs().max().item()
            print("directed r_state %d: %.3e" % (mode, err))
            assert err < 1e-5, (mode, err)
    assert (out[0] - out[1]).abs().max().item() < 2e-6
    assert torch.equal(out[0][0], out[1][0])


@gpu
@pytest.mark.parametrize("k", [0, 4, 8])
def test_rhs_teacher_forced_on_directed(gn, batches, k):
    """One f(t, y) on the oracle's states: the neighbour sum runs over the stored entries of A, not of A^T."""
    x, p, coo = x_of("directed"), params(), coo_of("directed")
    _, traj = orc.forward(x, p, coo, time_grid(), return_traj=True)
    y = traj[k]
    beta, gamma = x[:, 3].contiguous(), x[:, 4].contiguous()
    W, b = p["odefunc.linear.weight"], p["odefunc.linear.bias"]
    want = torch.stack(orc.rhs(y[0], y[1], y[2], beta, gamma, W, b, coo))
    got = gn.rollout.odefunc_eval(y.to(DEV), beta.to(DEV), gamma.to(DEV), batches("directed"),
                                  [W.to(DEV), b.to(DEV)] + [b.to(DEV)] * 6).cpu()
    scale = want.abs().max().item()
    err = (got - want).abs().max().item()
    print("directed rhs k=%d: %.3e (scale %.3e)" % (k, err, scale))
    assert err <= 6e-6 * scale, (err, scale)
    assert got.sum(0).abs().max().item() <= 1e-6 * scale


@gpu
def test_edgeless_graph(gn, lib, batches):
    """No edges: A I' = 0 in every row, so dS = -beta * 0 * S' and the stored training trajectory's S plane is bitwise
    S_0 at every grid point; probabilities against the oracle."""
    batch, x = batches("edgeless"), x_of("edgeless")
    L = lib.lib()
    T = len(time_grid())
    dt = gn.rollout.dt_array(time_grid())
    ps = dev_params()
    pstruct = gn.rollout._params_struct(ps)
    xd = x.to(DEV)
    traj = torch.empty((T, 3, batch.M, H), dtype=torch.float32, device=DEV)
    probs = torch.empty((T, batch.M, 3), dtype=torch.float32, device=DEV)
    ws_bytes = int(L.gnode_rollout_workspace_bytes(batch.handle, 1))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=DEV)
    lib.check(L.gnode_rollout_forward(batch.handle, ctypes.c_void_p(xd.data_ptr()), xd.stride(0), ctypes.byref(pstruct),
                                      T, dt.ctypes.data_as(lib.c_float_p), ctypes.c_void_p(traj.data_ptr()),
                                      ctypes.c_void_p(probs.data_ptr()), ctypes.c_void_p(ws.data_ptr()), ws_bytes,
                                      ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)), "gnode_rollout_forward")
    torch.cuda.synchronize()
    S = traj[:, 0].cpu()
    for k in range(1, T):
        assert torch.equal(S[k], S[0]), k
    assert not torch.equal(traj[-1, 1].cpu(), traj[0, 1].cpu())          # I still recovers
    assert (probs.cpu() - oracle_probs("edgeless")).abs().max().item() < 1e-5
    assert (infer(gn, batch, x) - oracle_probs("edgeless")).abs().max().item() < 1e-5


# ---------------------------------------------------------------------------------------------------------- backward
@gpu
@pytest.mark.parametrize("cot", ["dense", "sparse"])
@pytest.mark.parametrize("mode", ["adjoint", "discrete"])
@pytest.mark.parametrize("name", ["directed", "nearly_symmetric", "mixed"])
def test_reverse_sweep_against_fp64_oracle(gn, lib, batches, name, mode, cot):
    """Small batches (the sweep is replayed from a CUDA graph): parameter and input gradients against the float64 oracle,
    per tensor and per column, with and without auxiliary storage, with both tile kernels, and with the model frozen
    (grads_out = NULL, bwd_vjp2_kernel<false>). Rows with an empty CSR row (sinks, one-node and edgeless instances) have
    A I' = 0: their dL/dbeta is exactly 0."""
    batch, x, c = batches(name), x_of(name), cotangent(name, cot)
    zero_rows = torch.from_numpy(out_degree_zero_rows(name))
    assert (len(zero_rows) > 0) == (name != "nearly_symmetric")
    with switches(gn, lib) as s:
        for aux in (True, False):
            for bk in (2, 1):
                s.set(aux=aux, bwd_kernel=bk)
                gx, gp = cuda_grads(gn, batch, x, mode, cot, c, frozen=False)
                what = "%s %s %s aux=%d bwd=%d" % (name, mode, cot, aux, bk)
                assert float(gx[:, 5:].abs().max()) == 0.0
                assert_grads_close(what, gp, gx[:, :5], name, mode, cot)
                if len(zero_rows):
                    assert float(gx[zero_rows, 3].abs().max()) == 0.0, what
                    assert float(gx[zero_rows, 4].abs().max()) > 0.0, what
                gx_frozen, _ = cuda_grads(gn, batch, x, mode, cot, c, frozen=True)
                if bk == 2:                  # bwd_vjp2_kernel<false> computes the same input gradients bit for bit
                    assert torch.equal(gx_frozen, gx), what
                assert_grads_close(what + " frozen", None, gx_frozen[:, :5], name, mode, cot)


@gpu
@pytest.mark.parametrize("mode", ["adjoint", "discrete"])
def test_reverse_sweep_large_batch(gn, lib, mode):
    """More than 4 tiles per SM (no graph replay; the forward runs one launch per step): the directed graph repeated, a
    cotangent only on one probe trial. Parameter gradients and the probe's dL/dx against the oracle on the probe trial
    alone; every other trial's dL/dx is exactly 0."""
    n = _graphs.directed().shape[0]
    rows_needed = 4 * torch.cuda.get_device_properties(0).multi_processor_count * _graphs.TILE
    B = rows_needed // n + 1
    probe = B - 2
    graph = gn.DeviceGraph(_graphs.directed())
    batch = gn.DeviceBatch([graph] * B)
    assert (batch.M + _graphs.TILE - 1) // _graphs.TILE > rows_needed // _graphs.TILE
    xp = x_of("directed-probe")
    others = [torch.from_numpy(_graphs.dense_x([n], *_graphs.trial_inputs([n], 100 + b), H)) for b in range(B)]
    x = torch.cat([xp if b == probe else others[b] for b in range(B)])
    cp = cotangent("directed-probe", "dense")
    c = torch.zeros(cp.size(0), B * n, 3)
    c[:, probe * n:(probe + 1) * n] = cp
    with switches(gn, lib) as s:
        s.set(persistent=0)
        gx, gp = cuda_grads(gn, batch, x, mode, "dense", c, frozen=False)
        gx_frozen, _ = cuda_grads(gn, batch, x, mode, "dense", c, frozen=True)
    mine = slice(probe * n, (probe + 1) * n)
    assert_grads_close("large %s (B=%d)" % (mode, B), gp, gx[mine, :5], "directed-probe", mode, "dense")
    assert torch.equal(gx_frozen, gx)
    rest = torch.ones(B * n, dtype=torch.bool)
    rest[mine] = False
    assert float(gx[rest].abs().max()) == 0.0


@gpu
@pytest.mark.parametrize("mode", ["adjoint", "discrete"])
def test_descriptor_gradients_per_instance(gn, batches, mode):
    """rollout_trials with beta, gamma requiring grad on the mixed batch: gnode_trials_grad's per-instance sums against
    the oracle's per-instance sums of dL/dx[:, 3] and [:, 4]. Every one-node and edgeless instance has dL/dbeta exactly
    0 (A I' = 0 in all its rows) and a nonzero dL/dgamma."""
    graphs, inst, seeds, beta0, gamma0 = case("mixed")
    batch = batches("mixed")
    c = cotangent("mixed", "dense")
    beta = torch.tensor(beta0, dtype=torch.float32, device=DEV, requires_grad=True)
    gamma = torch.tensor(gamma0, dtype=torch.float32, device=DEV, requires_grad=True)
    trials = gn.rollout.TrialSet(seeds, beta, gamma, batch.sizes, DEV)
    probs = gn.rollout.rollout_trials(batch, trials, gn.rollout.dt_array(time_grid()), dev_params(), grad_mode=mode,
                                      beta=beta, gamma=gamma)
    (probs * c.to(DEV)).sum().backward()
    got = torch.stack((beta.grad, gamma.grad)).cpu().double()
    rows = _graphs.instance_rows(batch.sizes)
    per_inst = lambda g: torch.stack([torch.stack([g[r:r + n, col].double().sum() for r, n in zip(rows, batch.sizes)])
                                      for col in (3, 4)])
    want = per_inst(oracle("mixed", mode, "dense", "float64")[1])
    ref = per_inst(oracle("mixed", mode, "dense", "float32")[1])
    for i, what in enumerate(("beta", "gamma")):
        scale = want[i].abs().max().item()
        err = (got[i] - want[i]).abs().max().item() / scale
        e_ref = (ref[i] - want[i]).abs().max().item() / scale
        print("mixed %s per-instance dL/d%s: %.3e (fp32 oracle %.3e)" % (mode, what, err, e_ref))
        assert err <= max(1e-3, 2.0 * e_ref), (what, err, e_ref)
    no_edges = [i for i, g in enumerate(inst) if graphs[g].nnz == 0]
    assert len(no_edges) == 201
    assert float(got[0, no_edges].abs().max()) == 0.0
    assert float(got[1, no_edges].abs().min()) > 0.0


# ---------------------------------------------------------------------------------------------------------- Monte Carlo
MC_SIMS, MC_T, MC_BETA, MC_GAMMA = 2000, 8, 0.3, 0.2


def zscores(p1, p2, sims1, sims2):
    return (p1 - p2) / np.sqrt(p1 * (1 - p1) / sims1 + p2 * (1 - p2) / sims2 + 1e-12)


@functools.lru_cache(maxsize=None)
def mc_numpy(transpose, seed):
    A = _graphs.directed()
    A = A.T.tocsr() if transpose else A
    return orc.mc_sir_counts(A, [_graphs.OUT_HUB], MC_BETA, MC_GAMMA, MC_SIMS, MC_T, np.random.RandomState(seed)) / MC_SIMS


@gpu
def test_mc_kernel_spreads_along_edge_direction():
    """harness.monte_carlo_sir on an nx.DiGraph seeded at the out-hub (whose out- and in-neighbourhoods differ by ~2000
    nodes) against the numpy process on the same directed adjacency: infection travels from a row to its columns."""
    import networkx as nx
    from gn_ode_sir_b200 import harness
    G = nx.from_scipy_sparse_array(_graphs.directed(), create_using=nx.DiGraph)
    assert list(G.nodes()) == list(range(G.number_of_nodes()))
    S, I, R = harness.monte_carlo_sir(G, [_graphs.OUT_HUB], MC_BETA, MC_GAMMA, sims=MC_SIMS, T=MC_T, seed=3)
    ours = np.stack((S[0], I[0], R[0])) / MC_SIMS
    zz = zscores(ours[:, 1:], mc_numpy(False, 4)[:, 1:], MC_SIMS, MC_SIMS)
    print("directed MC: max|z| %.2f mean z^2 %.2f" % (np.abs(zz).max(), (zz ** 2).mean()))
    assert np.abs(zz).max() < 5.5 and (zz ** 2).mean() < 1.5


# ---------------------------------------------------------------------------------------------------------- sensitivity
@pytest.mark.parametrize("mode", ["adjoint", "discrete"])
@pytest.mark.parametrize("name,cot", [("directed", "dense"), ("directed", "sparse"), ("mixed", "dense"),
                                      ("mixed", "sparse"), ("directed-probe", "dense")])
def test_backward_tests_detect_a_gather_over_a(name, mode, cot):
    """CPU only. If the reverse sweep gathered A gAI instead of A^T gAI, its gradients would be the oracle's with the
    backward of the neighbour sum taken over A: that differs from the float64 gradients by at least 100x the GPU tests'
    bar on linear.weight, and on the beta and gamma columns of the directed graph. In the mixed batch the columns' scale
    is set by instances the transpose does not touch (karate, the edgeless instance), so their margin is smaller:
    measured 30x .. 90x, asserted 20x."""
    want_p, want_x = oracle(name, mode, cot, "float64")
    wrong_p, wrong_x = oracle(name, mode, cot, "float64", gather_over_a=True)
    pb, cb = bars(name, mode, cot)
    e_p = rel_err_params(wrong_p, want_p)
    e_x = rel_err_columns(wrong_x, want_x)
    print("%s %s %s, gather over A: linear.weight %.3e (bar %.1e), beta %.3e (bar %.1e), gamma %.3e (bar %.1e)"
          % (name, mode, cot, e_p["odefunc.linear.weight"], pb["odefunc.linear.weight"], e_x[3], cb[3], e_x[4], cb[4]))
    assert e_p["odefunc.linear.weight"] >= 100 * pb["odefunc.linear.weight"]
    margin = 20 if name == "mixed" else 100
    assert e_x[3] >= margin * cb[3] and e_x[4] >= margin * cb[4]


def test_mc_test_detects_infection_against_edge_direction():
    """CPU only. The numpy process spreading along A^T (a kernel that pulls infection from a node's own CSR row) lies far
    outside the z-score bar of the directed Monte-Carlo test."""
    zz = zscores(mc_numpy(True, 5)[:, 1:], mc_numpy(False, 4)[:, 1:], MC_SIMS, MC_SIMS)
    print("MC along A^T vs along A: max|z| %.1f" % np.abs(zz).max())
    assert np.abs(zz).max() > 100 * 5.5
