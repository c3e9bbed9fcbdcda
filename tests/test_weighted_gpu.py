"""GPU checks of weighted contact graphs (gnode_rollout_forward_weighted / gnode_rollout_backward_weighted;
rollout(..., contact_weight=)). The neighbour sum AI[r] = sum over stored (r, c), ascending c, of fl(w_rc I'[c]):
  * ones are the binary rollout bit for bit (probabilities, trajectory, auxiliary planes, every gradient, dL/dw);
  * zeros are a graph built without those entries bit for bit;
  * random weights in [0, 2], asymmetric and different per trial, match the float64 oracle with the bars of the
    edge-gradient tests; the weighted row identity sum_c w_rc dL/dw_rc = beta[r] dL/dbeta[r] holds;
  * replayed reverse sweeps honour weights written in place; the drop-in blocks equal rollout(); arguments are checked;
    two identical runs are bitwise equal."""
import ctypes
import functools

import numpy as np
import pytest
import scipy.sparse as sp
import torch

import _graphs
from _edge_grad_oracle import edge_coo, edge_offsets, per_instance_rel_err, row_sums, weighted
from _util import Golden
from oracle import gnode_oracle as orc
from test_edge_grad_gpu import PARAM_ORDER, case, cotangent

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
H = 64


@pytest.fixture(scope="module")
def gn():
    import gn_ode_sir_b200 as g
    g.build_library()
    return g


@pytest.fixture
def settings(gn):
    """restores the process-wide switches a test changes"""
    from gn_ode_sir_b200 import _lib
    L = _lib.lib()
    prev = (gn.rollout.AUX_STORAGE, L.gnode_get_persistent(), L.gnode_get_hub_relay(), L.gnode_get_step_kernel())
    yield L
    gn.rollout.AUX_STORAGE = prev[0]
    L.gnode_set_persistent(prev[1])
    L.gnode_set_hub_relay(prev[2])
    L.gnode_set_step_kernel(prev[3])


_batches = {}


def batch_for(gn, adjs, inst, key):
    if key not in _batches:
        dg = [gn.DeviceGraph(A) for A in adjs]
        _batches[key] = (dg, gn.DeviceBatch([dg[i] for i in inst]))
    return _batches[key][1]


def random_weights(nnz, seed):
    return 2.0 * torch.rand(nnz, generator=torch.Generator().manual_seed(seed))


def run(gn, adjs, inst, x, params, maxTime, deltaT, mode="adjoint", cot="dense", c=None, key=None, cw=None, ew=None,
        frozen=False, want_x=True, want_w=True, batch=None):
    """forward + backward through rollout(): (probs, dL/dw or None, dL/dx or None, {param: grad} or None).
    cw: contact weights (float32 CPU tensor) or None; ew: pass unit edge_weight instead (binary rollout)."""
    batch = batch if batch is not None else batch_for(gn, adjs, inst, key)
    xd = x.to(DEV).clone().requires_grad_(want_x)
    ps = [params[k].to(DEV).clone().requires_grad_(not frozen) for k in PARAM_ORDER]
    cwd = cw.to(DEV).clone().requires_grad_(want_w) if cw is not None else None
    ewd = torch.ones(batch.nnz, device=DEV, requires_grad=True) if ew else None
    dt = gn.rollout.dt_array(orc.time_grid(maxTime, deltaT))
    if cot == "dense":
        probs = gn.rollout.rollout(xd, batch, dt, ps, grad_mode=mode, edge_weight=ewd, contact_weight=cwd)
        loss = (probs * c.to(DEV)).sum()
    else:
        probs = gn.rollout.rollout(xd, batch, dt, ps, grad_mode=mode, out_steps=orc.unit_time_rows(maxTime, deltaT),
                                   edge_weight=ewd, contact_weight=cwd)
        loss = gn.rollout.l1_subsampled(probs, c.to(DEV), skip=1)
    loss.backward()
    torch.cuda.synchronize()
    gw = cwd.grad.clone() if (cwd is not None and want_w) else (ewd.grad.clone() if ewd is not None else None)
    return (probs.detach().clone(), gw, xd.grad.clone() if want_x else None,
            None if frozen else {k: p.grad.clone() for k, p in zip(PARAM_ORDER, ps)})


def infer(gn, batch, x, params, maxTime, deltaT, cw=None):
    dt = gn.rollout.dt_array(orc.time_grid(maxTime, deltaT))
    with torch.no_grad():
        return gn.rollout.rollout(x.to(DEV), batch, dt, [params[k].to(DEV) for k in PARAM_ORDER],
                                  contact_weight=cw.to(DEV) if cw is not None else None).clone()


def assert_same(a, b, what):
    pa, gwa, gxa, gpa = a
    pb, gwb, gxb, gpb = b
    assert torch.equal(pa, pb), (what, "probs", (pa - pb).abs().max().item())
    assert torch.equal(gxa, gxb), (what, "grad_x", (gxa - gxb).abs().max().item())
    for k in gpa:
        assert torch.equal(gpa[k], gpb[k]), (what, k, (gpa[k] - gpb[k]).abs().max().item())
    if gwa is not None and gwb is not None:
        assert torch.equal(gwa, gwb), (what, "dL/dw", (gwa - gwb).abs().max().item())


# ------------------------------------------------------------------------------------------------ 1. ones == binary
def traj_and_aux(gn, batch, x, params, maxTime, deltaT, cw):
    """(probs, traj, aux, aux_filled) of one training forward through the C ABI (aux planes are not exposed above)"""
    from gn_ode_sir_b200 import _lib
    L = _lib.lib()
    ro = gn.rollout
    dt = ro.dt_array(orc.time_grid(maxTime, deltaT))
    T, M = len(dt) + 1, batch.M
    xd = x.to(DEV).contiguous()
    ps = [params[k].to(DEV).contiguous() for k in PARAM_ORDER]
    traj = torch.zeros((T, 3, M, H), device=DEV)
    aux = torch.zeros(int(L.gnode_rollout_aux_bytes(batch.handle, T)) // 4, device=DEV)
    probs = torch.zeros((T, M, 3), device=DEV)
    ws_bytes = int(L.gnode_rollout_workspace_bytes(batch.handle, 1))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=DEV)
    filled = ctypes.c_int32(0)
    pst = ro._params_struct(ps)
    args = (batch.handle, ro._ptr(xd), xd.stride(0), ctypes.byref(pst), T, dt.ctypes.data_as(_lib.c_float_p), None, 0,
            ro._ptr(traj), ro._ptr(aux), ctypes.byref(filled), ro._ptr(probs))
    if cw is None:
        _lib.check(L.gnode_rollout_forward_aux(*args, ro._ptr(ws), ws_bytes, ro._stream()), "forward_aux")
    else:
        cwd = cw.to(DEV).contiguous()
        _lib.check(L.gnode_rollout_forward_weighted(*args, ro._ptr(cwd), ro._ptr(ws), ws_bytes, ro._stream()),
                   "forward_weighted")
    torch.cuda.synchronize()
    return probs, traj, aux, filled.value


@pytest.mark.parametrize("name", ["karate8", "directed", "wikivote6", "mixed"])
def test_ones_are_the_binary_rollout_bitwise(gn, settings, name):
    """contact_weight = ones: probabilities (inference and training forward), trajectory, aux planes, parameter
    gradients, dL/dx and dL/dw (against edge_weight) are the binary path's bits; persistent on / off, relay on / off."""
    L = settings
    adjs, inst, x, params, maxTime, deltaT = case(name)
    batch = batch_for(gn, adjs, inst, name)
    ones = torch.ones(batch.nnz)
    c = cotangent(name, "dense")
    for persistent in (0, 1):
        for relay in (1, 0):
            L.gnode_set_persistent(persistent)
            L.gnode_set_hub_relay(relay)
            what = "%s persistent=%d relay=%d" % (name, persistent, relay)
            assert torch.equal(infer(gn, batch, x, params, maxTime, deltaT), infer(gn, batch, x, params, maxTime, deltaT, ones)), what
            p0, t0, a0, f0 = traj_and_aux(gn, batch, x, params, maxTime, deltaT, None)
            p1, t1, a1, f1 = traj_and_aux(gn, batch, x, params, maxTime, deltaT, ones)
            assert f0 == f1 == 1 and torch.equal(p0, p1) and torch.equal(t0, t1) and torch.equal(a0, a1), what
            for aux in (True, False):
                gn.rollout.AUX_STORAGE = aux
                for mode in ("adjoint", "discrete"):
                    b = run(gn, adjs, inst, x, params, maxTime, deltaT, mode, c=c, batch=batch, ew=True)
                    w = run(gn, adjs, inst, x, params, maxTime, deltaT, mode, c=c, batch=batch, cw=ones)
                    assert_same(b, w, "%s aux=%d %s" % (what, aux, mode))


# ------------------------------------------------------------------------------------------------ 2. zeros == removed
def without(A, mask):
    """A with the stored entries where mask (in edges() order) is True removed, and the same weights vector layout"""
    A = sp.csr_matrix(A)
    r = np.repeat(np.arange(A.shape[0]), np.diff(A.indptr))
    cidx = A.indices[:A.indptr[-1]]
    o = np.lexsort((cidx, r))
    keep = ~mask
    B = sp.csr_matrix((np.ones(int(keep.sum())), (r[o][keep], cidx[o][keep])), shape=A.shape)
    return B


def zero_case_check(gn, settings, adjs_w, inst, adjs_b, x, params, maxTime, deltaT, cw, key, relays=(1,)):
    L = settings
    bw = batch_for(gn, adjs_w, inst, key + "-w")
    bb = batch_for(gn, adjs_b, inst, key + "-b")
    c = torch.randn(len(orc.time_grid(maxTime, deltaT)), x.size(0), 3, generator=torch.Generator().manual_seed(9))
    for relay in relays:
        L.gnode_set_hub_relay(relay)
        assert torch.equal(infer(gn, bw, x, params, maxTime, deltaT, cw), infer(gn, bb, x, params, maxTime, deltaT)), (key, relay)
        for mode in ("adjoint", "discrete"):
            w = run(gn, None, None, x, params, maxTime, deltaT, mode, c=c, batch=bw, cw=cw, want_w=False)
            b = run(gn, None, None, x, params, maxTime, deltaT, mode, c=c, batch=bb)
            assert_same(w, b, "%s relay=%d %s" % (key, relay, mode))


def test_zero_hub_row_is_the_graph_without_it(gn, settings):
    """wiki-vote: every entry of one row of degree > 512 weighted 0 == the graph without that row's entries (the row is
    summed by the in-order relay, and by one half-warp with the relay off)."""
    adjs, inst, x, params, maxTime, deltaT = case("wikivote6")
    A = sp.csr_matrix(adjs[0])
    deg = np.diff(A.indptr)
    hub = int(np.flatnonzero(deg > 512)[0])
    rows = np.repeat(np.arange(A.shape[0]), deg)
    mask = rows == hub
    cw = torch.ones(len(inst) * A.nnz)
    cw[torch.from_numpy(np.tile(mask, len(inst)))] = 0.0
    zero_case_check(gn, settings, adjs, inst, [without(A, mask)], x, params, maxTime, deltaT, cw, "wikivote-hub",
                    relays=(1, 0))


def test_zero_entries_of_the_directed_graph(gn, settings):
    adjs, inst, x, params, maxTime, deltaT = case("directed")
    A = sp.csr_matrix(adjs[0])
    mask = np.random.default_rng(3).random(A.nnz) < 0.2
    cw = torch.from_numpy(np.tile(np.where(mask, 0.0, 1.0), len(inst)).astype(np.float32))
    zero_case_check(gn, settings, adjs, inst, [without(A, mask)], x, params, maxTime, deltaT, cw, "directed-zero")


def test_all_zero_weights_are_the_edgeless_graph(gn, settings):
    adjs, inst, x, params, maxTime, deltaT = case("dolphins7")
    A = sp.csr_matrix(adjs[0])
    zero_case_check(gn, settings, adjs, inst, [sp.csr_matrix(A.shape)], x, params, maxTime, deltaT,
                    torch.zeros(len(inst) * A.nnz), "all-zero")


# ------------------------------------------------------------------------------------------------ 3. random vs oracle
@functools.lru_cache(maxsize=None)
def weights_of(name):
    adjs, inst = case(name)[:2]
    return random_weights(int(edge_offsets(adjs, inst)[-1]), 1000 + len(name))


@functools.lru_cache(maxsize=None)
def oracle(name, mode, cot):
    """float64 and fp32 oracle results at the case's random weights: (probs, dL/dw, dL/dx, {param: grad}) each"""
    adjs, inst, x, params, maxTime, deltaT = case(name)
    t = orc.time_grid(maxTime, deltaT)
    coo = edge_coo(adjs, inst)
    c = cotangent(name, cot)
    w32 = weights_of(name)
    out = []
    for dt in (torch.float64, torch.float32):
        prev = torch.get_default_dtype()
        torch.set_default_dtype(dt)
        try:
            xx = x.to(dt).clone().requires_grad_(True)
            p = {k: v.to(dt).clone().requires_grad_(k in orc.GRAD_KEYS) for k, v in params.items()}
            w = w32.to(dt).clone().requires_grad_(True)
            from _edge_grad_oracle import _AdjointRolloutW
            S0, I0, R0, beta, gamma = orc.encode(xx, p["linearS1.weight"], p["linearS1.bias"])
            W, b = p["odefunc.linear.weight"], p["odefunc.linear.bias"]
            if mode == "adjoint":
                traj = _AdjointRolloutW.apply(torch.stack((S0, I0, R0)), beta, gamma, W, b, w, coo, t)
            else:
                with weighted(w):
                    traj = orc.euler_rollout(S0, I0, R0, beta, gamma, W, b, coo, t)
            probs = orc.decode(traj[:, 0], traj[:, 1], traj[:, 2], p["linear3.weight"], p["linear3.bias"],
                               p["linearS2.weight"], p["linearS2.bias"])
            loss = (probs * c.to(dt)).sum() if cot == "dense" else orc.train_loss(probs, c, maxTime, deltaT)
            loss.backward()
            grads = {k: p[k].grad.detach().clone() for k in PARAM_ORDER if p[k].grad is not None}
            out.append((probs.detach(), w.grad.detach().clone(), xx.grad[:, :5].detach().clone(), grads))
        finally:
            torch.set_default_dtype(prev)
    return out


def rel(a, b):
    b = b.double()
    s = b.abs().max().item()
    return (a.double().cpu() - b).abs().max().item() / s if s > 0 else float("nan")


def check_against_oracle(gn, name, mode, cot, got, frozen):
    adjs, inst = case(name)[:2]
    (p64, w64, x64, g64), (p32, w32, x32, g32) = oracle(name, mode, cot)
    probs, gw, gx, gp = got
    if cot == "dense":
        bar = max(1e-5, 2 * (p32.double() - p64).abs().max().item())
        assert (probs.cpu().double() - p64).abs().max().item() <= bar, (name, "probs")
    off = edge_offsets(adjs, inst)
    err, ref = per_instance_rel_err(gw.cpu(), w64, off), per_instance_rel_err(w32, w64, off)
    for i in range(len(err)):
        if not np.isnan(err[i]):
            assert err[i] <= max(1e-3, 2 * ref[i]), (name, mode, cot, "dL/dw instance", i, err[i], ref[i])
    for j in range(5):
        e, r = rel(gx[:, j], x64[:, j]), rel(x32[:, j], x64[:, j])
        if not np.isnan(e):
            assert e <= max(1e-3, 2 * r), (name, mode, cot, "dL/dx column", j, e, r)
    if not frozen:
        for k in g64:
            if k == "linearS2.bias":     # exactly 0 in exact arithmetic (the softmax ignores a shift of all three logits)
                continue
            e, r = rel(gp[k], g64[k]), rel(g32[k], g64[k])
            assert e <= max(1e-3, 2 * r), (name, mode, cot, k, e, r)


NAMES = ["karate8", "dolphins7", "directed", "mixed", "ngraphs2", "wikivote6"]


@pytest.mark.parametrize("cot", ["dense", "sparse"])
@pytest.mark.parametrize("mode", ["adjoint", "discrete"])
@pytest.mark.parametrize("name", NAMES)
def test_random_weights_against_fp64_oracle(gn, settings, name, mode, cot):
    """weights in [0, 2], asymmetric, different per trial; with and without aux storage, trainable and frozen"""
    adjs, inst, x, params, maxTime, deltaT = case(name)
    cw = weights_of(name)
    c = cotangent(name, cot)
    for aux in (True, False):
        gn.rollout.AUX_STORAGE = aux
        got = run(gn, adjs, inst, x, params, maxTime, deltaT, mode, cot, c=c, key=name, cw=cw)
        check_against_oracle(gn, name, mode, cot, got, False)
        frozen = run(gn, adjs, inst, x, params, maxTime, deltaT, mode, cot, c=c, key=name, cw=cw, frozen=True)
        assert torch.equal(frozen[1], got[1]) and torch.equal(frozen[2], got[2])


@pytest.mark.parametrize("mode", ["adjoint", "discrete"])
def test_large_batch_probe_trial(gn, mode):
    """more than 4 tiles per SM (no graph replay): the directed graph repeated with random weights per trial, a
    cotangent on one probe trial only, against the oracle of the probe trial alone"""
    adjs, inst, x2, params, maxTime, deltaT = case("directed")
    A = adjs[0]
    n = A.shape[0]
    B = 4 * torch.cuda.get_device_properties(0).multi_processor_count * _graphs.TILE // n + 1
    probe = B - 2
    g = gn.DeviceGraph(A)
    batch = gn.DeviceBatch([g] * B)
    xp = x2[:n]
    x = torch.cat([xp if b == probe else torch.from_numpy(_graphs.dense_x([n], *_graphs.trial_inputs([n], 100 + b), H))
                   for b in range(B)])
    cw = random_weights(B * A.nnz, 77)
    cp = torch.randn(len(orc.time_grid(maxTime, deltaT)), n, 3, generator=torch.Generator().manual_seed(9))
    c = torch.zeros(cp.size(0), B * n, 3)
    c[:, probe * n:(probe + 1) * n] = cp
    probs, gw, gx, gp = run(gn, None, None, x, params, maxTime, deltaT, mode, c=c, cw=cw, batch=batch)
    wp = cw[probe * A.nnz:(probe + 1) * A.nnz]
    coo = edge_coo(adjs, [0])
    t = orc.time_grid(maxTime, deltaT)
    out = []
    for dt in (torch.float64, torch.float32):
        prev = torch.get_default_dtype()
        torch.set_default_dtype(dt)
        try:
            from _edge_grad_oracle import loss_and_edge_grads
            out.append(loss_and_edge_grads(xp.to(dt), {k: v.to(dt) for k, v in params.items()}, coo, t, cp.to(dt),
                                           mode, w=wp.to(dt)))
        finally:
            torch.set_default_dtype(prev)
    (w64, x64), (w32, x32) = out
    mine = gw[probe * A.nnz:(probe + 1) * A.nnz]
    assert rel(mine, w64) <= max(1e-3, 2 * rel(w32, w64))
    for j in (0, 1, 3, 4):
        assert rel(gx[probe * n:(probe + 1) * n, j], x64[:, j]) <= max(1e-3, 2 * rel(x32[:, j], x64[:, j])), j
    with weighted(wp.double()):
        p64 = orc.forward(xp.double(), {k: v.double() for k, v in params.items()}, coo, t)
    assert (probs[:, probe * n:(probe + 1) * n].cpu().double() - p64).abs().max().item() <= 1e-5


# ------------------------------------------------------------------------------------------------ 4. row identity
@pytest.mark.parametrize("mode", ["adjoint", "discrete"])
@pytest.mark.parametrize("name", ["directed", "wikivote6"])
def test_weighted_row_sums_equal_beta_times_dbeta(gn, name, mode):
    """sum_c w_rc dL/dw_rc = beta[r] dL/dbeta[r] from one sweep, bar max(1e-5, 2 x the fp32 oracle's own error)"""
    adjs, inst, x, params, maxTime, deltaT = case(name)
    cw = weights_of(name)
    coo = edge_coo(adjs, inst)
    _, gw, gx, _ = run(gn, adjs, inst, x, params, maxTime, deltaT, mode, c=cotangent(name, "dense"), key=name, cw=cw)
    want = x[:, 3].double() * gx[:, 3].cpu().double()
    scale = want.abs().max().item()
    err = (row_sums(gw.cpu() * cw, coo, x.size(0)) - want).abs().max().item() / scale
    _, (_, w32, x32, _) = oracle(name, mode, "dense")
    ref = (row_sums(w32 * cw, coo, x.size(0)) - x[:, 3].double() * x32[:, 3].double()).abs().max().item() / scale
    print("%s %s: weighted row sums vs beta dL/dbeta %.3e of scale (fp32 oracle %.3e)" % (name, mode, err, ref))
    assert scale > 0 and err <= max(1e-5, 2 * ref)


# ------------------------------------------------------------------------------------------------ 5. graph replay
def test_graph_replay_honours_weights_written_in_place(gn):
    """karate, B = 1 (captured, replayed sweep): the same contact_weight tensor rewritten in place between calls, and
    weighted / unweighted calls alternated over one block, each equal to what a fresh block computes"""
    g = Golden("sim_karate_b1")

    def block():
        of = gn.ode_sim.ODEfunc(g.adjs[0], 0.2, 0.1, g.H, DEV)
        blk = gn.ode_sim.ODEBlock(g.maxTime, g.deltaT, g.adjs[0].shape[0], [0, 1], g.H, of, DEV)
        blk.load_state_dict(g.params, strict=True)
        return blk.to(DEV)

    cot = g.weight().to(DEV)
    x = g.x_as_model_input().to(DEV)
    nnz = gn.DeviceGraph(g.adjs[0]).nnz
    values = {"a": random_weights(nnz, 1), "b": random_weights(nnz, 2), "c": torch.zeros(nnz)}

    def request(blk, cw):
        blk.zero_grad(set_to_none=True)
        S, I, R = blk(x, contact_weight=cw)
        (torch.cat((S, I, R), -1) * cot).sum().backward()
        torch.cuda.synchronize()
        out = {k: p.grad.clone() for k, p in blk.named_parameters() if p.grad is not None}
        out["probs"] = torch.cat((S, I, R), -1).detach().clone()
        if cw is not None:
            out["w"] = cw.grad.clone()
        return out

    def fresh(kind):
        cw = values[kind].view(1, -1).to(DEV).requires_grad_(True) if kind else None
        return request(block(), cw)

    want = {k: fresh(k) for k in ("a", "b", "c", None)}
    blk = block()
    cw = torch.zeros(1, nnz, device=DEV, requires_grad=True)
    for kind in ("a", "b", None, "a", "c", None, "b"):
        if kind:
            with torch.no_grad():
                cw.copy_(values[kind].view(1, -1))
            cw.grad = None
        got = request(blk, cw if kind else None)
        assert sorted(got) == sorted(want[kind]) and all(torch.equal(got[k], want[kind][k]) for k in got), kind
    assert not torch.equal(want["a"]["probs"], want["b"]["probs"])


# ------------------------------------------------------------------------------------------------ 6. blocks, checks
def test_dropin_blocks_take_contact_weight(gn):
    adjs, inst, x, params, maxTime, deltaT = case("dolphins7")
    N, B = adjs[0].shape[0], len(inst)
    c = cotangent("dolphins7", "dense").to(DEV)
    of = gn.ode_sim.ODEfunc(adjs[0], 0.2, 0.1, H, DEV)
    blk = gn.ode_sim.ODEBlock(maxTime, deltaT, N, [0, 1], H, of, DEV)
    blk.load_state_dict(params, strict=True)
    blk.to(DEV)
    batch = of.batch_for(B)
    cw = weights_of("dolphins7")
    want = run(gn, adjs, inst, x, params, maxTime, deltaT, c=c.cpu(), cw=cw, batch=batch, want_x=False)
    cwb = cw.view(B, -1).to(DEV).requires_grad_(True)
    S, I, R = blk(x.view(B, N, -1).to(DEV), contact_weight=cwb)
    (torch.cat((S, I, R), -1) * c).sum().backward()
    assert cwb.grad.shape == (B, batch.nnz // B) and torch.equal(cwb.grad.reshape(-1), want[1])
    assert torch.equal(torch.cat((S, I, R), -1).detach(), want[0])
    with torch.no_grad():                          # inference carries no R plane: compared with rollout()'s inference
        pr = blk.rollout_probs(x.view(B, N, -1).to(DEV), contact_weight=cwb.detach())
    assert torch.equal(pr, infer(gn, batch, x, params, maxTime, deltaT, cw))
    # compact descriptors: expanded into x, then the same rollout (with and without gradients)
    xs = x.view(B, N, -1)
    seeds = [np.flatnonzero(xs[b, :, 1].numpy() == 1.0) for b in range(B)]
    with torch.no_grad():
        S, I, R = blk.forward_trials(seeds, xs[:, 0, 3].tolist(), xs[:, 0, 4].tolist(), contact_weight=cwb.detach())
    assert (torch.cat((S, I, R), -1) - want[0]).abs().max().item() <= 1e-6
    cw2 = cw.view(B, -1).to(DEV).requires_grad_(True)
    S, I, R = blk.forward_trials(seeds, xs[:, 0, 3].tolist(), xs[:, 0, 4].tolist(), contact_weight=cw2)
    (torch.cat((S, I, R), -1) * c).sum().backward()
    assert (cw2.grad.reshape(-1) - want[1]).abs().max().item() <= 1e-6 * want[1].abs().max().item()
    # ngraphs
    adjs, inst, x, params, maxTime, deltaT = case("ngraphs2")
    of = gn.ode_ngraphs.ODEfunc(adjs, H, DEV)
    blk = gn.ode_ngraphs.ODEBlock(maxTime, deltaT, H, of, DEV)
    blk.load_state_dict(params, strict=True)
    blk.to(DEV)
    batch = of.batch_from_instances(inst)
    cw = weights_of("ngraphs2")
    c = cotangent("ngraphs2", "dense")
    want = run(gn, adjs, inst, x, params, maxTime, deltaT, c=c, cw=cw, batch=batch, want_x=False)
    cwd = cw.to(DEV).requires_grad_(True)
    S, I, R = blk(x.to(DEV), instances=inst, contact_weight=cwd)
    (torch.cat((S, I, R), -1) * c.to(DEV)).sum().backward()
    assert torch.equal(cwd.grad, want[1]) and torch.equal(torch.cat((S, I, R), -1).detach(), want[0])
    sizes = [adjs[g].shape[0] for g in inst]
    xs = [x[sum(sizes[:i]):sum(sizes[:i + 1])] for i in range(len(inst))]
    seeds = [np.flatnonzero(xi[:, 1].numpy() == 1.0) for xi in xs]
    with torch.no_grad():
        S, I, R = blk.forward_trials(inst, seeds, [float(xi[0, 3]) for xi in xs], [float(xi[0, 4]) for xi in xs],
                                     contact_weight=cwd.detach())
    assert (torch.cat((S, I, R), -1) - want[0]).abs().max().item() <= 1e-6


def test_edge_values_follow_the_edge_order(gn):
    A = sp.random(50, 50, density=0.1, random_state=np.random.default_rng(5), format="csr")
    A.data = np.arange(1, A.nnz + 1, dtype=np.float64)
    # scramble the stored order inside the rows: the per-row column sort must carry the values along
    A2 = sp.csr_matrix((A.data[::-1].copy(), A.indices[::-1].copy(), A.indptr.copy()), shape=A.shape)
    for i in range(50):
        s, e = A.indptr[i], A.indptr[i + 1]
        A2.indices[s:e] = A.indices[s:e][::-1]
        A2.data[s:e] = A.data[s:e][::-1]
    g = gn.DeviceGraph(A2)
    r, cidx = g.edges()
    assert np.array_equal(g.edge_values(), np.asarray(A[r, cidx]).ravel().astype(np.float32))


def test_contact_weight_is_checked(gn, settings):
    L = settings
    adjs, inst, x, params, maxTime, deltaT = case("karate8")
    batch = batch_for(gn, adjs, inst, "karate8")
    dt = gn.rollout.dt_array(orc.time_grid(maxTime, deltaT))
    ps = [params[k].to(DEV) for k in PARAM_ORDER]
    xd = x.to(DEV)
    ro = gn.rollout
    with pytest.raises(ValueError, match="one value per stored adjacency entry"):
        ro.rollout(xd, batch, dt, ps, contact_weight=torch.ones(batch.nnz + 1, device=DEV))
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        ro.rollout(xd, batch, dt, ps, contact_weight=torch.ones(batch.nnz))
    with pytest.raises(RuntimeError, match="float32"):
        ro.rollout(xd, batch, dt, ps, contact_weight=torch.ones(batch.nnz, device=DEV, dtype=torch.float64))
    bad = torch.ones(batch.nnz, device=DEV)
    bad[3] = float("nan")
    with pytest.raises(ValueError, match="finite"):
        ro.rollout(xd, batch, dt, ps, contact_weight=bad)
    bad[3] = float("inf")
    with pytest.raises(ValueError, match="finite"):
        ro.rollout(xd, batch, dt, ps, contact_weight=bad)
    with pytest.raises(ValueError, match="not both"):
        ro.rollout(xd, batch, dt, ps, edge_weight=torch.ones(batch.nnz, device=DEV),
                   contact_weight=torch.ones(batch.nnz, device=DEV))
    for sk in (6, 7, 3, 0):
        L.gnode_set_step_kernel(sk)
        with pytest.raises(RuntimeError, match="step kernel 5"):
            ro.rollout(xd, batch, dt, ps, contact_weight=torch.ones(batch.nnz, device=DEV))
    L.gnode_set_step_kernel(5)
    # the unweighted rollout on the other step kernels is untouched
    assert torch.equal(infer(gn, batch, x, params, maxTime, deltaT), infer(gn, batch, x, params, maxTime, deltaT,
                                                                           torch.ones(batch.nnz)))


# ------------------------------------------------------------------------------------------------ 7. reproducible
def test_weighted_runs_are_bitwise_reproducible(gn):
    for name in ("wikivote6", "mixed"):
        adjs, inst, x, params, maxTime, deltaT = case(name)
        cw = weights_of(name)
        c = cotangent(name, "dense")
        a = run(gn, adjs, inst, x, params, maxTime, deltaT, c=c, key=name, cw=cw)
        b = run(gn, adjs, inst, x, params, maxTime, deltaT, c=c, key=name, cw=cw)
        assert_same(a, b, name)
