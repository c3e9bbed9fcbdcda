"""GPU checks of the edge gradients dL/dw (gnode_rollout_backward_edges, bwd_edge_kernel; rollout(..., edge_weight=)).
Against the float64 oracle (tests/_edge_grad_oracle.py) per instance, with the bar of the input-gradient tests:
err / scale <= max(1e-3, 2 x the fp32 oracle's own error), in both grad modes, with and without auxiliary storage, with
dense and sparse (L1 at the unit-time grid points) cotangents, with the model trainable and frozen. Then the exact zeros,
the row-sum identity sum_c dL/dw_rc = beta[r] dL/dbeta[r], the promise that asking for edges changes nothing else, the
graph replay, the drop-in blocks' keyword, and the argument checks."""
import functools

import numpy as np
import pytest
import torch

import _graphs
from _edge_grad_oracle import (DELTAT, MAXTIME, PARAM_SEED, directed_case, edge_coo, edge_offsets, oracle_pair,
                               per_instance_rel_err, row_sums)
from _util import Golden
from oracle import gnode_oracle as orc

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
H = 64
PARAM_ORDER = ("odefunc.linear.weight", "odefunc.linear.bias", "linearS1.weight", "linearS1.bias",
               "linear3.weight", "linear3.bias", "linearS2.weight", "linearS2.bias")


@pytest.fixture(scope="module")
def gn():
    import gn_ode_sir_b200 as g
    g.build_library()
    return g


@pytest.fixture
def aux_storage(gn):
    prev = gn.rollout.AUX_STORAGE
    yield
    gn.rollout.AUX_STORAGE = prev


@functools.lru_cache(maxsize=None)
def case(name):
    """(adjs, inst, x [M, 3+H], params, maxTime, deltaT)"""
    if name == "karate8":                          # 8 trials of karate: the sweep is captured and replayed
        g = Golden("sim_karate_b8")
        return [g.adjs[0]], [0] * 8, g.x, g.params, g.maxTime, g.deltaT
    if name == "dolphins7":                        # M = 7 * 62 = 434 rows: not a tile multiple
        A = Golden("sim_dolphins_b4").adjs[0]
        x = torch.cat([orc.synthetic_trial(A.shape[0], 64, 300 + b) for b in range(7)])
        return [A], [0] * 7, x, orc.default_params(64, seed=77), 6, 0.25
    if name == "directed":                         # out-hub (degree 2000) and in-hub: A and A^T differ
        adjs, inst, x = directed_case()
        return adjs, inst, x, orc.default_params(64, seed=PARAM_SEED), MAXTIME, DELTAT
    if name == "mixed":                            # 205 instances: one-node, edgeless, directed 127/128/129, karate
        graphs, inst = _graphs.mixed()
        sizes = [graphs[i].shape[0] for i in inst]
        seeds, beta, gamma = _graphs.trial_inputs(sizes, seed=5)
        return graphs, inst, torch.from_numpy(_graphs.dense_x(sizes, seeds, beta, gamma)), \
            orc.default_params(64, seed=PARAM_SEED), MAXTIME, DELTAT
    if name == "ngraphs2":                         # two different graphs in one batch
        adjs = Golden("ng_mixed_b5").adjs[:2]
        x = torch.cat([orc.synthetic_trial(adjs[g].shape[0], 64, 500 + g, graph_marker=g + 1) for g in range(2)])
        return adjs, [0, 1], x, orc.default_params(64, seed=8), 5, 0.5
    if name == "wikivote6":                        # hub rows of degree ~1000, 6-point grid
        g = Golden("sim_wikivote_b2")
        return [g.adjs[0]], [0, 0], g.x, g.params, 3, 0.5
    if name == "T1":                               # no Euler step
        g = Golden("sim_karate_b8")
        return [g.adjs[0]], [0] * 8, g.x, g.params, 0.5, 0.5
    raise KeyError(name)


_batches = {}


def batch_of(gn, name):
    if name not in _batches:
        adjs, inst = case(name)[:2]
        dg = [gn.DeviceGraph(A) for A in adjs]
        _batches[name] = (dg, gn.DeviceBatch([dg[i] for i in inst]))
    return _batches[name][1]


def cotangent(name, cot):
    adjs, inst, x, params, maxTime, deltaT = case(name)
    M = x.size(0)
    if cot == "dense":
        return torch.randn(len(orc.time_grid(maxTime, deltaT)), M, 3, generator=torch.Generator().manual_seed(9))
    steps = orc.unit_time_rows(maxTime, deltaT)
    return torch.rand(M, len(steps), 3, generator=torch.Generator().manual_seed(2), dtype=torch.float64)


@functools.lru_cache(maxsize=None)
def oracle(name, mode, cot):
    adjs, inst, x, params, maxTime, deltaT = case(name)
    t = orc.time_grid(maxTime, deltaT)
    c = cotangent(name, cot)
    if cot == "dense":
        return oracle_pair(x, params, edge_coo(adjs, inst), t, c, mode)
    weight = lambda probs: orc.train_loss(probs, c, maxTime, deltaT)
    return oracle_pair(x, params, edge_coo(adjs, inst), t, None, mode, weight=weight)


def run(gn, name, mode, cot, frozen=False, edges=True, want_x=False, batch=None, x=None, c=None):
    """One forward + backward through rollout(): (probs, dL/dw or None, dL/dx or None, {key: dL/dparam} or None)."""
    adjs, inst, x0, params, maxTime, deltaT = case(name)
    batch = batch if batch is not None else batch_of(gn, name)
    x = (x if x is not None else x0).to(DEV).clone().requires_grad_(want_x)
    c = c if c is not None else cotangent(name, cot)
    ps = [params[k].to(DEV).clone().requires_grad_(not frozen) for k in PARAM_ORDER]
    ew = torch.ones(batch.nnz, device=DEV, requires_grad=True) if edges else None
    dt = gn.rollout.dt_array(orc.time_grid(maxTime, deltaT))
    if cot == "dense":
        probs = gn.rollout.rollout(x, batch, dt, ps, grad_mode=mode, edge_weight=ew)
        loss = (probs * c.to(DEV)).sum()
    else:
        probs = gn.rollout.rollout(x, batch, dt, ps, grad_mode=mode, out_steps=orc.unit_time_rows(maxTime, deltaT),
                                   edge_weight=ew)
        loss = gn.rollout.l1_subsampled(probs, c.to(DEV), skip=1)
    loss.backward()
    torch.cuda.synchronize()
    return (probs.detach().clone(), ew.grad.clone() if edges else None, x.grad.clone() if want_x else None,
            None if frozen else {k: p.grad.clone() for k, p in zip(PARAM_ORDER, ps)})


def assert_per_instance(what, got, name, mode, cot):
    adjs, inst = case(name)[:2]
    off = edge_offsets(adjs, inst)
    (w64, _), (w32, _) = oracle(name, mode, cot)
    assert got.shape == (int(off[-1]),)
    got = got.cpu()
    err = per_instance_rel_err(got, w64, off)
    ref = per_instance_rel_err(w32, w64, off)
    for i, (e0, e1) in enumerate(zip(off[:-1], off[1:])):
        if np.isnan(err[i]):                       # empty slice, or an instance whose true gradient is exactly 0
            if e1 > e0:
                assert float(got[e0:e1].abs().max()) == 0.0, (what, i)
            continue
        bar = max(1e-3, 2.0 * ref[i])
        assert err[i] <= bar, (what, i, err[i], bar)
    ok = ~np.isnan(err)
    print("%s: worst instance %.3e of its bar (%d instances with edges)"
          % (what, np.max(err[ok] / np.maximum(1e-3, 2.0 * ref[ok])), ok.sum()))


NAMES = ["karate8", "dolphins7", "directed", "mixed", "ngraphs2", "wikivote6"]


@pytest.mark.parametrize("cot", ["dense", "sparse"])
@pytest.mark.parametrize("mode", ["adjoint", "discrete"])
@pytest.mark.parametrize("name", NAMES)
def test_edge_grads_against_fp64_oracle(gn, aux_storage, name, mode, cot):
    """Per instance against the float64 oracle, with and without auxiliary storage; frozen (grads_out = NULL) gives the
    same bits as trainable."""
    for aux in (True, False):
        gn.rollout.AUX_STORAGE = aux
        _, ge, _, _ = run(gn, name, mode, cot)
        assert_per_instance("%s %s %s aux=%d" % (name, mode, cot, aux), ge, name, mode, cot)
        _, ge_frozen, _, _ = run(gn, name, mode, cot, frozen=True)
        assert torch.equal(ge_frozen, ge)


def test_edge_grads_are_zero_without_an_euler_step(gn):
    _, ge, _, _ = run(gn, "T1", "adjoint", "dense", want_x=True)
    assert ge.numel() == batch_of(gn, "T1").nnz > 0 and float(ge.abs().max()) == 0.0


def test_edgeless_and_one_node_instances_have_empty_slices(gn):
    graphs, inst = case("mixed")[:2]
    batch = batch_of(gn, "mixed")
    assert np.array_equal(batch.edge_offsets, edge_offsets(graphs, inst)) and batch.nnz == batch.edge_offsets[-1]
    empty = [i for i, g in enumerate(inst) if graphs[g].nnz == 0]
    assert len(empty) == 201 and all(batch.edge_offsets[i] == batch.edge_offsets[i + 1] for i in empty)
    rows, cols = batch.graphs[inst.index(1)].edges()
    assert np.array_equal(np.stack((rows, cols)), edge_coo(graphs, [1]))


@pytest.mark.parametrize("mode", ["adjoint", "discrete"])
def test_large_batch_probe_trial(gn, mode):
    """More than 4 tiles per SM (no graph replay): the directed graph repeated, a cotangent only on one probe trial. The
    probe's edge gradients against the oracle of the probe alone; every other trial's edge gradient is exactly 0."""
    adjs, inst, x2, params, maxTime, deltaT = case("directed")
    n = adjs[0].shape[0]
    rows_needed = 4 * torch.cuda.get_device_properties(0).multi_processor_count * _graphs.TILE
    B = rows_needed // n + 1
    probe = B - 2
    graph = gn.DeviceGraph(adjs[0])
    batch = gn.DeviceBatch([graph] * B)
    xp = x2[:n]
    others = [torch.from_numpy(_graphs.dense_x([n], *_graphs.trial_inputs([n], 100 + b), H)) for b in range(B)]
    x = torch.cat([xp if b == probe else others[b] for b in range(B)])
    cp = torch.randn(len(orc.time_grid(maxTime, deltaT)), n, 3, generator=torch.Generator().manual_seed(9))
    c = torch.zeros(cp.size(0), B * n, 3)
    c[:, probe * n:(probe + 1) * n] = cp
    _, ge, _, _ = run(gn, "directed", mode, "dense", batch=batch, x=x, c=c)
    nnz = adjs[0].nnz
    mine = ge[probe * nnz:(probe + 1) * nnz].cpu()
    (w64, _), (w32, _) = oracle_pair(xp, params, edge_coo(adjs, [0]), orc.time_grid(maxTime, deltaT), cp, mode)
    scale = w64.abs().max().item()
    err, ref = (mine.double() - w64).abs().max().item() / scale, (w32.double() - w64).abs().max().item() / scale
    print("large %s (B=%d): %.3e (bar %.3e)" % (mode, B, err, max(1e-3, 2 * ref)))
    assert err <= max(1e-3, 2.0 * ref)
    rest = torch.ones(B * nnz, dtype=torch.bool)
    rest[probe * nnz:(probe + 1) * nnz] = False
    assert float(ge[rest].abs().max()) == 0.0


@pytest.mark.parametrize("mode", ["adjoint", "discrete"])
@pytest.mark.parametrize("name", ["directed", "wikivote6"])
def test_row_sums_equal_beta_times_dbeta(gn, name, mode):
    """sum over row r's entries of dL/dw = beta[r] dL/dbeta[r], both sides from one sweep. The identity is exact, but
    the two sides round differently in fp32: dL/dbeta reads the forward's A I' (one fp32 sum over the row), the edge
    gradients one dot product per entry. On the directed graph's out-hub row (2000 entries) the fp32 oracle itself
    misses 1e-5 of scale (3.8e-5 adjoint, 5.3e-5 discrete), so the bar is max(1e-5, 2 x the fp32 oracle's own error),
    as for every other comparison in the suite."""
    adjs, inst, x = case(name)[:3]
    coo = edge_coo(adjs, inst)
    _, ge, gx, _ = run(gn, name, mode, "dense", want_x=True)
    want = x[:, 3].double() * gx[:, 3].cpu().double()
    got = row_sums(ge.cpu(), coo, x.size(0))
    scale = want.abs().max().item()
    err = (got - want).abs().max().item() / scale
    _, (w32, x32) = oracle(name, mode, "dense")
    ref = (row_sums(w32, coo, x.size(0)) - x[:, 3].double() * x32[:, 3].double()).abs().max().item() / scale
    bar = max(1e-5, 2.0 * ref)
    print("%s %s: row sums vs beta dL/dbeta %.3e of scale (fp32 oracle %.3e, bar %.3e)" % (name, mode, err, ref, bar))
    assert scale > 0 and err <= bar


@pytest.mark.parametrize("mode", ["adjoint", "discrete"])
def test_asking_for_edges_changes_nothing_else(gn, aux_storage, mode):
    """Probabilities, parameter gradients and dL/dx are bitwise those of a sweep without edges; edge gradients are
    bitwise reproducible; a sweep without edges launches no more kernels than before, one with edges one per step more."""
    from gn_ode_sir_b200 import _lib
    L = _lib.lib()
    for aux in (True, False):
        gn.rollout.AUX_STORAGE = aux
        for name in ("directed", "mixed"):
            T = len(orc.time_grid(*case(name)[4:]))
            n0 = L.gnode_launch_count()
            p0, _, gx0, gp0 = run(gn, name, mode, "dense", edges=False, want_x=True)
            n1 = L.gnode_launch_count()
            p1, ge1, gx1, gp1 = run(gn, name, mode, "dense", want_x=True)
            n2 = L.gnode_launch_count()
            _, ge2, _, _ = run(gn, name, mode, "dense", want_x=True)
            assert torch.equal(p0, p1) and torch.equal(gx0, gx1) and torch.equal(ge1, ge2)
            assert all(torch.equal(gp0[k], gp1[k]) for k in gp0)
            # one edge launch per reverse step with an adjoint (dense cotangent: all T - 1 of them)
            assert (n2 - n1) - (n1 - n0) == T - 1, (name, aux, n1 - n0, n2 - n1)


def test_graph_replay_follows_the_edge_request(gn):
    """karate, B = 1 (a captured and replayed reverse sweep): requests with and without edges, with and without
    parameters, alternated over the same buffers, each reproduce what a fresh block computes."""
    g = Golden("sim_karate_b1")

    def block():
        of = gn.ode_sim.ODEfunc(g.adjs[0], 0.2, 0.1, g.H, DEV)
        blk = gn.ode_sim.ODEBlock(g.maxTime, g.deltaT, g.adjs[0].shape[0], [0, 1], g.H, of, DEV)
        blk.load_state_dict(g.params, strict=True)
        return blk.to(DEV)

    w = g.weight().to(DEV)
    x = g.x_as_model_input().to(DEV)
    nnz = gn.DeviceGraph(g.adjs[0]).nnz

    def request(blk, kind):
        blk.zero_grad(set_to_none=True)
        blk.requires_grad_(kind != "frozen-edges")
        ew = torch.ones(1, nnz, device=DEV, requires_grad=True) if kind != "params" else None
        S, I, R = blk(x, edge_weight=ew)
        (torch.cat((S, I, R), -1) * w).sum().backward()
        torch.cuda.synchronize()
        pg = {k: p.grad.clone() for k, p in blk.named_parameters() if p.grad is not None}
        return (ew.grad.clone() if ew is not None else None), pg

    kinds = ("edges", "params", "frozen-edges")
    fresh = {k: request(block(), k) for k in kinds}
    blk = block()
    for kind in ("edges", "params", "edges", "frozen-edges", "params", "frozen-edges", "edges"):
        ge, pg = request(blk, kind)
        want_ge, want_pg = fresh[kind]
        assert (ge is None) == (want_ge is None), kind
        if ge is not None:
            assert ge.shape == (1, nnz) and torch.equal(ge, want_ge), kind
        assert sorted(pg) == sorted(want_pg) and all(torch.equal(pg[k], want_pg[k]) for k in pg), kind
    assert torch.equal(fresh["edges"][0], fresh["frozen-edges"][0]) and float(fresh["edges"][0].abs().max()) > 0


def test_dropin_blocks_take_edge_weight(gn):
    """sim: forward and forward_trials with a [B, nnz] edge_weight; ngraphs: forward with instances. Each equals the
    rollout() edge gradient of the same batch bit for bit."""
    adjs, inst, x, params, maxTime, deltaT = case("dolphins7")
    N, B = adjs[0].shape[0], len(inst)
    c = cotangent("dolphins7", "dense").to(DEV)
    of = gn.ode_sim.ODEfunc(adjs[0], 0.2, 0.1, H, DEV)
    blk = gn.ode_sim.ODEBlock(maxTime, deltaT, N, [0, 1], H, of, DEV)
    blk.load_state_dict(params, strict=True)
    blk.to(DEV)
    nnz = of.device_graph().nnz
    ew = torch.ones(B, nnz, device=DEV, requires_grad=True)
    S, I, R = blk(x.view(B, N, -1).to(DEV), edge_weight=ew)
    (torch.cat((S, I, R), -1) * c).sum().backward()
    _, want, _, _ = run(gn, "dolphins7", "adjoint", "dense", batch=of.batch_for(B))
    assert ew.grad.shape == (B, nnz) and torch.equal(ew.grad.reshape(-1), want)
    # the same trials from compact descriptors
    xs = x.view(B, N, -1)
    seeds = [np.flatnonzero(xs[b, :, 1].numpy() == 1.0) for b in range(B)]
    ew2 = torch.ones(B, nnz, device=DEV, requires_grad=True)
    S, I, R = blk.forward_trials(seeds, xs[:, 0, 3].tolist(), xs[:, 0, 4].tolist(), edge_weight=ew2)
    (torch.cat((S, I, R), -1) * c).sum().backward()
    scale = want.abs().max().item()
    assert (ew2.grad.reshape(-1) - want).abs().max().item() <= 1e-6 * scale
    # ngraphs
    adjs, inst, x, params = case("ngraphs2")[:4]
    of = gn.ode_ngraphs.ODEfunc(adjs, H, DEV)
    blk = gn.ode_ngraphs.ODEBlock(5, 0.5, H, of, DEV)
    blk.load_state_dict(params, strict=True)
    blk.to(DEV)
    batch = of.batch_from_instances(inst)
    ew = torch.ones(batch.nnz, device=DEV, requires_grad=True)
    S, I, R = blk(x.to(DEV), instances=inst, edge_weight=ew)
    (torch.cat((S, I, R), -1) * cotangent("ngraphs2", "dense").to(DEV)).sum().backward()
    _, want, _, _ = run(gn, "ngraphs2", "adjoint", "dense", batch=batch)
    assert torch.equal(ew.grad, want)


def test_edge_weight_is_checked(gn):
    adjs, inst, x, params, maxTime, deltaT = case("karate8")
    batch = batch_of(gn, "karate8")
    dt = gn.rollout.dt_array(orc.time_grid(maxTime, deltaT))
    ps = [params[k].to(DEV) for k in PARAM_ORDER]
    xd = x.to(DEV)
    ew = torch.ones(batch.nnz, device=DEV)
    ew[5] = 0.0
    with pytest.raises(ValueError, match="build a graph without it"):
        gn.rollout.rollout(xd, batch, dt, ps, edge_weight=ew)
    with pytest.raises(ValueError, match="one value per stored adjacency entry"):
        gn.rollout.rollout(xd, batch, dt, ps, edge_weight=torch.ones(batch.nnz + 1, device=DEV))
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        gn.rollout.rollout(xd, batch, dt, ps, edge_weight=torch.ones(batch.nnz))
