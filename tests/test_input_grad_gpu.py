"""GPU checks of the input gradients dL/dx[:, :5] = dL/d{S0, I0, R0, beta, gamma} of the reverse sweep
(gnode_rollout_backward_input) and of the descriptors' dL/dbeta[i], dL/dgamma[i] (gnode_trials_grad).
Against the float64 oracle, per column and scale-relative, with the bar of tests/test_backward_gpu.py:
max(1e-3, 2 x the fp32 oracle's own error against float64)."""
import numpy as np
import pytest
import torch

from _util import Golden
from _input_grad_oracle import loss_and_input_grads
from oracle import gnode_oracle as orc

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


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


def make_block(gn, variant, adjs, maxTime, deltaT, params, H, mode):
    if variant == "sim":
        of = gn.ode_sim.ODEfunc(adjs[0], 0.2, 0.1, H, DEV)
        blk = gn.ode_sim.ODEBlock(maxTime, deltaT, adjs[0].shape[0], [0, 1], H, of, DEV)
    else:
        of = gn.ode_ngraphs.ODEfunc(adjs, H, DEV)
        blk = gn.ode_ngraphs.ODEBlock(maxTime, deltaT, H, of, DEV)
    blk.load_state_dict(params, strict=True)
    blk.to(DEV)
    blk.grad_mode = mode
    return blk


def cuda_loss(gn, blk, x, w=None, labels=None, out_steps=None):
    probs = blk.rollout_probs(x, out_steps=out_steps)
    if labels is not None:
        return gn.rollout.l1_subsampled(probs, labels, skip=1)
    return (probs * w).sum()


def cuda_input_grad(gn, blk, x, frozen=False, **kw):
    """x.grad [M, cols] (and the parameters' .grad) after one backward through the drop-in block."""
    blk.zero_grad(set_to_none=True)
    blk.requires_grad_(not frozen)
    xin = x.to(DEV).clone().requires_grad_(True)
    cuda_loss(gn, blk, xin, **kw).backward()
    torch.cuda.synchronize()
    pg = {k: (p.grad.detach().clone() if p.grad is not None else None) for k, p in blk.named_parameters()}
    return xin.grad.detach().clone(), pg


def oracle_input_grads(x, params, coo, t, weight64, weight32, mode):
    _, _, g32 = loss_and_input_grads(x, params, coo, t, weight32, mode)
    torch.set_default_dtype(torch.float64)
    try:
        p64 = {k: v.double() for k, v in params.items()}
        _, _, g64 = loss_and_input_grads(x.double(), p64, coo, t, weight64, mode)
    finally:
        torch.set_default_dtype(torch.float32)
    return g64, g32


def assert_columns_close(got, want64, ref32, what):
    got = got.cpu().double()
    for c, name in enumerate(("S0", "I0", "R0", "beta", "gamma")):
        scale = want64[:, c].abs().max().item()
        if scale == 0.0:
            assert float(got[:, c].abs().max()) == 0.0, (what, name)
            continue
        err = (got[:, c] - want64[:, c]).abs().max().item() / scale
        e_ref = (ref32[:, c].double() - want64[:, c]).abs().max().item() / scale
        print("%s %s: ours %.3e, fp32 oracle %.3e" % (what, name, err, e_ref))
        assert err <= max(1e-3, 2.0 * e_ref), (what, name, err, e_ref)


def case_inputs(name):
    """(variant, adjs, inst_graph, x [M, 3+H], params, maxTime, deltaT, H)"""
    if name.startswith("dolphins"):                # M = 7 * 62 = 434 rows: not a tile multiple
        A = Golden("sim_dolphins_b4").adjs[0]
        x = torch.cat([orc.synthetic_trial(A.shape[0], 64, 300 + b) for b in range(7)])
        return "sim", [A], [0] * 7, x, orc.default_params(64, seed=77), 6, 0.25, 64
    if name == "ngraphs2":                         # two graphs, marker column x[row0, 5] = graph + 1
        adjs = Golden("ng_mixed_b5").adjs[:2]
        x = torch.cat([orc.synthetic_trial(adjs[g].shape[0], 64, 500 + g, graph_marker=g + 1) for g in range(2)])
        return "ngraphs", adjs, [0, 1], x, orc.default_params(64, seed=8), 5, 0.5, 64
    if name == "wikivote6":                        # hub rows (degree 1065) in the A^T gather, 6-point grid
        g = Golden("sim_wikivote_b2")
        return "sim", [g.adjs[0]], [0, 0], g.x, g.params, 3, 0.5, 64
    if name == "T1":                               # no Euler step: the beta and gamma columns are exactly 0
        g = Golden("sim_karate_b8")
        return "sim", [g.adjs[0]], [0] * 8, g.x, g.params, 0.5, 0.5, 64
    if name == "hidden16":                         # 16 channels, zero-padded to the 64-wide kernels
        A = Golden("sim_karate_b8").adjs[0]
        x = torch.cat([orc.synthetic_trial(A.shape[0], 16, 70 + b) for b in range(3)])
        return "sim", [A], [0] * 3, x, orc.default_params(16, seed=4), 5, 0.5, 16
    raise KeyError(name)


CASES = ["dolphins", "dolphins-noaux", "dolphins-l1", "dolphins-l1-noaux", "ngraphs2", "wikivote6", "T1", "hidden16"]


@pytest.mark.parametrize("mode", ["adjoint", "discrete"])
@pytest.mark.parametrize("name", CASES)
def test_input_grads_against_fp64_oracle(gn, aux_storage, name, mode):
    variant, adjs, inst, x, params, maxTime, deltaT, H = case_inputs(name)
    gn.rollout.AUX_STORAGE = not name.endswith("noaux")
    t = orc.time_grid(maxTime, deltaT)
    M = x.size(0)
    coo = orc.batch_coo(adjs, inst)
    blk = make_block(gn, variant, adjs, maxTime, deltaT, params, H, mode)
    if "-l1" in name:                              # sparse cotangent: unit-time grid points + fused L1
        steps = gn.rollout.unit_time_steps(maxTime, deltaT)
        y = torch.rand(M, len(steps), 3, generator=torch.Generator().manual_seed(2), dtype=torch.float64)
        got, _ = cuda_input_grad(gn, blk, x, labels=y.to(DEV), out_steps=steps)
        weight = lambda probs: orc.train_loss(probs, y, maxTime, deltaT)
        want, ref32 = oracle_input_grads(x, params, coo, t, weight, weight, mode)
    else:
        w = torch.randn(len(t), M, 3, generator=torch.Generator().manual_seed(9))
        got, _ = cuda_input_grad(gn, blk, x, w=w.to(DEV))
        want, ref32 = oracle_input_grads(x, params, coo, t, w.double(), w, mode)
    assert got.shape == x.shape
    assert float(got[:, 5:].abs().max()) == 0.0                 # graph marker and unused bg channels: no gradient
    if name == "T1":
        assert len(t) == 1 and float(got[:, 3:5].abs().max()) == 0.0
    assert_columns_close(got[:, :5], want, ref32, "%s %s" % (name, mode))


def karate(gn, mode="adjoint", B=8):
    g = Golden("sim_karate_b8" if B == 8 else "sim_karate_b1")
    blk = make_block(gn, "sim", g.adjs, g.maxTime, g.deltaT, g.params, g.H, mode)
    return g, blk, g.weight().to(DEV)


@pytest.mark.parametrize("mode", ["adjoint", "discrete"])
def test_unchanged_paths_are_bitwise(gn, mode):
    """Parameter gradients do not depend on whether x wants a gradient; grad_x of a frozen model (no weight-gradient
    phase) is grad_x computed together with the parameter gradients; two runs agree bit for bit."""
    g, blk, w = karate(gn, mode)
    x = g.x_as_model_input()
    blk.zero_grad(set_to_none=True)
    blk.requires_grad_(True)
    cuda_loss(gn, blk, x.to(DEV), w=w).backward()
    p_only = {k: p.grad.clone() for k, p in blk.named_parameters() if p.grad is not None}
    gx, p_with_x = cuda_input_grad(gn, blk, x, w=w)
    for k, v in p_only.items():
        assert torch.equal(v, p_with_x[k]), k
    gx_frozen, p_frozen = cuda_input_grad(gn, blk, x, frozen=True, w=w)
    assert all(v is None for v in p_frozen.values())
    assert torch.equal(gx_frozen, gx)
    gx2, _ = cuda_input_grad(gn, blk, x, w=w)
    assert torch.equal(gx2, gx)
    assert float(gx[..., 3:5].abs().max()) > 0.0


def test_graph_replay_follows_the_gradient_request(gn):
    """karate, B = 1 (a captured and replayed reverse sweep): calls with and without x.requires_grad_() and with a
    frozen model, alternated over the same buffers, each reproduce what a fresh block computes for that request."""
    kinds = ("x", "params", "frozen")

    def run(blk, g, w, kind):
        blk.zero_grad(set_to_none=True)
        blk.requires_grad_(kind != "frozen")
        xin = g.x_as_model_input().to(DEV).clone().requires_grad_(kind != "params")
        cuda_loss(gn, blk, xin, w=w).backward()
        torch.cuda.synchronize()
        pg = {k: p.grad.clone() for k, p in blk.named_parameters() if p.grad is not None}
        return (xin.grad.clone() if xin.grad is not None else None), pg

    fresh = {}
    for kind in kinds:
        g, blk, w = karate(gn, B=1)
        fresh[kind] = run(blk, g, w, kind)
    g, blk, w = karate(gn, B=1)
    for kind in ("x", "params", "x", "frozen", "params", "frozen", "x", "params"):
        gx, pg = run(blk, g, w, kind)
        want_gx, want_pg = fresh[kind]
        assert (gx is None) == (want_gx is None), kind
        if gx is not None:
            assert torch.equal(gx, want_gx), kind
        assert sorted(pg) == sorted(want_pg), kind
        for k in pg:
            assert torch.equal(pg[k], want_pg[k]), (kind, k)
    assert torch.equal(fresh["x"][0], fresh["frozen"][0])


def descriptor_case(gn, variant, mode):
    if variant == "sim":
        A = Golden("sim_dolphins_b4").adjs[0]
        adjs, inst = [A], [0, 0, 0]
    else:
        adjs = Golden("ng_mixed_b5").adjs[:2]
        inst = [1, 0, 1]
    sizes = [adjs[i].shape[0] for i in inst]
    seeds = [[0, 5], [3], [1, 2, 7]]
    beta0, gamma0 = [0.31, 0.17, 0.44], [0.12, 0.29, 0.21]
    params = orc.default_params(64, seed=13)
    blk = make_block(gn, variant, adjs, 5, 0.5, params, 64, mode)
    return adjs, inst, sizes, seeds, beta0, gamma0, params, blk


@pytest.mark.parametrize("mode", ["adjoint", "discrete"])
@pytest.mark.parametrize("variant", ["sim", "ngraphs"])
def test_descriptor_beta_gamma_gradients(gn, variant, mode):
    """forward_trials with beta, gamma as CUDA tensors requiring grad: beta.grad[i] is the float64 sum of the dense
    path's dL/dx[rows of i, 3] (gamma: column 4), and agrees with the oracle."""
    adjs, inst, sizes, seeds, beta0, gamma0, params, blk = descriptor_case(gn, variant, mode)
    M = sum(sizes)
    t = orc.time_grid(5, 0.5)
    w = torch.randn(len(t), M, 3, generator=torch.Generator().manual_seed(17))
    wd = w.to(DEV)
    beta = torch.tensor(beta0, device=DEV, requires_grad=True)
    gamma = torch.tensor(gamma0, device=DEV, requires_grad=True)
    blk.requires_grad_(False)
    if variant == "sim":
        S, I, R = blk.forward_trials(seeds, beta, gamma)
    else:
        S, I, R = blk.forward_trials(inst, seeds, beta, gamma)
    (torch.cat((S, I, R), -1) * wd).sum().backward()
    assert beta.grad.shape == (3,) and gamma.grad.shape == (3,)
    # dense path: the same x through rollout() with x requiring grad
    x = torch.zeros(M, 3 + 64)
    row0 = np.concatenate([[0], np.cumsum(sizes)[:-1]])
    for i, (r, n) in enumerate(zip(row0, sizes)):
        x[r:r + n, 0] = 1.0
        x[r + np.asarray(seeds[i]), 0] = 0.0
        x[r + np.asarray(seeds[i]), 1] = 1.0
        x[r:r + n, 3], x[r:r + n, 4] = beta0[i], gamma0[i]
        if variant == "ngraphs":
            x[r, 5] = inst[i] + 1
    if variant == "sim":
        gx, _ = cuda_input_grad(gn, blk, x, frozen=True, w=wd)
    else:
        blk.zero_grad(set_to_none=True)
        xin = x.to(DEV).requires_grad_(True)
        (blk.rollout_probs(xin, instances=inst) * wd).sum().backward()
        gx = xin.grad
    gx = gx.cpu().double()
    for col, got in ((3, beta.grad), (4, gamma.grad)):
        want = torch.stack([gx[r:r + n, col].sum() for r, n in zip(row0, sizes)])
        err = (got.cpu().double() - want).abs().max().item() / want.abs().max().item()
        assert err < 1e-6, (col, err)
    # against the oracle: per-instance sums of its dL/dx columns 3, 4
    want64, ref32 = oracle_input_grads(x, params, orc.batch_coo(adjs, inst), t, w.double(), w, mode)
    for col, got in ((3, beta.grad), (4, gamma.grad)):
        w64 = torch.stack([want64[r:r + n, col].sum() for r, n in zip(row0, sizes)])
        r32 = torch.stack([ref32[r:r + n, col].double().sum() for r, n in zip(row0, sizes)])
        scale = w64.abs().max().item()
        err = (got.cpu().double() - w64).abs().max().item() / scale
        e_ref = (r32 - w64).abs().max().item() / scale
        assert err <= max(1e-3, 2.0 * e_ref), (col, err, e_ref)


def test_frozen_model_input_gradient(gn):
    """The motivating use: a frozen model, only x wants a gradient (calibration, seed sensitivity, attribution)."""
    g, blk, w = karate(gn)
    blk.requires_grad_(False)
    x = g.x_as_model_input().to(DEV).clone().requires_grad_()
    S, I, R = blk(x)
    loss = (torch.cat((S, I, R), -1) * w).sum()
    loss.backward()
    assert x.grad is not None and x.grad.shape == x.shape
    assert float(x.grad[..., :5].abs().max()) > 0.0
    assert all(p.grad is None for p in blk.parameters())
