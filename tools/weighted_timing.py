"""CUDA-event timing of weighted contact graphs at the epinions size (607k rows: 8 trials of a 75,879-node
Barabasi-Albert graph, T = 40, adjoint mode, dense cotangent, auxiliary storage): the inference rollout, the training
forward and the reverse sweep, each for the binary graph, contact_weight = ones and random weights in [0, 2]. The three
weightings alternate round by round in one process; every number is the median over rounds of the mean of `iters`
back-to-back calls, with the [min .. max] over rounds. Also checks that ones give the binary probabilities and
gradients bit for bit at this size.

    python tools/weighted_timing.py [--rounds 7] [--iters 3]
"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import gn_ode_sir_b200 as gn
from gn_ode_sir_b200 import _lib, synth

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from input_grad_timing import card                                          # noqa: E402

N, M_EDGES, B = 75879, 5, 8                     # epinions-size stand-in, as tools/input_grad_timing.py


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--iters", type=int, default=3, help="calls per timed window")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the rollout runs on the GPU only"
    dev = torch.device("cuda:0")
    print("card:", card())
    print("times: median over %d rounds of the mean of %d back-to-back calls (CUDA events); [min .. max] over rounds"
          % (args.rounds, args.iters))
    H = _lib.GNODE_H
    A = synth.barabasi_albert_csr(N, M_EDGES, 0)
    torch.manual_seed(0)
    of = gn.ode_sim.ODEfunc(A, 0.2, 0.1, H, dev)
    blk = gn.ode_sim.ODEBlock(20, 0.5, N, [0, 1], H, of, dev).to(dev)
    ps = [p.detach().contiguous() for p in blk._params()]
    pg = [p.clone().requires_grad_(True) for p in ps]
    batch = of.batch_for(B)
    M, dt = batch.M, blk._dt
    T = len(dt) + 1
    x = torch.stack([synth.synthetic_trial(N, H, b) for b in range(B)]).to(dev).view(M, -1).contiguous()
    gp = torch.randn(T, M, 3, device=dev)
    weights = {"binary": None, "ones": torch.ones(batch.nnz, device=dev),
               "random": 2.0 * torch.rand(batch.nnz, generator=torch.Generator().manual_seed(1)).to(dev)}
    print("M=%d rows, nnz=%d stored entries, T=%d, persistent=%d" % (M, batch.nnz, T, _lib.lib().gnode_get_persistent()))
    ro = gn.rollout

    def inference(cw):
        with torch.no_grad():
            return ro.rollout(x, batch, dt, ps, contact_weight=cw)

    def training(cw, ev=None):
        for p in pg:
            p.grad = None
        if ev:
            ev[0].record()
        probs = ro.rollout(x, batch, dt, pg, contact_weight=cw)
        if ev:
            ev[1].record()
        probs.backward(gp)
        if ev:
            ev[2].record()
        return probs.detach(), [p.grad for p in pg]

    # bitwise: ones == binary at this size
    pb, gb = training(None)
    po, go = training(weights["ones"])
    same = torch.equal(pb, po) and all(torch.equal(a, b) for a, b in zip(gb, go))
    same = same and torch.equal(inference(None), inference(weights["ones"]))
    print("contact_weight = ones vs binary, probabilities (inference, training) and parameter gradients: %s"
          % ("bitwise equal" if same else "DIFFER"))
    del pb, gb, po, go
    kinds = list(weights)
    for k in kinds:                                    # warm-up
        inference(weights[k])
        training(weights[k])
    torch.cuda.synchronize()
    times = {(k, p): [] for k in kinds for p in ("inference", "train forward", "sweep")}
    for r in range(args.rounds):
        for k in (kinds if r % 2 == 0 else kinds[::-1]):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.iters):
                inference(weights[k])
            e1.record()
            torch.cuda.synchronize()
            times[(k, "inference")].append(e0.elapsed_time(e1) / args.iters)
            fw, sw = 0.0, 0.0
            for _ in range(args.iters):
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
                training(weights[k], ev)
                torch.cuda.synchronize()
                fw += ev[0].elapsed_time(ev[1])
                sw += ev[1].elapsed_time(ev[2])
            times[(k, "train forward")].append(fw / args.iters)
            times[(k, "sweep")].append(sw / args.iters)
    for phase in ("inference", "train forward", "sweep"):
        base = np.median(times[("binary", phase)])
        print("%s:" % phase)
        for k in kinds:
            t = np.asarray(times[(k, phase)])
            print("    %-7s %9.3f ms [%.3f .. %.3f]  %+.1f %% vs binary" % (k, np.median(t), t.min(), t.max(),
                                                                          100 * (np.median(t) / base - 1)))


if __name__ == "__main__":
    main()
