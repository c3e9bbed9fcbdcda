"""CUDA-event timing of the reverse sweep with edge gradients (gnode_rollout_backward_edges) at the epinions size
(607k rows: 8 trials of a 75,879-node Barabasi-Albert graph, T = 40, adjoint mode, dense cotangent, auxiliary storage),
in three modes: parameters only (what training runs), parameters + dL/dw, and dL/dw only with the model frozen (no
weight-gradient phase). One forward; every mode replays the same sweep over the same stored state and cotangent.

--parent-lib PATH: a build of an earlier commit (same C ABI up to gnode_rollout_backward_aux). Its parameters-only sweep
is timed in the same process, alternated round by round with this build's, over the same buffers, and its gradient
vector is compared with this build's bit for bit.

    python tools/edge_grad_timing.py [--parent-lib build/parent/libgnode_b200.so] [--rounds 7] [--iters 5]
"""
import argparse
import ctypes
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import gn_ode_sir_b200 as gn
from gn_ode_sir_b200 import _lib, synth
from gn_ode_sir_b200.rollout import _params_struct, _ptr

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from input_grad_timing import ParentLib, card                              # noqa: E402

N, M_EDGES, B = 75879, 5, 8                     # epinions-size stand-in, as tools/input_grad_timing.py


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--iters", type=int, default=5, help="sweeps per timed window")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the reverse sweep runs on the GPU only"
    dev = torch.device("cuda:0")
    L = _lib.lib()
    parent = ParentLib(args.parent_lib) if args.parent_lib else None
    print("card:", card())
    print("library:", os.environ.get("GNODE_B200_LIB", gn.LIB_PATH), "| parent:", args.parent_lib)
    print("times: median over %d rounds of the mean of %d back-to-back sweeps (CUDA events); [min .. max] over rounds"
          % (args.rounds, args.iters))
    H = _lib.GNODE_H
    A = synth.barabasi_albert_csr(N, M_EDGES, 0)
    torch.manual_seed(0)
    of = gn.ode_sim.ODEfunc(A, 0.2, 0.1, H, dev)
    blk = gn.ode_sim.ODEBlock(20, 0.5, N, [0, 1], H, of, dev).to(dev)
    ps = [p.detach().contiguous() for p in blk._params()]
    pstruct = _params_struct(ps)
    batch = of.batch_for(B)
    M, dt = batch.M, blk._dt
    T = len(dt) + 1
    dtp = dt.ctypes.data_as(_lib.c_float_p)
    x = torch.stack([synth.synthetic_trial(N, H, b) for b in range(B)]).to(dev).view(M, -1).contiguous()
    traj = torch.empty((T, 3, M, H), dtype=torch.float32, device=dev)
    aux = torch.empty(int(L.gnode_rollout_aux_bytes(batch.handle, T)) // 4, dtype=torch.float32, device=dev)
    probs = torch.empty((T, M, 3), dtype=torch.float32, device=dev)
    ws = torch.empty(int(L.gnode_rollout_workspace_bytes(batch.handle, 1)), dtype=torch.uint8, device=dev)
    filled = ctypes.c_int32(0)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(L.gnode_rollout_forward_aux(batch.handle, _ptr(x), x.stride(0), ctypes.byref(pstruct), T, dtp, None,
                                           T, _ptr(traj), _ptr(aux), ctypes.byref(filled), _ptr(probs), _ptr(ws),
                                           ws.numel(), stream), "gnode_rollout_forward_aux")
    auxp = _ptr(aux) if filled.value == 1 else None
    del ws
    gp = torch.randn(T, M, 3, device=dev)
    bws = torch.empty(int(L.gnode_backward_workspace_bytes(batch.handle)), dtype=torch.uint8, device=dev)
    grads = {k: torch.empty(_lib.GRAD_COUNT, dtype=torch.float32, device=dev) for k in ("new", "parent", "with-edges")}
    ge = {k: torch.empty(batch.nnz, dtype=torch.float32, device=dev) for k in ("params+edges", "edges-only")}
    print("M=%d rows, nnz=%d stored entries, T=%d, auxiliary storage %s" % (M, batch.nnz, T, "on" if auxp else "off"))

    def sweep(mode):
        if mode == "parent":
            parent._check(parent.L.gnode_rollout_backward_aux(
                pb, _ptr(x), x.stride(0), ctypes.byref(pstruct), T, dtp, _ptr(traj), auxp, _ptr(gp), None, 0,
                _lib.GRAD_ADJOINT, _ptr(grads["parent"]), _ptr(pws), pws.numel(), stream))
            return
        g = {"params": _ptr(grads["new"]), "params+edges": _ptr(grads["with-edges"])}.get(mode)
        e = _ptr(ge[mode]) if mode in ge else None
        _lib.check(L.gnode_rollout_backward_edges(batch.handle, _ptr(x), x.stride(0), ctypes.byref(pstruct), T, dtp,
                                                  _ptr(traj), auxp, _ptr(gp), None, 0, _lib.GRAD_ADJOINT, g, None, 0,
                                                  e, _ptr(bws), bws.numel(), stream), "gnode_rollout_backward_edges")

    modes = ["params", "params+edges", "edges-only"]
    if parent is not None:
        pb = parent.batch(A, B)
        pws = torch.empty(int(parent.L.gnode_backward_workspace_bytes(pb)), dtype=torch.uint8, device=dev)
        modes = ["parent"] + modes
    for mode in modes:                                  # warm-up
        for _ in range(2):
            sweep(mode)
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    times = {k: [] for k in modes}
    for r in range(args.rounds):
        order = modes if r % 2 == 0 else modes[::-1]      # alternate the order round by round
        for mode in order:
            ev[0].record()
            for _ in range(args.iters):
                sweep(mode)
            ev[1].record()
            torch.cuda.synchronize()
            times[mode].append(ev[0].elapsed_time(ev[1]) / args.iters)
    line = "epinions-size N=%d B=%d M=%d" % (N, B, M)
    for mode in modes:
        t = np.asarray(times[mode])
        line += "\n    %-13s %8.3f ms [%.3f .. %.3f]" % (mode, np.median(t), t.min(), t.max())
    print(line)
    for mode in modes:
        sweep(mode)
    torch.cuda.synchronize()
    if parent is not None:
        print("parameter gradients, parent vs this build's parameters-only sweep: %s"
              % ("bitwise equal" if torch.equal(grads["parent"], grads["new"]) else "DIFFER"))
    print("parameter gradients with and without edges: %s"
          % ("bitwise equal" if torch.equal(grads["new"], grads["with-edges"]) else "DIFFER"))
    print("edge gradients, parameters + edges vs edges only: %s"
          % ("bitwise equal" if torch.equal(ge["params+edges"], ge["edges-only"]) else "DIFFER"))
    print("edge gradients: max |dL/dw| %.3e, nonzero %d of %d"
          % (ge["edges-only"].abs().max().item(), int((ge["edges-only"] != 0).sum()), batch.nnz))


if __name__ == "__main__":
    main()
