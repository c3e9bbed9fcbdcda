"""CUDA-event timing of the reverse sweep (gnode_rollout_backward_input) in three modes, on the configurations of
tools/train_timing.py: parameters only (what training runs), parameters + dL/dx, and dL/dx only with the model frozen
(no weight-gradient phase). One forward (trajectory + auxiliary storage) per configuration; every mode replays the same
sweep over the same stored state and cotangent.

--parent-lib PATH: a build of an earlier commit (same C ABI up to gnode_rollout_backward_aux). Its parameters-only sweep
is timed in the same process, alternated round by round with this build's, over the same buffers, and its gradient
vector is compared with this build's bit for bit.

    python tools/input_grad_timing.py [--parent-lib build/parent/libgnode_b200.so] [--rounds 7] [--iters 5]
"""
import argparse
import ctypes
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import gn_ode_sir_b200 as gn
from gn_ode_sir_b200 import _lib, synth
from gn_ode_sir_b200.rollout import _params_struct, _ptr

CONFIGS = (("karate-size", 34, 2, 1), ("fb-social-size", 1893, 7, 8), ("fb-social-size", 1893, 7, 64),
           ("epinions-size", 75879, 5, 4), ("epinions-size", 75879, 5, 8))


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                      # noqa: BLE001 -- the query is informational
        q = "power limit not readable (%s)" % e
    return "%s | power.limit, clocks.max.sm: %s" % (name, q)


class ParentLib:
    """The subset of an earlier build's C ABI the parameters-only sweep needs, with its own graph / batch handles."""

    def __init__(self, path):
        L = ctypes.CDLL(path)
        sig = _lib.SIGNATURES
        for name in ("gnode_graph_create", "gnode_batch_create", "gnode_backward_workspace_bytes",
                     "gnode_rollout_backward_aux", "gnode_last_error"):
            fn = getattr(L, name)
            fn.restype, fn.argtypes = sig[name]
        self.L = L

    def batch(self, A, B):
        indptr = np.ascontiguousarray(A.indptr, dtype=np.int32)
        indices = np.ascontiguousarray(A.indices, dtype=np.int32)
        g = ctypes.c_void_p()
        self._check(self.L.gnode_graph_create(A.shape[0], int(indptr[-1]), indptr.ctypes.data_as(_lib.c_int32_p),
                                              indices.ctypes.data_as(_lib.c_int32_p), ctypes.byref(g)))
        b = ctypes.c_void_p()
        self._check(self.L.gnode_batch_create((ctypes.c_void_p * B)(*([g.value] * B)), B, ctypes.byref(b)))
        return b

    def _check(self, rc):
        if rc != 0:
            raise RuntimeError("parent library: %s" % self.L.gnode_last_error().decode())


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
    for name, n, m, B in CONFIGS:
        A = synth.barabasi_albert_csr(n, m, 0)
        N = A.shape[0]
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
        grads = {k: torch.empty(_lib.GRAD_COUNT, dtype=torch.float32, device=dev) for k in ("new", "parent")}
        gx = torch.zeros_like(x)

        def sweep(mode):
            if mode == "parent":
                parent._check(parent.L.gnode_rollout_backward_aux(
                    pb, _ptr(x), x.stride(0), ctypes.byref(pstruct), T, dtp, _ptr(traj), auxp, _ptr(gp), None, 0,
                    _lib.GRAD_ADJOINT, _ptr(grads["parent"]), _ptr(pws), pws.numel(), stream))
                return
            g = _ptr(grads["new"]) if mode in ("params", "params+x") else None
            gxp = _ptr(gx) if mode in ("params+x", "x-only") else None
            _lib.check(L.gnode_rollout_backward_input(batch.handle, _ptr(x), x.stride(0), ctypes.byref(pstruct), T,
                                                      dtp, _ptr(traj), auxp, _ptr(gp), None, 0, _lib.GRAD_ADJOINT, g,
                                                      gxp, gx.stride(0), _ptr(bws), bws.numel(), stream),
                       "gnode_rollout_backward_input")

        modes = ["params", "params+x", "x-only"]
        if parent is not None:
            pb = parent.batch(A, B)
            pws = torch.empty(int(parent.L.gnode_backward_workspace_bytes(pb)), dtype=torch.uint8, device=dev)
            modes = ["parent"] + modes
        for mode in modes:                              # warm-up (module load, graph capture of small batches)
            for _ in range(2):
                sweep(mode)
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        times = {k: [] for k in modes}
        for r in range(args.rounds):
            order = modes if r % 2 == 0 else modes[::-1]  # alternate the order round by round
            for mode in order:
                ev[0].record()
                for _ in range(args.iters):
                    sweep(mode)
                ev[1].record()
                torch.cuda.synchronize()
                times[mode].append(ev[0].elapsed_time(ev[1]) / args.iters)
        line = "%-15s N=%-6d B=%-3d M=%-7d" % (name, N, B, M)
        for mode in modes:
            t = np.asarray(times[mode])
            line += " | %s %8.3f ms [%.3f .. %.3f]" % (mode, np.median(t), t.min(), t.max())
        print(line)
        if parent is not None:
            sweep("parent")
            sweep("params")
            torch.cuda.synchronize()
            same = torch.equal(grads["parent"], grads["new"])
            print("    parameter gradients, parent vs this build: %s" % ("bitwise equal" if same else "DIFFER"))
        sys.stdout.flush()


if __name__ == "__main__":
    main()
