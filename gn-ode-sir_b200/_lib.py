"""ctypes binding of the C ABI declared in include/gnode_b200.h.

The product path has no fallback: if libgnode_b200.so is missing or a call fails,
a RuntimeError is raised (never a silent CPU / eager path).
"""
import ctypes
import os

from ._build import LIB_PATH

c_void_p, c_int, c_int32, c_int64, c_size_t = (ctypes.c_void_p, ctypes.c_int, ctypes.c_int32,
                                               ctypes.c_int64, ctypes.c_size_t)
c_float_p = ctypes.POINTER(ctypes.c_float)
c_int32_p = ctypes.POINTER(ctypes.c_int32)

GNODE_H = 64
GNODE_TRIAL_LDX = 8            # row stride of the compact x written by gnode_rollout_forward_trials
GRAD_ADJOINT, GRAD_DISCRETE = 0, 1
GRAD_LAYOUT = (("odefunc.linear.weight", (GNODE_H, GNODE_H)), ("odefunc.linear.bias", (GNODE_H,)),
               ("linearS1.weight", (GNODE_H, 1)), ("linearS1.bias", (GNODE_H,)),
               ("linear3.weight", (4, GNODE_H)), ("linear3.bias", (4,)),
               ("linearS2.weight", (1, 4)), ("linearS2.bias", (1,)))
GRAD_COUNT = sum(s[0] * (s[1] if len(s) > 1 else 1) for _, s in GRAD_LAYOUT)   # 4553


class GnodeParams(ctypes.Structure):
    _fields_ = [(n, c_void_p) for n in ("lin_w", "lin_b", "s1_w", "s1_b", "l3_w", "l3_b", "s2_w", "s2_b")]


# symbol -> (restype, argtypes); tests/test_cabi.py checks this table against include/gnode_b200.h
SIGNATURES = {
    "gnode_last_error": (ctypes.c_char_p, []),
    "gnode_version": (c_int, []),
    "gnode_launch_count": (c_int64, []),
    "gnode_set_variant": (c_int, [c_int]),
    "gnode_get_variant": (c_int, []),
    "gnode_set_step_kernel": (c_int, [c_int]),
    "gnode_get_step_kernel": (c_int, []),
    "gnode_set_r_state": (c_int, [c_int]),
    "gnode_get_r_state": (c_int, []),
    "gnode_set_persistent": (c_int, [c_int]),
    "gnode_get_persistent": (c_int, []),
    "gnode_set_hub_relay": (c_int, [c_int]),
    "gnode_get_hub_relay": (c_int, []),
    "gnode_set_bwd_kernel": (c_int, [c_int]),
    "gnode_get_bwd_kernel": (c_int, []),
    "gnode_debug_phase_cycles": (c_int, [ctypes.POINTER(ctypes.c_longlong)]),
    "gnode_graph_create": (c_int, [c_int32, c_int64, c_int32_p, c_int32_p, ctypes.POINTER(c_void_p)]),
    "gnode_graph_destroy": (c_int, [c_void_p]),
    "gnode_graph_info": (c_int, [c_void_p, c_int32_p, ctypes.POINTER(c_int64), c_int32_p, c_int32_p]),
    "gnode_batch_create": (c_int, [ctypes.POINTER(c_void_p), c_int32, ctypes.POINTER(c_void_p)]),
    "gnode_batch_destroy": (c_int, [c_void_p]),
    "gnode_batch_rows": (c_int64, [c_void_p]),
    "gnode_aggregate": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "gnode_odefunc_eval": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, ctypes.POINTER(GnodeParams),
                                   c_void_p, c_void_p, c_void_p]),
    "gnode_rollout_workspace_bytes": (c_size_t, [c_void_p, c_int]),
    "gnode_rollout_forward": (c_int, [c_void_p, c_void_p, c_int64, ctypes.POINTER(GnodeParams), c_int32,
                                      c_float_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "gnode_rollout_forward_sel": (c_int, [c_void_p, c_void_p, c_int64, ctypes.POINTER(GnodeParams), c_int32,
                                          c_float_p, c_int32_p, c_int32, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "gnode_expand_trials": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "gnode_rollout_trials_workspace_bytes": (c_size_t, [c_void_p, c_int]),
    "gnode_rollout_forward_trials": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                             ctypes.POINTER(GnodeParams), c_int32, c_float_p, c_int32_p, c_int32,
                                             c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "gnode_backward_workspace_bytes": (c_size_t, [c_void_p]),
    "gnode_rollout_backward": (c_int, [c_void_p, c_void_p, c_int64, ctypes.POINTER(GnodeParams), c_int32,
                                       c_float_p, c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_size_t,
                                       c_void_p]),
    "gnode_rollout_backward_sel": (c_int, [c_void_p, c_void_p, c_int64, ctypes.POINTER(GnodeParams), c_int32,
                                           c_float_p, c_void_p, c_void_p, c_int32_p, c_int32, c_int32, c_void_p,
                                           c_void_p, c_size_t, c_void_p]),
    "gnode_rollout_aux_bytes": (c_size_t, [c_void_p, c_int32]),
    "gnode_rollout_forward_aux": (c_int, [c_void_p, c_void_p, c_int64, ctypes.POINTER(GnodeParams), c_int32,
                                          c_float_p, c_int32_p, c_int32, c_void_p, c_void_p, c_int32_p, c_void_p,
                                          c_void_p, c_size_t, c_void_p]),
    "gnode_rollout_backward_aux": (c_int, [c_void_p, c_void_p, c_int64, ctypes.POINTER(GnodeParams), c_int32,
                                           c_float_p, c_void_p, c_void_p, c_void_p, c_int32_p, c_int32, c_int32,
                                           c_void_p, c_void_p, c_size_t, c_void_p]),
    "gnode_rollout_backward_input": (c_int, [c_void_p, c_void_p, c_int64, ctypes.POINTER(GnodeParams), c_int32,
                                             c_float_p, c_void_p, c_void_p, c_void_p, c_int32_p, c_int32, c_int32,
                                             c_void_p, c_void_p, c_int64, c_void_p, c_size_t, c_void_p]),
    "gnode_rollout_backward_edges": (c_int, [c_void_p, c_void_p, c_int64, ctypes.POINTER(GnodeParams), c_int32,
                                             c_float_p, c_void_p, c_void_p, c_void_p, c_int32_p, c_int32, c_int32,
                                             c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_size_t, c_void_p]),
    "gnode_rollout_forward_weighted": (c_int, [c_void_p, c_void_p, c_int64, ctypes.POINTER(GnodeParams), c_int32,
                                               c_float_p, c_int32_p, c_int32, c_void_p, c_void_p, c_int32_p, c_void_p,
                                               c_void_p, c_void_p, c_size_t, c_void_p]),
    "gnode_backward_weighted_workspace_bytes": (c_size_t, [c_void_p]),
    "gnode_rollout_backward_weighted": (c_int, [c_void_p, c_void_p, c_int64, ctypes.POINTER(GnodeParams), c_int32,
                                                c_float_p, c_void_p, c_void_p, c_void_p, c_int32_p, c_int32, c_int32,
                                                c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_size_t,
                                                c_void_p]),
    "gnode_trials_grad": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "gnode_mc_sir_workspace_bytes": (c_size_t, [c_void_p, c_int32]),
    "gnode_mc_sir": (c_int, [c_void_p, c_void_p, c_int32, ctypes.c_float, ctypes.c_float, c_int32, c_int32,
                             ctypes.c_uint64, c_void_p, c_void_p, c_size_t, c_void_p]),
    "gnode_l1_scratch_bytes": (c_size_t, []),
    "gnode_l1_loss_grad": (c_int, [c_void_p, c_void_p, c_int64, c_int32, c_int32, ctypes.c_float, c_void_p, c_void_p,
                                   c_void_p, c_void_p]),
}

_lib = None


def lib():
    """The loaded library; raises loudly when it has not been built."""
    global _lib
    if _lib is None:
        path = os.environ.get("GNODE_B200_LIB", LIB_PATH)      # another build of the same ABI (A/B measurements)
        if not os.path.exists(path):
            raise RuntimeError(
                "libgnode_b200.so is missing (%s). Build it with `python -c \"import __graft_entry__ as g; "
                "g.build()\"`. There is no CPU fallback for the GN-ODE rollout." % path)
        handle = ctypes.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)          # AttributeError if the symbol is not exported
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def check(rc, what):
    if rc != 0:
        msg = lib().gnode_last_error()
        raise RuntimeError("%s failed (code %d): %s" % (what, rc, msg.decode() if msg else "?"))
