"""Shared helpers for the test-suite (golden fixture loading, oracle inputs)."""
import contextlib
import glob
import os

import numpy as np
import scipy.sparse
import torch

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLDEN_CASES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))
# On the larger graphs the reference's own fp32 run is not reproducible to 1e-5 (hidden states grow to ~1e3, SURVEY H1:
# its fp32-vs-fp64 difference is 4e-5 (ng_train5) .. 2e-3 (wiki-vote), and its wiki-vote fp32 GRADIENT differs from the
# fp64 one by ~100 %): those cases are judged against the float64 run, err(ours) <= max(bar, 2 * err(reference fp32)).
LARGE_CASES = [c for c in GOLDEN_CASES if any(k in c for k in ("fbsocial", "openflights", "wikivote", "train5"))]
STRICT_CASES = [c for c in GOLDEN_CASES if c not in LARGE_CASES]
# The fixtures were written with 8 intra-op threads. On CPU, torch splits elementwise ops (sigmoid) and GEMMs into
# per-thread ranges, and where a range ends decides which elements take the vectorised path and which the scalar tail:
# the fp32 results' last bits follow the thread count, so bit-exact comparisons with the fixtures run with 8 threads.
GOLDEN_THREADS = 8


@contextlib.contextmanager
def golden_threads():
    prev = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    try:
        yield
    finally:
        torch.set_num_threads(prev)


class Golden:
    """One fixture written by tests/golden/make_golden.py (outputs of the reference's classes)."""

    def __init__(self, name):
        z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
        self.name = name
        self.variant = str(z["variant"])
        self.H = int(z["H"])
        self.maxTime, self.deltaT = int(z["maxTime"]), float(z["deltaT"])
        self.tstride = int(z["tstride"])
        self.inst_graph = [int(g) for g in z["inst_graph"]]
        self.adjs = []
        gi = 0
        while "g%d_indptr" % gi in z:
            indptr, indices = z["g%d_indptr" % gi], z["g%d_indices" % gi]
            n = len(indptr) - 1
            self.adjs.append(scipy.sparse.csr_matrix(
                (np.ones(len(indices), dtype=np.int64), indices, indptr), shape=(n, n)))
            gi += 1
        self.x = torch.from_numpy(z["x"])
        self.params = {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("p:")}
        self.probs32 = torch.from_numpy(z["probs32"])
        self.probs64 = torch.from_numpy(z["probs64"])
        self.has_grads = any(k.startswith("g32:") for k in z.files)
        self.grads = {}
        for k in z.files:
            if k[:4] in ("g32:", "g64:"):
                prec, mode, key = k.split(":", 2)
                self.grads.setdefault((prec, mode), {})[key] = torch.from_numpy(z[k])
        self.M = self.x.shape[0]
        self.T = len(np.arange(0, self.maxTime, self.deltaT))
        self.w_seed = int(z["w_seed"])

    def weight(self):
        return torch.randn(self.T, self.M, 3, dtype=torch.float32,
                           generator=torch.Generator().manual_seed(self.w_seed))

    def sizes(self):
        return [self.adjs[g].shape[0] for g in self.inst_graph]

    def x_as_model_input(self):
        """sim: [B, N, 3+H] like the reference DataLoader; ngraphs: [sum N, 3+H]."""
        if self.variant == "sim":
            return self.x.view(len(self.inst_graph), -1, self.x.shape[1])
        return self.x
