"""Device-resident graphs and block-diagonal batches.

Replaces the host-side scipy CSR the reference keeps in ``ODEfunc.A`` /
``ODEfunc.A_list`` (ode_nn_ngraph_sim.py:41, ode_nn_ngraphs.py:41) and the
``scipy.sparse.block_diag`` + index upload it redoes at every Euler step
(ode_nn_ngraph_sim.py:68-71, ode_nn_ngraphs.py:65-71): the pattern is uploaded
once per graph, and one small descriptor is built once per distinct batch shape.
"""
import ctypes

import numpy as np

from . import _lib


class DeviceGraph:
    """CSR pattern of one graph in HBM (gnode_graph_t). indptr / indices keep the host copy of what was uploaded: the
    columns of every row in ascending order, the order of the device CSR and of the edge gradients."""

    def __init__(self, A):
        import scipy.sparse
        A = scipy.sparse.csr_matrix(A)          # accepts csr_array / csr_matrix / anything scipy converts
        if A.shape[0] != A.shape[1]:
            raise ValueError("adjacency must be square, got %r" % (A.shape,))
        self.n = int(A.shape[0])
        indptr = np.ascontiguousarray(A.indptr, dtype=np.int32)
        indices = np.asarray(A.indices[:indptr[-1]], dtype=np.int32)
        rows = np.repeat(np.arange(self.n, dtype=np.int32), np.diff(indptr))
        order = np.lexsort((indices, rows))                                      # per-row column sort
        indices = np.ascontiguousarray(indices[order])
        self.indptr, self.indices = indptr, indices
        self._values = np.asarray(A.data[:indptr[-1]])[order]
        self.nnz = int(indptr[-1])
        h = ctypes.c_void_p()
        L = _lib.lib()
        _lib.check(L.gnode_graph_create(self.n, self.nnz, indptr.ctypes.data_as(_lib.c_int32_p),
                                        indices.ctypes.data_as(_lib.c_int32_p), ctypes.byref(h)),
                   "gnode_graph_create")
        self.handle = h
        n, nnz, md, sym = ctypes.c_int32(), ctypes.c_int64(), ctypes.c_int32(), ctypes.c_int32()
        _lib.check(L.gnode_graph_info(h, ctypes.byref(n), ctypes.byref(nnz), ctypes.byref(md), ctypes.byref(sym)),
                   "gnode_graph_info")
        self.max_degree, self.symmetric = int(md.value), bool(sym.value)

    def edges(self):
        """(row, col) of every stored entry, int64, in the order of the edge gradients (rollout's edge_weight)."""
        return np.repeat(np.arange(self.n, dtype=np.int64), np.diff(self.indptr)), self.indices.astype(np.int64)

    def edge_values(self):
        """A's stored values (float32) in edges() order: a weighted matrix's weights as rollout's contact_weight."""
        return self._values.astype(np.float32)

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                _lib.lib().gnode_graph_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class DeviceBatch:
    """Block-diagonal batch: instance i = graphs[i] (gnode_batch_t)."""

    def __init__(self, graphs):
        self.graphs = list(graphs)              # keep the graphs alive
        arr = (ctypes.c_void_p * len(self.graphs))(*[g.handle for g in self.graphs])
        h = ctypes.c_void_p()
        _lib.check(_lib.lib().gnode_batch_create(arr, len(self.graphs), ctypes.byref(h)), "gnode_batch_create")
        self.handle = h
        self.M = int(_lib.lib().gnode_batch_rows(h))
        self.sizes = [g.n for g in self.graphs]
        # edge vector of the batch (edge gradients): instance after instance, edge_offsets[i] = first entry of instance i
        self.edge_offsets = np.concatenate(([0], np.cumsum([g.nnz for g in self.graphs]))).astype(np.int64)
        self.nnz = int(self.edge_offsets[-1])

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                _lib.lib().gnode_batch_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class BatchCache:
    """Small LRU of DeviceBatch objects keyed by the tuple of graph ids."""

    def __init__(self, capacity=64):
        self.capacity = capacity
        self._d = {}

    def get(self, graphs):
        key = tuple(id(g) for g in graphs)
        b = self._d.pop(key, None)
        if b is None:
            b = DeviceBatch(graphs)
        self._d[key] = b
        while len(self._d) > self.capacity:
            self._d.pop(next(iter(self._d)))
        return b
