"""``SumTree`` — drop-in for slimdqn/sample_collection/sum_tree.py with the float64 node array resident in
HBM and ``set`` / ``query`` running as CUDA kernels that reproduce the reference's arithmetic bit for bit
(csrc/sumtree.cu).  Same methods, attributes and exception types as the reference (:8-102)."""
from __future__ import annotations

import ctypes as C
import weakref

import numpy as np

from .. import _lib as L


class SumTree:
    def __init__(self, capacity: int, device: int = 0) -> None:
        assert capacity > 0, "Capacity to sum tree must be positive."  # sum_tree.py:12
        lib = L.lib()
        self._lib = lib
        h = C.c_void_p()
        L.check(lib.idqn_sumtree_create(int(capacity), int(device), C.byref(h)))
        self._h = h
        self._finalizer = weakref.finalize(self, lib.idqn_sumtree_destroy, h)
        self._capacity = capacity
        self._depth = int(lib.idqn_sumtree_depth(h))
        self._first_leaf_offset = (2 ** (self._depth - 1)) - 1
        self._n_nodes = int(lib.idqn_sumtree_num_nodes(h))
        self.device = int(device)

    @property
    def max_recorded_priority(self) -> float:
        """sum_tree.py:18,32 — tracked on the device (the learner-side priority updates never visit the host)."""
        v = C.c_double()
        L.check(self._lib.idqn_sumtree_max_recorded(self._h, C.byref(v)))
        return float(v.value)

    @property
    def _nodes(self) -> np.ndarray:
        """Host copy of the node array (tests reach into it, tests/test_sum_tree.py:36-38)."""
        out = np.empty(self._n_nodes, np.float64)
        L.check(self._lib.idqn_sumtree_read_nodes(self._h, L.ptr(out)))
        return out

    def write_nodes(self, nodes, max_recorded_priority: float) -> None:
        """Restore a saved tree: ``_nodes`` and ``max_recorded_priority`` uploaded unchanged.  (Replaying ``set`` on the
        leaves would not give the same nodes: each f64 node depends on the order of the adds that built it.)"""
        n = np.ascontiguousarray(nodes, dtype=np.float64)
        if n.shape != (self._n_nodes,):
            raise ValueError(f"{n.shape} nodes for a tree of {self._n_nodes}")
        L.check(self._lib.idqn_sumtree_write_nodes(self._h, L.ptr(n), float(max_recorded_priority)))

    def set(self, indices, values) -> None:  # sum_tree.py:20-47
        if isinstance(indices, (int, np.integer)):
            indices = np.asarray([indices], np.int32)
        if isinstance(values, (int, float, np.floating, np.integer)):
            values = np.asarray([values], np.float64)
        indices, values = np.asarray(indices), np.asarray(values)
        assert indices.shape == values.shape, "Indices and values must have the same shape."
        assert (values >= 0.0).all(), "Values must be positive."
        if indices.size == 0:
            return
        idx = np.ascontiguousarray(indices.ravel(), dtype=np.int32)
        val = np.ascontiguousarray(values.ravel(), dtype=np.float64)
        L.check(self._lib.idqn_sumtree_set(self._h, L.ptr(idx), L.ptr(val), idx.size))

    def set_at_max(self, index: int) -> None:
        """``set(index, max_recorded_priority)`` without reading the maximum back: how a NEW element enters a prioritised
        buffer (it will be sampled at least once)."""
        L.check(self._lib.idqn_sumtree_set_at_max(self._h, int(index)))

    def update_from_learner(self, engine, leaves) -> None:
        """``set(leaves, mean_k |TD_k|)`` with the per-sample TD errors of ``engine``'s last step taken on the device,
        ordered behind that step; no host synchronisation."""
        lv = np.ascontiguousarray(np.asarray(leaves).ravel(), dtype=np.int32)
        L.check(self._lib.idqn_sumtree_update_from_learner(self._h, engine.h, L.ptr(lv), lv.size))

    def get(self, index):  # sum_tree.py:49-51
        scalar = np.ndim(index) == 0
        idx = np.ascontiguousarray(np.atleast_1d(index).ravel(), dtype=np.int32)
        out = np.empty(idx.size, np.float64)
        L.check(self._lib.idqn_sumtree_get(self._h, L.ptr(idx), L.ptr(out), idx.size))
        return out[0] if scalar else out.reshape(np.shape(index))

    @property
    def root(self) -> float:  # sum_tree.py:53-56
        r = C.c_double()
        L.check(self._lib.idqn_sumtree_root(self._h, C.byref(r)))
        return np.float64(r.value)

    def query(self, targets):  # sum_tree.py:58-102
        scalar = isinstance(targets, (int, float))
        t = np.ascontiguousarray(np.atleast_1d(np.asarray(targets, dtype=np.float64)).ravel())
        out = np.empty(t.size, np.int32)
        L.check(self._lib.idqn_sumtree_query(self._h, L.ptr(t), L.ptr(out), t.size))  # ValueError if out of range
        return out if not scalar else out  # the reference returns a length-1 array for scalars too (:71-72)

    def sample_unit(self, unit_uniforms) -> np.ndarray:
        """Leaves for targets ``root * u`` — the device half of ``rng.uniform(0, root)`` + ``query``
        (samplers.py:110-111) without reading the root back to the host."""
        u = np.ascontiguousarray(np.asarray(unit_uniforms, dtype=np.float64).ravel())
        out = np.empty(u.size, np.int32)
        L.check(self._lib.idqn_sumtree_sample(self._h, L.ptr(u), L.ptr(out), u.size))
        return out
