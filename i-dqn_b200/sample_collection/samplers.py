"""Sampling distributions — drop-in for slimdqn/sample_collection/samplers.py.

The key<->index bookkeeping (O(1) swap-remove) and the PCG64 draws stay on the host, as SURVEY App. A
recommends (32 numbers per step; numpy *is* the reference's generator, so the stream is bit-identical); the
SumTree arithmetic of the prioritised sampler runs on the GPU."""
from __future__ import annotations

import os

import numpy as np

from .. import checkpoint as ckpt
from . import ReplayItemID
from .sum_tree import SumTree


class UniformSamplingDistribution:
    """samplers.py:13-49."""

    def __init__(self, seed: int) -> None:
        self._rng_key = np.random.default_rng(seed)
        self._key_to_index = {}
        self._index_to_key = []

    def add(self, key: ReplayItemID) -> None:
        self._key_to_index[key] = len(self._index_to_key)
        self._index_to_key.append(key)

    def remove(self, key: ReplayItemID) -> None:
        assert key in self._key_to_index, ValueError(f"Key {key} not found.")
        hole = self._key_to_index.pop(key)
        tail = self._index_to_key.pop()
        if tail != key:  # the last key moves into the hole (samplers.py:31-37)
            self._index_to_key[hole] = tail
            self._key_to_index[tail] = hole

    def sample(self, size: int):
        assert self._index_to_key, ValueError("No keys to sample from.")
        picks = self._rng_key.integers(len(self._index_to_key), size=size)
        table = self._index_to_key
        return np.fromiter((table[i] for i in picks), dtype=np.int32, count=size)

    # ---- checkpoint: the key table and the generator state (a reloaded sampler draws the same keys) ----------------
    def _meta(self) -> dict:
        return {"type": type(self).__name__}

    def save(self, directory: str) -> None:
        os.makedirs(directory, exist_ok=True)
        np.save(os.path.join(directory, "index_to_key.npy"), np.asarray(self._index_to_key, np.int64))
        ckpt.write_json(os.path.join(directory, "sampler.json"),
                        {**self._meta(), "bit_generator": self._rng_key.bit_generator.state})

    def load(self, directory: str) -> None:
        meta = ckpt.read_json(os.path.join(directory, "sampler.json"))
        for k, v in self._meta().items():
            if meta.get(k) != v:
                raise ValueError(f"sampler checkpoint has {k}={meta.get(k)!r}, this sampler {v!r}")
        self._index_to_key = [int(k) for k in np.load(os.path.join(directory, "index_to_key.npy"))]
        self._key_to_index = {k: i for i, k in enumerate(self._index_to_key)}
        self._rng_key.bit_generator.state = meta["bit_generator"]


class PrioritizedSamplingDistribution(UniformSamplingDistribution):
    """samplers.py:52-116 with the sum tree on the device."""

    def __init__(self, seed: int, max_capacity: int, priority_exponent: float = 1.0, device: int = 0) -> None:
        self._max_capacity = max_capacity
        self._priority_exponent = priority_exponent
        self._sum_tree = SumTree(self._max_capacity, device=device)
        super().__init__(seed=seed)

    AT_MAX = object()  # default priority of add(): the tree's max_recorded_priority (sum_tree.py:18,32)

    def add(self, key: ReplayItemID, priority=AT_MAX) -> None:
        """samplers.py:66-73.  Without a priority the element enters at ``max_recorded_priority`` so that it is sampled
        at least once -- the wiring the reference ships the pieces for but never connects (its ``collect_single_sample``
        passes no priority, utils.py:27-35, and its ``add`` would raise a TypeError there)."""
        super().add(key)
        if priority is PrioritizedSamplingDistribution.AT_MAX:
            self._sum_tree.set_at_max(self._key_to_index[key])
            return
        if priority is None:
            priority = 0.0
        # scalar power, exactly as samplers.py:72 (numpy's vectorised pow can differ from the scalar one by 1 ulp)
        self._sum_tree.set(self._key_to_index[key], 0.0 if priority == 0.0 else priority ** self._priority_exponent)

    def update(self, keys, priorities) -> None:
        if not isinstance(keys, np.ndarray):
            keys = np.asarray([keys], dtype=np.int32)
        priorities = np.where(priorities == 0.0, 0.0, priorities ** self._priority_exponent)  # array power, :81
        leaves = np.fromiter((self._key_to_index[int(k)] for k in keys), dtype=np.int32, count=len(keys))
        self._sum_tree.set(leaves, np.atleast_1d(priorities))

    def update_from_learner(self, keys, engine) -> None:
        """``update(keys, priorities)`` with priorities = mean over the heads of the |TD error| of ``engine``'s last step
        (replay_buffer.py:232-237 fed from the learner).  With priority_exponent == 1 nothing leaves the device."""
        leaves = np.fromiter((self._key_to_index[int(k)] for k in keys), dtype=np.int32, count=len(keys))
        if self._priority_exponent == 1.0:
            self._sum_tree.update_from_learner(engine, leaves)
        else:  # the array power stays numpy's (bit-exact with the reference): priorities visit the host
            td = engine.td_abs().astype(np.float64)
            pr = td[0].copy()
            for k in range(1, td.shape[0]):
                pr += td[k]
            self.update(np.asarray(keys), pr / td.shape[0])

    def remove(self, key: ReplayItemID) -> None:
        hole = self._key_to_index[key]
        tail = len(self._index_to_key) - 1
        if hole == tail:
            self._sum_tree.set(hole, 0.0)
        else:  # mirror the swap-remove inside the tree (samplers.py:96-102)
            self._sum_tree.set(np.asarray([hole, tail], dtype=np.int32),
                               np.asarray([self._sum_tree.get(tail), 0.0], dtype=np.float64))
        super().remove(key)

    def _meta(self) -> dict:
        return {**super()._meta(), "max_capacity": int(self._max_capacity),
                "priority_exponent": float(self._priority_exponent)}

    def save(self, directory: str) -> None:
        super().save(directory)
        np.save(os.path.join(directory, "sum_tree_nodes.npy"), self._sum_tree._nodes)
        ckpt.write_json(os.path.join(directory, "sum_tree.json"),
                        {"max_recorded_priority": self._sum_tree.max_recorded_priority})

    def load(self, directory: str) -> None:
        """The tree's nodes are uploaded as saved (``write_nodes``), never rebuilt through ``set``."""
        super().load(directory)
        self._sum_tree.write_nodes(np.load(os.path.join(directory, "sum_tree_nodes.npy")),
                                   ckpt.read_json(os.path.join(directory, "sum_tree.json"))["max_recorded_priority"])

    def sample(self, size: int):
        # samplers.py:105-108: an all-zero tree falls back to the uniform sampler (the reference spells the intent as
        # ``super().sample(size).keys``, which cannot work on an ndarray; the fallback itself is what is kept).  The
        # root is NOT read back every step: the device reports an empty tree as an out-of-range target, and only
        # then the host looks at the root, rewinds the generator (the reference draws no uniforms in this branch) and
        # samples uniformly -- the PCG64 stream stays the reference's in both branches.
        rng_state = self._rng_key.bit_generator.state
        # rng.uniform(0.0, root) == 0.0 + root * rng.random(): the product is formed on the device (__dmul_rn),
        # so the root never has to come back to the host on the step path.
        units = self._rng_key.random(size)
        try:
            leaves = self._sum_tree.sample_unit(units)
        except ValueError:
            if self._sum_tree.root != 0.0:
                raise
            self._rng_key.bit_generator.state = rng_state
            return super().sample(size)
        table = self._index_to_key
        return np.fromiter((table[i] for i in leaves), dtype=np.int32, count=size)
