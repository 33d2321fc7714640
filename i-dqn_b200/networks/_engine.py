"""Host-side owner of one ``idqn_handle``: configuration, the arena <-> Flax-pytree mapping and the live
device-resident views handed out as ``agent.params`` / ``agent.target_params`` / ``agent.optimizer_state``."""
from __future__ import annotations

import ctypes as C
import os
import weakref
from collections import namedtuple
from typing import Any, Dict, List, Optional, Sequence

import numpy as np

from .. import _lib as L

# optax state containers the reference exposes through ``agent.optimizer_state`` (idqn.py:53)
ScaleByAdamState = namedtuple("ScaleByAdamState", ["count", "mu", "nu"])
EmptyState = namedtuple("EmptyState", [])


def _get(obj, name):
    """Field of a ReplayElement-like batch (attribute access) or of a dict."""
    if isinstance(obj, dict):
        return obj[name]
    return getattr(obj, name)


class Leaf:
    """Live view of one parameter leaf ([K, *shape], or [*shape] for DQN) living in a device arena."""

    def __init__(self, engine: "Engine", which: int, index: int, squeeze: bool):
        self._engine, self._which, self._index, self._squeeze = engine, which, index, squeeze
        info = engine.leaves[index]
        self.shape = tuple(info["shape"]) if squeeze else (engine.K,) + tuple(info["shape"])
        self.dtype = np.dtype(np.float32)
        self.ndim = len(self.shape)
        self.size = int(np.prod(self.shape))

    def __array__(self, dtype=None, copy=None):
        a = self._engine.download_leaf(self._which, self._index)
        a = a[0] if self._squeeze else a
        return a.astype(dtype) if dtype is not None else a

    def __getitem__(self, item):
        return np.asarray(self)[item]

    def __repr__(self):
        return f"Leaf(device, which={self._which}, shape={self.shape})"


def _module(inner: Dict[str, Any], name: str, create: bool = False) -> Dict[str, Any]:
    """The {"kernel", "bias"} dict of module ``name``; "Stack_0/Conv_1" is flax's nested ``inner["Stack_0"]["Conv_1"]``."""
    node = inner
    for part in name.split("/"):
        node = node.setdefault(part, {}) if create else node[part]
    return node


def _map_leaves(fn, tree):
    if isinstance(tree, dict):
        return {k: _map_leaves(fn, v) for k, v in tree.items()}
    return fn(tree)


class Tree(dict):
    """``{"params": {"Conv_0": {"kernel": Leaf, "bias": Leaf}, ...}}`` backed by an engine arena.

    It is a *live view* of device memory (not an immutable snapshot like a jax pytree): pass it back to the
    owning agent's methods and no data moves; ``np.asarray(leaf)`` / ``to_host()`` copy out."""

    def __init__(self, engine: "Engine", which: int, squeeze: bool):
        inner: Dict[str, Any] = {}
        for i, info in enumerate(engine.leaves):
            _module(inner, info["module"], create=True)[info["kind"]] = Leaf(engine, which, i, squeeze)
        super().__init__(params=inner)
        self._engine_ref = weakref.ref(engine)
        self._which = which
        self._squeeze = squeeze

    def copy(self):  # idqn.py:78 ``self.params.copy()``
        return self

    def to_host(self) -> Dict[str, Any]:
        return {"params": _map_leaves(np.asarray, self["params"])}

    def is_view_of(self, engine: "Engine", which: int) -> bool:
        return self._engine_ref() is engine and self._which == which


class CountView:
    def __init__(self, engine: "Engine", squeeze: bool):
        self._engine, self._squeeze = engine, squeeze
        self.shape = () if squeeze else (engine.K,)
        self.dtype = np.dtype(np.int32)

    def __array__(self, dtype=None, copy=None):
        c = self._engine.get_count()
        c = c[0] if self._squeeze else c
        return np.asarray(c, dtype=dtype) if dtype is not None else np.asarray(c)

    def __int__(self):
        return int(np.asarray(self))

    def __repr__(self):
        return f"CountView({np.asarray(self)!r})"


class Engine:
    """One ``idqn_handle`` (K heads on one device)."""

    def __init__(self, observation_dim, n_actions: int, n_heads: int, features: Sequence[int], architecture_type: str,
                 learning_rate: float, gamma: float, update_horizon: int, adam_eps: float, batch_size: int = 32,
                 device: int = 0, flags: int = 0):
        self.lib = L.lib()
        if architecture_type not in ("cnn", "fc", "impala"):
            raise ValueError(f"architecture_type={architecture_type!r}: expected 'cnn', 'impala' or 'fc'")
        features = [int(f) for f in features]
        if int(n_actions) > L.MAX_ACTIONS:
            raise ValueError(f"n_actions={n_actions}: the fused final-layer kernels hold at most {L.MAX_ACTIONS} actions")
        if len(features) > L.MAX_FEATURES:
            raise ValueError("too many feature layers")
        obs = tuple(int(d) for d in np.atleast_1d(observation_dim))
        cfg = L.Config()
        cfg.arch = {"cnn": L.ARCH_CNN, "impala": L.ARCH_IMPALA, "fc": L.ARCH_FC}[architecture_type]
        if architecture_type in ("cnn", "impala"):
            if len(obs) != 3:
                raise ValueError(f"{architecture_type} needs observation_dim=(H, W, C)")
            cfg.obs[:] = obs
        else:
            cfg.obs[:] = (int(np.prod(obs)), 1, 1)
        cfg.n_actions, cfg.n_heads, cfg.n_features = int(n_actions), int(n_heads), len(features)
        for i, f in enumerate(features):
            cfg.features[i] = f
        cfg.batch_size = int(batch_size)
        cfg.learning_rate, cfg.adam_eps = float(learning_rate), float(adam_eps)
        cfg.gamma_n = float(np.float32(float(gamma) ** int(update_horizon)))  # idqn.py:122 python float -> f32
        # IDQN_FLAGS in the environment ORs extra IDQN_F_* bits into every handle (A/B runs under ncu / compute-sanitizer)
        cfg.device, cfg.flags = int(device), int(flags) | int(os.environ.get("IDQN_FLAGS", "0"))
        self.cfg = cfg
        self.K, self.B, self.A = int(n_heads), int(batch_size), int(n_actions)
        self.architecture_type = architecture_type
        self.obs_shape = obs
        self.in_elems = int(np.prod(obs))
        self.device = int(device)
        h = C.c_void_p()
        L.check(self.lib.idqn_create(C.byref(cfg), C.byref(h)))
        self.h = h
        self._finalizer = weakref.finalize(self, self.lib.idqn_destroy, h)
        self.stride = int(self.lib.idqn_arena_stride(h))
        self._inflight = [None, None]  # host arrays of the two most recent submit_host calls
        self.leaves: List[Dict[str, Any]] = []
        for i in range(self.lib.idqn_leaf_count(h)):
            off, size, ndim = C.c_int64(), C.c_int64(), C.c_int32()
            shape = np.zeros(4, np.int32)
            name = C.create_string_buffer(16)
            L.check(self.lib.idqn_leaf_info(h, i, C.byref(off), C.byref(size), L.ptr(shape), C.byref(ndim), name))
            self.leaves.append(dict(module=name.value.decode(), kind="kernel" if i % 2 == 0 else "bias",
                                    offset=off.value, size=size.value, shape=tuple(int(s) for s in shape[:ndim.value])))
        self.n_params = sum(l["size"] for l in self.leaves)

    # ---- arena <-> pytree ------------------------------------------------------------------------
    def close(self):
        self._finalizer()

    def upload_leaf(self, which: int, index: int, value) -> None:
        info = self.leaves[index]
        a = np.ascontiguousarray(np.asarray(value, dtype=np.float32)).reshape(self.K, info["size"])
        for k in range(self.K):
            row = np.ascontiguousarray(a[k])
            L.check(self.lib.idqn_upload(self.h, which, k, info["offset"], L.ptr(row), info["size"]))

    def download_leaf(self, which: int, index: int) -> np.ndarray:
        info = self.leaves[index]
        out = np.empty((self.K, info["size"]), np.float32)
        for k in range(self.K):
            row = out[k]
            L.check(self.lib.idqn_download(self.h, which, k, info["offset"], L.ptr(row), info["size"]))
        return out.reshape((self.K,) + info["shape"])

    def upload_tree(self, which: int, tree, squeezed: bool = False) -> None:
        inner = tree["params"] if "params" in tree else tree
        for i, info in enumerate(self.leaves):
            v = np.asarray(_module(inner, info["module"])[info["kind"]], dtype=np.float32)
            if squeezed:
                v = v[None]
            if v.shape != (self.K,) + info["shape"]:
                raise ValueError(f"{info['module']}/{info['kind']}: expected {(self.K,) + info['shape']}, got {v.shape}")
            self.upload_leaf(which, i, v)

    def download_tree(self, which: int, squeezed: bool = False) -> Dict[str, Any]:
        inner: Dict[str, Any] = {}
        for i, info in enumerate(self.leaves):
            a = self.download_leaf(which, i)
            _module(inner, info["module"], create=True)[info["kind"]] = a[0] if squeezed else a
        return {"params": inner}

    def download_arena(self, which: int) -> np.ndarray:
        out = np.empty((self.K, self.stride), np.float32)
        for k in range(self.K):
            row = out[k]
            L.check(self.lib.idqn_download(self.h, which, k, 0, L.ptr(row), self.stride))
        return out

    def layer_output_shapes(self):
        """[(B, OH, OW, OC)] of every hidden layer (the final Dense is fused into the loss kernel)."""
        from .architectures._shapes import CNN_SPECS, same_out
        shapes = []
        if self.architecture_type == "impala":
            # engine layer order: per Stack [Conv_0, pool, Conv_1, Conv_2, Conv_3, Conv_4], then the dense trunk
            h, w, _ = self.obs_shape
            for i in range(3):
                f = int(self.cfg.features[i])
                shapes.append((self.B, h, w, f))
                h, w = same_out(h, 2), same_out(w, 2)
                shapes.extend([(self.B, h, w, f)] * 5)
            start = 3
        elif self.architecture_type == "cnn":
            h, w, _ = self.obs_shape
            for i, (_, s) in enumerate(CNN_SPECS):
                h, w = same_out(h, s), same_out(w, s)
                shapes.append((self.B, h, w, int(self.cfg.features[i])))
            start = 3
        else:
            start = 0
        for i in range(start, int(self.cfg.n_features)):
            shapes.append((self.B, 1, 1, int(self.cfg.features[i])))
        return shapes

    def download_activation(self, net: int, layer: int) -> np.ndarray:
        shape = self.layer_output_shapes()[layer]
        out = np.empty(shape, np.float32)
        L.check(self.lib.idqn_download_activation(self.h, net, layer, L.ptr(out), out.size))
        return out

    def get_count(self) -> np.ndarray:
        c = np.zeros(self.K, np.int32)
        L.check(self.lib.idqn_get_count(self.h, L.ptr(c)))
        return c

    def set_count(self, count) -> None:
        c = np.ascontiguousarray(np.broadcast_to(np.asarray(count, np.int32), (self.K,)))
        L.check(self.lib.idqn_set_count(self.h, L.ptr(c)))

    # ---- the step -----------------------------------------------------------------------------------
    def pack_batch(self, batch):
        """(state, next_state, is_u8, action i32, reward f32, terminal u8) as C-contiguous arrays — the dtype flow
        of the reference's jit boundary (SURVEY App. A): int64->int32, float64->float32, bool->u8."""
        s, s2 = np.asarray(_get(batch, "state")), np.asarray(_get(batch, "next_state"))
        if s.shape[0] != self.B:
            raise ValueError(f"batch has {s.shape[0]} samples, the engine was built for batch_size={self.B}")
        u8 = s.dtype == np.uint8 and s2.dtype == np.uint8
        dt = np.uint8 if u8 else np.float32
        s = np.ascontiguousarray(s, dtype=dt).reshape(self.B, -1)
        s2 = np.ascontiguousarray(s2, dtype=dt).reshape(self.B, -1)
        if s.shape[1] != self.in_elems:
            raise ValueError(f"sample has {s.shape[1]} elements, the network expects {self.in_elems}")
        a = np.ascontiguousarray(np.asarray(_get(batch, "action")), dtype=np.int32).reshape(self.B)
        if a.min() < 0 or a.max() >= self.A:
            raise ValueError("action outside [0, n_actions)")
        r = np.ascontiguousarray(np.asarray(_get(batch, "reward")), dtype=np.float32).reshape(self.B)
        d = np.ascontiguousarray(np.asarray(_get(batch, "is_terminal")).astype(bool), dtype=np.uint8).reshape(self.B)
        return s, s2, int(u8), a, r, d

    def learn_host(self, batch, want_losses: bool = True) -> Optional[np.ndarray]:
        if not want_losses:
            # nobody reads this step's losses (update_online_params, idqn.py:65-72, only accumulates them on the device):
            # take the two-slot pipelined staging -- the H2D copies of this batch run on the copy stream while the
            # previous step still computes and the call returns as soon as everything is enqueued, which is how the
            # reference's own call behaves (jax dispatches learn_on_batch asynchronously)
            self.submit_host(batch)
            return None
        s, s2, u8, a, r, d = self.pack_batch(batch)
        losses = np.zeros(self.K, np.float32) if want_losses else None
        L.check(self.lib.idqn_learn_on_batch_host(self.h, L.ptr(s), L.ptr(s2), u8, L.ptr(a), L.ptr(r), L.ptr(d),
                                                  L.ptr(losses) if want_losses else None))
        return losses

    def submit_host(self, batch) -> int:
        """Pipelined host path: enqueue the H2D copies (copy stream) and the step; returns a ticket.  The arrays of
        ``batch`` must stay alive and unmodified until ``wait_losses(ticket)``."""
        s, s2, u8, a, r, d = self.pack_batch(batch)
        ticket = C.c_int64(0)
        L.check(self.lib.idqn_submit_batch_host(self.h, L.ptr(s), L.ptr(s2), u8, L.ptr(a), L.ptr(r), L.ptr(d),
                                                C.byref(ticket)))
        self._inflight[ticket.value & 1] = (s, s2, a, r, d)  # keep converted copies alive
        return ticket.value

    def wait_losses(self, ticket: int) -> np.ndarray:
        losses = np.zeros(self.K, np.float32)
        L.check(self.lib.idqn_wait_losses(self.h, C.c_int64(ticket), L.ptr(losses)))
        return losses

    def learn_dev(self, s_ptr: int, s2_ptr: int, u8: int, a_ptr: int, r_ptr: int, d_ptr: int,
                  want_losses: bool = False) -> Optional[np.ndarray]:
        losses = np.zeros(self.K, np.float32) if want_losses else None
        L.check(self.lib.idqn_learn_on_batch_dev(self.h, C.c_void_p(s_ptr), C.c_void_p(s2_ptr), int(u8),
                                                 C.c_void_p(a_ptr), C.c_void_p(r_ptr), C.c_void_p(d_ptr),
                                                 L.ptr(losses) if want_losses else None))
        return losses

    def set_loss_accumulation(self, on: bool) -> None:
        """idqn.py:72 — whether the following steps add their losses to the device-side running sums."""
        L.check(self.lib.idqn_set_loss_accumulation(self.h, int(bool(on))))

    def td_abs(self) -> np.ndarray:
        """|Q(s_b, a_b) - y_b| per head and sample of the most recent step, float32 [K, B]."""
        out = np.zeros((self.K, self.B), np.float32)
        L.check(self.lib.idqn_read_td_abs(self.h, L.ptr(out)))
        return out

    def cumulated_losses(self, reset: bool = False) -> np.ndarray:
        out = np.zeros(self.K, np.float64)
        L.check(self.lib.idqn_read_cumulated_losses(self.h, L.ptr(out), int(reset)))
        return out

    def shift_params(self):
        L.check(self.lib.idqn_shift_params(self.h))

    def sync_target(self):
        L.check(self.lib.idqn_sync_target(self.h))

    def copy_online_to_target(self):
        L.check(self.lib.idqn_copy_online_to_target(self.h))

    def apply(self, which: int, head: int, x) -> np.ndarray:
        x = np.asarray(x)
        u8 = x.dtype == np.uint8
        x = np.ascontiguousarray(x, dtype=np.uint8 if u8 else np.float32)
        n = x.size // self.in_elems
        if n * self.in_elems != x.size:
            raise ValueError(f"input of {x.size} elements is not a multiple of the observation size {self.in_elems}")
        q = np.zeros((n, self.A), np.float32)
        L.check(self.lib.idqn_apply_host(self.h, which, head, L.ptr(x), int(u8), n, L.ptr(q)))
        return q

    def best_action(self, which: int, head: int, state) -> int:
        x = np.asarray(state)
        u8 = x.dtype == np.uint8
        if not u8 and self.architecture_type == "cnn":
            # the Atari wrapper hands over float32 frames holding 0..255 (environments/atari.py:43-45): as uint8 they
            # take the learning step's own kernels (exact: the network divides by 255 either way)
            xu = x.astype(np.uint8)
            if np.array_equal(xu, x):
                x, u8 = xu, True
        x = np.ascontiguousarray(x, dtype=np.uint8 if u8 else np.float32)
        if x.size != self.in_elems:
            raise ValueError(f"state has {x.size} elements, expected {self.in_elems}")
        out = C.c_int32()
        L.check(self.lib.idqn_best_action(self.h, which, head, L.ptr(x), int(u8), C.byref(out)))
        return int(out.value)

    def select_action(self, state, key, n_actions: int, epsilon: float):
        """utils.py:8-15 in one C call: the three threefry draws, and on a greedy step best_action of the drawn head as
        one CUDA-graph launch.  Returns (action, explored, head)."""
        from .. import _prng
        x = np.asarray(state)
        u8 = x.dtype == np.uint8
        if not u8 and self.architecture_type == "cnn":
            xu = x.astype(np.uint8)  # atari.py:43-45 hands over float32 frames holding 0..255
            if np.array_equal(xu, x):
                x, u8 = xu, True
        x = np.ascontiguousarray(x, dtype=np.uint8 if u8 else np.float32)
        if x.size != self.in_elems:
            raise ValueError(f"state has {x.size} elements, expected {self.in_elems}")
        k = _prng.as_key(key)
        out, info = C.c_int32(), np.zeros(2, np.int32)
        L.check(self.lib.idqn_select_action(self.h, L.ptr(x), int(u8), int(k[0]), int(k[1]), int(n_actions),
                                            float(epsilon), C.byref(out), L.ptr(info)))
        return int(out.value), bool(info[0]), int(info[1])

    def select_actions(self, states, keys, n_actions: int, epsilon: float):
        """``select_action`` for N environments in one C call: env i draws with ``keys[i]`` and the greedy ones share one
        device pass per chunk of up to B states.  Returns (actions int32[N], explored bool[N], heads int32[N])."""
        from .. import _prng
        ks = np.ascontiguousarray([_prng.as_key(k) for k in keys], np.uint32).reshape(-1, 2)
        n = len(ks)
        x = np.asarray(states)
        u8 = x.dtype == np.uint8
        if not u8 and self.architecture_type == "cnn":
            xu = x.astype(np.uint8)  # atari.py:43-45 hands over float32 frames holding 0..255
            if np.array_equal(xu, x):
                x, u8 = xu, True
        x = np.ascontiguousarray(x, dtype=np.uint8 if u8 else np.float32)
        if x.size != n * self.in_elems:
            raise ValueError(f"states have {x.size} elements, expected {n} x {self.in_elems} for {n} keys")
        out, info = np.zeros(n, np.int32), np.zeros((n, 2), np.int32)
        L.check(self.lib.idqn_select_actions(self.h, L.ptr(x), int(u8), n, L.ptr(ks), int(n_actions), float(epsilon),
                                             L.ptr(out), L.ptr(info)))
        return out, info[:, 0].astype(bool), info[:, 1].copy()

    def mark_head_planes_dirty(self, which: int, head: int) -> None:
        """One head of an arena was rewritten behind the library's back (neighbour exchange): rebuild its planes."""
        L.check(self.lib.idqn_mark_head_planes_dirty(self.h, which, int(head)))

    def mark_planes_dirty(self, which: int) -> None:
        """An arena was written through its raw pointer (NCCL recv / peer copy): rebuild its bf16 operand planes."""
        L.check(self.lib.idqn_mark_planes_dirty(self.h, which))

    def arena_ptr(self, which: int) -> int:
        return int(self.lib.idqn_arena_ptr(self.h, which))
