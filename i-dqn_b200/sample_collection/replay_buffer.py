"""``ReplayBuffer`` — drop-in for slimdqn/sample_collection/replay_buffer.py with the element store resident
in HBM (csrc/replay.cu) instead of a host ``OrderedDict`` of snappy blobs.

What stays on the host (env-rate, a few hundred bytes per step): the n-step/frame-stack accumulator
(:103-200) and the sampler's key bookkeeping.  What moves to the device: element storage (``add`` uploads
the two stacks once, :207-210) and the batch assembly of ``sample`` (:222-230), which becomes one coalesced
gather kernel writing straight into the learner's batch staging (``learn_step_on``), so the per-step
dict-lookup + decompress + np.stack + H2D path of the reference disappears.

FIFO semantics are the reference's: keys are the cumulative ``add_count`` (:207), the oldest key is evicted
once ``add_count > max_capacity`` (:211-213); key ``k`` lives in slot ``k % max_capacity``.

``frame_store=True`` keeps each observation once (the memory saving the reference gets from ``compress=True``,
:36-57,204-205): a device ring of frames plus, per element, the frame ids of its two stacks.  The host side of it
(which frames exist, when the ring must grow) is plain bookkeeping over a store object with ``put_frame`` /
``put_element`` / ``grow``."""
from __future__ import annotations

import collections
import ctypes as C
import dataclasses
import os
import typing
import weakref
import zlib
from typing import Any, Iterable, Iterator, Optional

import numpy as np

from .. import _lib as L
from .. import checkpoint as ckpt
from . import ReplayItemID


class TransitionElement(typing.NamedTuple):  # replay_buffer.py:18-23
    observation: Any
    action: int
    reward: float
    is_terminal: bool
    episode_end: bool = False


@dataclasses.dataclass(frozen=True)
class ReplayElement:  # replay_buffer.py:26-69
    state: Any
    action: Any
    reward: Any
    next_state: Any
    is_terminal: Any
    episode_end: Any

    def replace(self, **changes) -> "ReplayElement":
        return dataclasses.replace(self, **changes)

    # The reference packs with snappy (:36-57), which is a host-storage detail; the device store keeps raw
    # bytes.  pack/unpack are kept for API parity (round trip pinned by tests/test_replay_buffer.py:21-49 of the
    # reference) on top of zlib from the standard library.
    @staticmethod
    def compress(buffer: np.ndarray):
        buffer = np.ascontiguousarray(buffer)
        return (zlib.compress(buffer.tobytes(), 1), buffer.shape, buffer.dtype.str)

    @staticmethod
    def uncompress(packed) -> np.ndarray:
        blob, shape, dtype = packed
        return np.frombuffer(zlib.decompress(blob), dtype=dtype).reshape(shape).copy()

    def pack(self) -> "ReplayElement":
        return self.replace(state=self.compress(self.state), next_state=self.compress(self.next_state))

    def unpack(self) -> "ReplayElement":
        return self.replace(state=self.uncompress(self.state), next_state=self.uncompress(self.next_state))


class _Store:
    """What both device stores share: the host gather, and the bulk slot transfers and digest of a checkpoint."""

    def gather(self, slots: np.ndarray):
        n = len(slots)
        slots = np.ascontiguousarray(slots, dtype=np.int64)
        s = np.empty((n,) + self.shape, self.dtype)
        s2 = np.empty((n,) + self.shape, self.dtype)
        a, r = np.empty(n, np.int32), np.empty(n, np.float64)
        d, e = np.empty(n, np.uint8), np.empty(n, np.uint8)
        L.check(self.lib.idqn_replay_gather_host(self.h, L.ptr(slots), n, L.ptr(s), L.ptr(s2), L.ptr(a), L.ptr(r),
                                                 L.ptr(d), L.ptr(e)))
        return s, s2, a.astype(np.int64), r, d.astype(bool), e.astype(bool)

    def _slot_stacks(self, n: int):
        raise NotImplementedError

    def read_slots(self, lo: int, n: int):
        """(state stacks or frame-id rows, next_state stacks or None, action i32, reward f64, terminal u8,
        episode_end u8) of slots [lo, lo + n)."""
        s, s2 = self._slot_stacks(n)
        a, r = np.empty(n, np.int32), np.empty(n, np.float64)
        d, e = np.empty(n, np.uint8), np.empty(n, np.uint8)
        L.check(self.lib.idqn_replay_read_slots(self.h, int(lo), int(n), L.ptr(s), None if s2 is None else L.ptr(s2),
                                                L.ptr(a), L.ptr(r), L.ptr(d), L.ptr(e)))
        return s, s2, a, r, d, e

    def write_slots(self, lo: int, s, s2, a, r, d, e) -> None:
        like, like2 = self._slot_stacks(0)
        s = np.ascontiguousarray(s, like.dtype)
        s2 = None if like2 is None else np.ascontiguousarray(s2, like2.dtype)
        a, r = np.ascontiguousarray(a, np.int32), np.ascontiguousarray(r, np.float64)
        d, e = np.ascontiguousarray(d, np.uint8), np.ascontiguousarray(e, np.uint8)
        if s.shape[1:] != like.shape[1:] or any(len(x) != len(s) for x in (a, r, d, e)):
            raise ValueError("slot arrays do not match the store")
        L.check(self.lib.idqn_replay_write_slots(self.h, int(lo), len(s), L.ptr(s), None if s2 is None else L.ptr(s2),
                                                 L.ptr(a), L.ptr(r), L.ptr(d), L.ptr(e)))

    def digest(self, n_live: int, id_lo: int = 0, id_hi: int = 0) -> list:
        """idqn_replay_digest: six digests computed on the device (see include/idqn_b200.h)."""
        out = np.zeros(6, np.uint64)
        L.check(self.lib.idqn_replay_digest(self.h, int(n_live), int(id_lo), int(id_hi), L.ptr(out)))
        return [int(x) for x in out]


class _DeviceStore(_Store):
    """Fixed-slot element store in HBM."""

    def __init__(self, n_slots: int, obs_shape, obs_dtype, device: int):
        self.lib = L.lib()
        self.shape, self.dtype = tuple(obs_shape), np.dtype(obs_dtype)
        self.state_bytes = int(np.prod(self.shape)) * self.dtype.itemsize
        self.n_slots, self.device = int(n_slots), int(device)
        h = C.c_void_p()
        L.check(self.lib.idqn_replay_create(self.n_slots, self.state_bytes, self.device, C.byref(h)))
        self.h = h
        self._finalizer = weakref.finalize(self, self.lib.idqn_replay_destroy, h)

    def put(self, slot: int, el: ReplayElement) -> None:
        s = np.ascontiguousarray(el.state, dtype=self.dtype)
        s2 = np.ascontiguousarray(el.next_state, dtype=self.dtype)
        if s.shape != self.shape or s2.shape != self.shape:
            raise ValueError(f"element shape {s.shape} differs from the store's {self.shape}")
        L.check(self.lib.idqn_replay_put(self.h, int(slot), L.ptr(s), L.ptr(s2), int(el.action), float(el.reward),
                                         int(bool(el.is_terminal)), int(bool(el.episode_end))))

    def _slot_stacks(self, n: int):
        return np.empty((n,) + self.shape, self.dtype), np.empty((n,) + self.shape, self.dtype)


class _FrameStore(_Store):
    """Frame store in HBM (idqn_replay_create_frames): a ring of ``n_frames`` observations (frame id ``f`` in ring slot
    ``f % n_frames``) and, per element slot, ``2 * stack`` frame ids (-1: a zero frame)."""

    def __init__(self, n_slots: int, frame_shape, frame_dtype, stack: int, n_frames: int, device: int):
        self.lib = L.lib()
        self.frame_shape, self.dtype, self.stack = tuple(frame_shape), np.dtype(frame_dtype), int(stack)
        self.shape = self.frame_shape + (self.stack,)  # of a stack, as _DeviceStore.shape
        self.frame_bytes = int(np.prod(self.frame_shape)) * self.dtype.itemsize
        self.n_slots, self.device, self._n_frames = int(n_slots), int(device), int(n_frames)
        h = C.c_void_p()
        L.check(self.lib.idqn_replay_create_frames(self.n_slots, self.frame_bytes, self.stack, self.dtype.itemsize,
                                                   self._n_frames, self.device, C.byref(h)))
        self.h = h
        self._finalizer = weakref.finalize(self, self.lib.idqn_replay_destroy, h)

    @property
    def n_frames(self) -> int:
        return self._n_frames

    def put_frame(self, frame_id: int, frame) -> None:
        f = np.ascontiguousarray(frame, dtype=self.dtype)
        if f.shape != self.frame_shape:
            raise ValueError(f"observation shape {f.shape} differs from the store's {self.frame_shape}")
        L.check(self.lib.idqn_replay_put_frame(self.h, int(frame_id), L.ptr(f)))

    def put_element(self, slot: int, frame_ids, action, reward, is_terminal, episode_end) -> None:
        ids = np.ascontiguousarray(frame_ids, dtype=np.int64)
        L.check(self.lib.idqn_replay_put_element(self.h, int(slot), L.ptr(ids), int(action), float(reward),
                                                 int(bool(is_terminal)), int(bool(episode_end))))

    def grow(self, n_frames: int, live_lo: int, live_hi: int) -> None:
        L.check(self.lib.idqn_replay_grow_frames(self.h, int(n_frames), int(live_lo), int(live_hi)))
        self._n_frames = int(n_frames)

    def _slot_stacks(self, n: int):
        return np.empty((n, 2 * self.stack), np.int64), None

    def read_frames(self, id_lo: int, id_hi: int) -> np.ndarray:
        """frames of ids [id_lo, id_hi) in id order"""
        out = np.empty((id_hi - id_lo,) + self.frame_shape, self.dtype)
        L.check(self.lib.idqn_replay_read_frames(self.h, int(id_lo), int(id_hi), L.ptr(out)))
        return out

    def write_frames(self, id_lo: int, frames) -> None:
        f = np.ascontiguousarray(frames, dtype=self.dtype)
        if f.shape[1:] != self.frame_shape:
            raise ValueError(f"frame shape {f.shape[1:]} differs from the store's {self.frame_shape}")
        L.check(self.lib.idqn_replay_write_frames(self.h, int(id_lo), int(id_lo) + len(f), L.ptr(f)))


class _MemoryView(collections.abc.Mapping):
    """``rb._memory`` of the reference (an OrderedDict key -> ReplayElement) as a read-only view of the
    device store: live keys in insertion order, elements fetched on access."""

    def __init__(self, rb: "ReplayBuffer"):
        self._rb = rb

    def _range(self) -> range:
        rb = self._rb
        return range(max(0, rb.add_count - rb._max_capacity), rb.add_count)

    def __len__(self) -> int:
        return len(self._range())

    def __iter__(self) -> Iterator[int]:
        return iter(self._range())

    def __contains__(self, key) -> bool:
        return isinstance(key, (int, np.integer)) and int(key) in self._range()

    def __getitem__(self, key) -> ReplayElement:
        if key not in self:
            raise KeyError(key)
        s, s2, a, r, d, e = self._rb._store.gather(np.asarray([int(key) % self._rb._max_capacity]))
        return ReplayElement(s[0], int(a[0]), float(r[0]), s2[0], bool(d[0]), bool(e[0]))


class ReplayBuffer:
    def __init__(
        self,
        sampling_distribution,
        batch_size: int,
        max_capacity: int,
        stack_size: int = 4,
        update_horizon: int = 1,
        gamma: float = 0.99,
        checkpoint_duration: int = 4,
        compress: bool = True,
        clipping: callable = None,
        *,
        device: int = 0,
        frame_store: bool = False,
        n_envs: int = 1,
    ):
        if int(n_envs) != n_envs or n_envs < 1:
            raise ValueError(f"n_envs must be a positive integer, got {n_envs!r}")
        self.add_count = 0
        self._max_capacity = max_capacity
        self._compress = compress  # accepted for signature parity; HBM slots hold raw bytes
        self._sampling_distribution = sampling_distribution
        self._checkpoint_duration = checkpoint_duration
        self._batch_size = batch_size
        self._stack_size = stack_size
        self._update_horizon = update_horizon
        self._gamma = gamma
        self._clipping = clipping
        self._device = device
        self._store: Optional[_DeviceStore] = None
        self._memory = _MemoryView(self)
        # one n-step / frame-stack accumulator per environment (``add(..., env=i)``); ``_trajectory`` is environment 0's
        self._n_envs = int(n_envs)
        self._trajectories: "list[collections.deque[TransitionElement]]" = [
            collections.deque(maxlen=self._update_horizon + self._stack_size) for _ in range(self._n_envs)]
        self._trajectory = self._trajectories[0]
        self._frame_store = frame_store
        if frame_store:
            # frame id of each trajectory entry once an emitted element has referred to it (None before), per environment
            self._env_frame_ids: "list[collections.deque[Optional[int]]]" = [
                collections.deque(maxlen=self._trajectory.maxlen) for _ in range(self._n_envs)]
            self._frame_ids = self._env_frame_ids[0]
            self._next_frame_id = 0
            # (key, smallest frame id) of live elements with that id increasing: the front is the smallest of all
            self._live_min: "collections.deque[tuple[int, int]]" = collections.deque()

    # ---- n-step / frame-stack accumulator (replay_buffer.py:103-200) ---------------------------------
    def _window(self, env: int = 0) -> Optional[tuple[int, list[int]]]:
        """The element environment ``env``'s trajectory emits now, as (pivot, trajectory index of each of the 2 * stack
        stack positions: state, then next_state; -1 = zero), or None."""
        traj, n, stack = self._trajectories[env], self._update_horizon, self._stack_size
        length = len(traj)
        newest = traj[-1]
        if not (length > n or (length > 1 and newest.is_terminal)):
            return None
        # a terminal cuts the n-step window short when the trajectory is still shorter than n (:116-118)
        horizon = length - 1 if (newest.is_terminal and length <= n) else n
        pivot = length - horizon - 1  # newest frame of the state stack; its action is the element's action
        # missing history stays zero (:125,136)
        state = [max(pivot - (stack - 1) + pos, -1) for pos in range(stack)]
        next_state = [max(length - stack + pos, -1) for pos in range(stack)]
        return pivot, state + next_state

    def _scalars(self, pivot: int, env: int = 0) -> tuple[Any, float, bool]:
        traj, n = self._trajectories[env], self._update_horizon
        ret = 0.0
        for t in range(pivot, min(pivot + n, len(traj))):  # discounted n-step return (:153-165)
            ret += traj[t].reward * (self._gamma ** (t - pivot))
        return traj[pivot].action, ret, traj[-1].is_terminal

    def _make_replay_element(self, window, env: int = 0) -> ReplayElement:
        pivot, positions = window
        traj, stack = self._trajectories[env], self._stack_size
        frame = np.asarray(traj[-1].observation)
        state = np.zeros(frame.shape + (stack,), frame.dtype)
        next_state = np.zeros(frame.shape + (stack,), frame.dtype)
        for pos in range(stack):
            t_state, t_next = positions[pos], positions[stack + pos]
            if t_state >= 0:
                state[..., pos] = traj[t_state].observation
            if t_next >= 0:
                next_state[..., pos] = traj[t_next].observation
        action, ret, terminal = self._scalars(pivot, env)
        return ReplayElement(state=state, action=action, reward=ret, next_state=next_state, is_terminal=terminal,
                             episode_end=terminal)

    def _windows(self, transition: TransitionElement, env: int = 0) -> Iterator[tuple[int, list[int]]]:
        traj = self._trajectories[env]
        traj.append(transition)
        if self._frame_store:
            self._env_frame_ids[env].append(None)
        if transition.is_terminal:  # drain: one element per remaining start frame (:189-194)
            while (window := self._window(env)) is not None:
                yield window
                traj.popleft()
                if self._frame_store:
                    self._env_frame_ids[env].popleft()
            self._clear_trajectory(env)
        else:
            if (window := self._window(env)) is not None:
                yield window
            if transition.episode_end:  # truncation (:199-200)
                self._clear_trajectory(env)

    def _clear_trajectory(self, env: int = 0) -> None:
        self._trajectories[env].clear()
        if self._frame_store:
            self._env_frame_ids[env].clear()

    def _check_env(self, env) -> int:
        if not isinstance(env, (int, np.integer)) or not 0 <= env < self._n_envs:
            raise ValueError(f"env={env!r} is not one of this buffer's {self._n_envs} environments")
        return int(env)

    def accumulate(self, transition: TransitionElement, env: int = 0) -> Iterable[ReplayElement]:
        env = self._check_env(env)
        for window in self._windows(transition, env):
            yield self._make_replay_element(window, env)

    # ---- frame store bookkeeping ----------------------------------------------------------------------
    # Invariant: every frame id a live element or the trajectory refers to lies in [next id - n_frames, next id), so
    # writing id f into ring slot f % n_frames never overwrites a frame still in use.  An id leaves that set for good
    # (the trajectory only drops entries, elements are evicted in FIFO order), so its smallest member never decreases.
    # With several environments the set holds every environment's trajectory ids; a newly assigned id is still the
    # largest of all, so the argument holds.  An environment that is never stepped again keeps its trajectory's frames
    # in use for good: the ring grows to hold them next to everything written after them.
    _frame_store_type = _FrameStore  # anything with put_frame / put_element / grow / n_frames (a host model in tests)

    def _open_frame_store(self, frame: np.ndarray) -> _FrameStore:
        cap, stack = self._max_capacity, self._stack_size
        n_frames = cap + cap // 64 + stack + self._update_horizon
        return self._frame_store_type(cap, frame.shape, frame.dtype, stack, n_frames, self._device)

    def _lowest_frame_in_use(self) -> int:
        ids = [f for frame_ids in self._env_frame_ids for f in frame_ids if f is not None]
        if self._live_min:
            ids.append(self._live_min[0][1])
        return min(ids, default=self._next_frame_id)

    def _new_frame_id(self, observation) -> int:
        store, f = self._store, self._next_frame_id
        lo = self._lowest_frame_in_use()
        if f - lo >= store.n_frames:  # many short episodes: more frames in use than the ring holds
            n_frames = store.n_frames
            while f - lo >= n_frames:
                n_frames = (5 * n_frames + 3) // 4  # ceil(1.25 n)
            store.grow(n_frames, lo, f)
        store.put_frame(f, observation)
        self._next_frame_id = f + 1
        return f

    def _add_frames(self, key: int, window, env: int = 0) -> None:
        pivot, positions = window
        traj, frame_ids = self._trajectories[env], self._env_frame_ids[env]
        while self._live_min and self._live_min[0][0] <= key - self._max_capacity:  # the element `key` replaces
            self._live_min.popleft()
        for t in sorted({t for t in positions if t >= 0}):  # ids in trajectory order, on first use
            if frame_ids[t] is None:
                frame_ids[t] = self._new_frame_id(traj[t].observation)
        ids = [frame_ids[t] if t >= 0 else -1 for t in positions]
        action, ret, terminal = self._scalars(pivot, env)
        self._store.put_element(key % self._max_capacity, ids, action, ret, terminal, terminal)
        smallest = min(f for f in ids if f >= 0)
        while self._live_min and self._live_min[-1][1] >= smallest:
            self._live_min.pop()
        self._live_min.append((key, smallest))

    # ---- add / sample / update (replay_buffer.py:202-237) -----------------------------------------------
    def add(self, transition: TransitionElement, *, env: int = 0, **kwargs: Any) -> None:
        """Add a transition of environment ``env`` (one of ``n_envs``); elements get keys in the order they are emitted,
        whichever environment emits them.  ``kwargs`` go to the sampler."""
        env = self._check_env(env)
        for window in self._windows(transition, env):
            key = ReplayItemID(self.add_count)
            if self._frame_store:
                if self._store is None:
                    self._store = self._open_frame_store(np.asarray(transition.observation))
                self._add_frames(key, window, env)
            else:
                element = self._make_replay_element(window, env)
                if self._store is None:
                    self._store = _DeviceStore(self._max_capacity, np.shape(element.state),
                                               np.asarray(element.state).dtype, self._device)
                self._store.put(key % self._max_capacity, element)
            self._sampling_distribution.add(key, **kwargs)
            self.add_count += 1
            if self.add_count > self._max_capacity:
                self._sampling_distribution.remove(ReplayItemID(self.add_count - self._max_capacity - 1))

    def sample(self, size=None) -> ReplayElement:
        assert self.add_count, ValueError("No samples in replay buffer!")
        if size is None:
            size = self._batch_size
        keys = self._sampling_distribution.sample(size)
        self.last_keys = keys
        s, s2, a, r, d, e = self._store.gather(np.asarray(keys, np.int64) % self._max_capacity)
        return ReplayElement(state=s, action=a, reward=r, next_state=s2, is_terminal=d, episode_end=e)

    def learn_step_on(self, engine, want_losses: bool = False):
        """``update_online_params`` fast path (idqn.py:65-72): sample keys, gather on the device into the
        learner's staging and run the step — no batch ever visits the host.  Returns False when this buffer
        cannot feed ``engine`` directly (different device / element layout)."""
        st = self._store
        assert self.add_count, ValueError("No samples in replay buffer!")
        if st is None or st.device != engine.device or self._batch_size != engine.B:
            return False
        u8 = st.dtype == np.uint8
        if not (u8 or st.dtype == np.float32) or int(np.prod(st.shape)) != engine.in_elems:
            return False
        keys = self._sampling_distribution.sample(self._batch_size)
        slots = np.ascontiguousarray(np.asarray(keys, np.int64) % self._max_capacity)
        losses = np.zeros(engine.K, np.float32) if want_losses else None
        L.check(st.lib.idqn_learn_from_replay(engine.h, st.h, L.ptr(slots), len(slots), int(u8),
                                              L.ptr(losses) if want_losses else None))
        self.last_keys = keys
        return losses if want_losses else True

    def update(self, keys, **kwargs: Any) -> None:
        self._sampling_distribution.update(keys, **kwargs)

    def update_from_learner(self, engine) -> None:
        """``update(last sampled keys, priorities = |TD error| of the step that just consumed them)`` with the priorities
        taken from the learner on the device (replay_buffer.py:232-237 wired to the learning step)."""
        upd = getattr(self._sampling_distribution, "update_from_learner", None)
        if upd is None:
            raise TypeError("update_from_learner needs a PrioritizedSamplingDistribution")
        upd(self.last_keys, engine)

    # ---- checkpoint -----------------------------------------------------------------------------------------------
    # Dopamine's save/load (the origin of ``checkpoint_duration``, replay_buffer.py:82,93 of the reference, which never
    # uses it) for the device store: the accumulator, the frame bookkeeping, the live part of the store streamed in
    # chunks, the sampler and the device-computed digests the load checks what landed in HBM against.
    _DIGESTS = ("state/frames", "next_state/rows", "action", "reward", "terminal", "episode_end")

    def _config(self) -> dict:
        config = {"max_capacity": int(self._max_capacity), "stack_size": int(self._stack_size),
                  "update_horizon": int(self._update_horizon), "gamma": float(self._gamma),
                  "batch_size": int(self._batch_size), "frame_store": bool(self._frame_store),
                  "sampler": type(self._sampling_distribution).__name__}
        if self._n_envs != 1:  # a checkpoint without the key is of one environment
            config["n_envs"] = self._n_envs
        return config

    @staticmethod
    def _trajectory_file(env: int, field: str) -> str:
        return f"trajectory_{field}.npy" if env == 0 else f"trajectory{env}_{field}.npy"

    def _slot_files(self):
        return ("rows" if self._frame_store else "state", "next_state", "action", "reward", "terminal", "episode_end")

    def save(self, directory: str) -> None:
        """Write this buffer into ``directory`` (created if missing).  Waits for learner steps still reading the store."""
        os.makedirs(directory, exist_ok=True)
        join = lambda name: os.path.join(directory, name)
        meta = {"config": self._config(), "add_count": int(self.add_count), "trajectory": len(self._trajectory),
                "store": None}
        if self._n_envs != 1:  # environment i's accumulator in trajectory{i}_*.npy (environment 0's as with one)
            meta["trajectories"] = [len(t) for t in self._trajectories]
        for env, traj in enumerate(self._trajectories):
            if traj:
                name = lambda field: join(self._trajectory_file(env, field))
                np.save(name("observation"), np.stack([np.asarray(t.observation) for t in traj]))
                np.save(name("action"), np.asarray([int(t.action) for t in traj], np.int64))
                np.save(name("reward"), np.asarray([float(t.reward) for t in traj], np.float64))
                np.save(name("flags"),
                        np.asarray([(bool(t.is_terminal), bool(t.episode_end)) for t in traj], np.uint8).reshape(-1, 2))
        if self._frame_store:
            meta["frame_ids"] = [-1 if f is None else int(f) for f in self._frame_ids]
            if self._n_envs != 1:
                meta["env_frame_ids"] = [[-1 if f is None else int(f) for f in ids] for ids in self._env_frame_ids]
            meta["next_frame_id"] = int(self._next_frame_id)
            meta["live_min"] = [[int(k), int(f)] for k, f in self._live_min]
        st = self._store
        if st is not None:
            n_live = min(self.add_count, self._max_capacity)
            lo, hi = (self._lowest_frame_in_use(), self._next_frame_id) if self._frame_store else (0, 0)
            meta["store"] = {"shape": list(st.frame_shape if self._frame_store else st.shape), "dtype": st.dtype.str,
                             "n_frames": int(st.n_frames) if self._frame_store else None, "n_live": n_live,
                             "frames": [lo, hi], "digest": st.digest(n_live, lo, hi)}
            if self._frame_store:
                per = ckpt.rows_per_chunk(st.frame_bytes)
                w = ckpt.NpyWriter(join("frames.npy"), (hi - lo,) + st.frame_shape, st.dtype)
                for f in range(lo, hi, per):
                    w.write(st.read_frames(f, min(f + per, hi)))
                w.close()
            writers = []
            per = ckpt.rows_per_chunk(16 * self._stack_size + 14 if self._frame_store else 2 * st.state_bytes + 14)
            for k in range(0, n_live, per):
                arrays = st.read_slots(k, min(per, n_live - k))
                if not writers:
                    writers = [None if a is None else ckpt.NpyWriter(join(name + ".npy"), (n_live,) + a.shape[1:], a.dtype)
                               for name, a in zip(self._slot_files(), arrays)]
                for wr, a in zip(writers, arrays):
                    if wr is not None:
                        wr.write(a)
            for wr in writers:
                if wr is not None:
                    wr.close()
        if getattr(self, "last_keys", None) is not None:
            np.save(join("last_keys.npy"), np.asarray(self.last_keys))
        if hasattr(self._sampling_distribution, "save"):
            self._sampling_distribution.save(join("sampler"))
        ckpt.write_json(join("replay.json"), meta)

    def load(self, directory: str) -> None:
        """Restore a buffer written by ``save`` into this one, which must have been just constructed with the same
        configuration (ValueError otherwise).  The store is re-created at its saved size and its contents are checked
        against the saved digests on the device (ValueError on a mismatch; the buffer is then unusable)."""
        join = lambda name: os.path.join(directory, name)
        meta = ckpt.read_json(join("replay.json"))
        if self.add_count != 0 or self._store is not None or any(self._trajectories):
            raise ValueError("ReplayBuffer.load needs a buffer nothing has been added to")
        saved = {"n_envs": 1, **meta["config"]}
        for k, v in {"n_envs": 1, **self._config()}.items():
            if saved[k] != v:
                raise ValueError(f"replay checkpoint has {k}={saved[k]!r}, this buffer {v!r}")
        for env, length in enumerate(meta.get("trajectories", [meta["trajectory"]])):
            if length:
                name = lambda field: join(self._trajectory_file(env, field))
                obs, act, rew = np.load(name("observation")), np.load(name("action")), np.load(name("reward"))
                flags = np.load(name("flags"))
                for t in range(length):
                    self._trajectories[env].append(TransitionElement(obs[t], int(act[t]), float(rew[t]),
                                                                     bool(flags[t, 0]), bool(flags[t, 1])))
        if self._frame_store:
            for ids, saved_ids in zip(self._env_frame_ids, meta.get("env_frame_ids", [meta["frame_ids"]])):
                ids.extend(None if f < 0 else f for f in saved_ids)
            self._next_frame_id = meta["next_frame_id"]
            self._live_min.extend((k, f) for k, f in meta["live_min"])
        sm = meta["store"]
        if sm is not None:
            shape, dtype, n_live = tuple(sm["shape"]), np.dtype(sm["dtype"]), sm["n_live"]
            lo, hi = sm["frames"]
            if self._frame_store:
                st = self._store = self._frame_store_type(self._max_capacity, shape, dtype, self._stack_size,
                                                          sm["n_frames"], self._device)
                rd = ckpt.NpyReader(join("frames.npy"))
                per = ckpt.rows_per_chunk(st.frame_bytes)
                for f in range(lo, hi, per):
                    st.write_frames(f, rd.read(min(per, hi - f)))
                rd.close()
            else:
                st = self._store = _DeviceStore(self._max_capacity, shape, dtype, self._device)
            readers = [ckpt.NpyReader(join(n + ".npy")) if n != "next_state" or not self._frame_store else None
                       for n in self._slot_files()]
            per = ckpt.rows_per_chunk(16 * self._stack_size + 14 if self._frame_store else 2 * st.state_bytes + 14)
            for k in range(0, n_live, per):
                m = min(per, n_live - k)
                st.write_slots(k, *[None if rd is None else rd.read(m) for rd in readers])
            for rd in readers:
                if rd is not None:
                    rd.close()
            got = st.digest(n_live, lo, hi)
            bad = [n for n, a, b in zip(self._DIGESTS, got, sm["digest"]) if a != b]
            if bad:
                raise ValueError(f"replay digest mismatch in {', '.join(bad)}: {directory} does not hold the saved store")
        self.add_count = meta["add_count"]
        if os.path.exists(join("last_keys.npy")):
            self.last_keys = np.load(join("last_keys.npy"))
        if hasattr(self._sampling_distribution, "load"):
            self._sampling_distribution.load(join("sampler"))
