"""Host bookkeeping of ReplayBuffer(frame_store=True) over a NumPy model of the device frame ring (no GPU): every live
element's stacks rebuilt from the ring equal what the element store keeps, the ring never overwrites a frame still in
use, and the ring grows when many short episodes need more frames than it holds."""
import os

import numpy as np
import pytest


class NumpyFrames:
    """The device frame store's contract: frame id f in ring slot f % n_frames, rows of frame ids (-1 = zeros)."""

    def __init__(self, n_slots, frame_shape, dtype, stack, n_frames, device):
        self.frame_shape, self.stack = tuple(frame_shape), stack
        self.ring = np.zeros((n_frames,) + self.frame_shape, dtype)
        self.rows = np.full((n_slots, 2 * stack), -1, np.int64)
        self.scalars = [None] * n_slots
        self.frame_puts, self.grows = [], 0

    @property
    def n_frames(self):
        return len(self.ring)

    def put_frame(self, frame_id, frame):
        self.ring[frame_id % self.n_frames] = frame
        self.frame_puts.append(frame_id)

    def put_element(self, slot, frame_ids, action, reward, is_terminal, episode_end):
        assert len(frame_ids) == 2 * self.stack
        self.rows[slot] = frame_ids
        self.scalars[slot] = (action, reward, is_terminal, episode_end)

    def grow(self, n_frames, live_lo, live_hi):
        assert n_frames > self.n_frames and 0 <= live_hi - live_lo <= self.n_frames
        ring = np.zeros((n_frames,) + self.frame_shape, self.ring.dtype)
        for f in range(live_lo, live_hi):  # re-home the live ids
            ring[f % n_frames] = self.ring[f % self.n_frames]
        self.ring = ring
        self.grows += 1

    def stacks(self, slot):
        out = np.zeros((2,) + self.frame_shape + (self.stack,), self.ring.dtype)
        for i, f in enumerate(self.rows[slot]):
            if f >= 0:
                out[i // self.stack][..., i % self.stack] = self.ring[f % self.n_frames]
        return out[0], out[1]


class KeysOnly:
    def add(self, key, **kwargs):
        pass

    def remove(self, key):
        pass


def make_buffers(stack, n, gamma, cap):
    from idqn_b200.sample_collection.replay_buffer import ReplayBuffer

    class HostFrameBuffer(ReplayBuffer):
        _frame_store_type = NumpyFrames

    rb = HostFrameBuffer(KeysOnly(), 8, cap, stack, n, gamma, compress=False, frame_store=True)
    ref = ReplayBuffer(None, 8, cap, stack, n, gamma, compress=False)  # element mode: the same elements, whole
    return rb, ref


def drive(rb, ref, transitions):
    """add every transition; after each add check the invariant and every live element against the element mode"""
    emitted, lowest = [], []
    for tr in transitions:
        emitted.extend(ref.accumulate(tr))
        rb.add(tr)
        assert rb.add_count == len(emitted)
        st = rb._store
        if st is None:
            continue
        hi, F = rb._next_frame_id, st.n_frames
        live = range(max(0, rb.add_count - rb._max_capacity), rb.add_count)
        in_use = [f for k in live for f in st.rows[k % rb._max_capacity] if f >= 0]
        in_use += [f for f in rb._frame_ids if f is not None]
        assert all(hi - F <= f < hi for f in in_use), (hi, F, min(in_use))
        lowest.append(rb._lowest_frame_in_use())
        for k in live:
            s, s2 = st.stacks(k % rb._max_capacity)
            e = emitted[k]
            np.testing.assert_array_equal(s, e.state)
            np.testing.assert_array_equal(s2, e.next_state)
            a, r, d, end = st.scalars[k % rb._max_capacity]
            assert a == e.action and np.float64(r).tobytes() == np.float64(e.reward).tobytes()
            assert d == e.is_terminal and end == e.episode_end
    st = rb._store
    assert st.frame_puts == list(range(len(st.frame_puts))), "frame ids are handed out in increasing order"
    assert all(a <= b for a, b in zip(lowest, lowest[1:])), "the lowest frame id in use never decreases"
    return emitted


@pytest.mark.parametrize("ci", [0, 1, 2, 3])
def test_frame_bookkeeping_rebuilds_the_golden_elements(golden_dir, ci):
    from idqn_b200.sample_collection.replay_buffer import TransitionElement
    g = np.load(os.path.join(golden_dir, "replay_buffer.npz"))
    p = f"cfg{ci}_"
    stack, n, gamma, cap = g[p + "cfg"]
    rb, ref = make_buffers(int(stack), int(n), float(gamma), int(cap))
    drive(rb, ref, [TransitionElement(g[p + "obs"][t], int(g[p + "act"][t]), float(g[p + "rew"][t]),
                                      bool(g[p + "term"][t]), bool(g[p + "trunc"][t]))
                    for t in range(g[p + "obs"].shape[0])])
    keys = list(rb._memory.keys())
    np.testing.assert_array_equal(keys, g[p + "keys"])
    assert rb.add_count == int(g[p + "add_count"])
    st = rb._store
    stacks = [st.stacks(k % rb._max_capacity) for k in keys]
    np.testing.assert_array_equal(np.stack([s for s, _ in stacks]), g[p + "state"])
    np.testing.assert_array_equal(np.stack([s2 for _, s2 in stacks]), g[p + "next_state"])
    assert np.asarray([st.scalars[k % rb._max_capacity][1] for k in keys]).tobytes() == g[p + "reward"].tobytes()


@pytest.mark.parametrize("stack,n", [(4, 1), (1, 3), (2, 2)])
def test_short_episodes_grow_the_ring(stack, n):
    """capacity 8, two-step episodes ending alternately in a terminal and a truncation: more frames per element than
    the initial ring holds"""
    from idqn_b200.sample_collection.replay_buffer import TransitionElement
    rng = np.random.default_rng(stack * 10 + n)
    rb, ref = make_buffers(stack, n, 0.9, 8)
    trs = []
    for t in range(80):
        end = t % 2 == 1
        term = end and t % 4 == 1
        trs.append(TransitionElement(rng.integers(0, 256, (3, 2)).astype(np.uint8), int(rng.integers(0, 6)),
                                     float(rng.integers(-1, 2)), term, end))
    drive(rb, ref, trs)
    assert rb._store.grows >= 1
    assert rb._store.n_frames > 8 + stack + n


def test_long_n_step_window_keeps_frames_the_trajectory_still_needs():
    """stack 1, n = 3: an element's state frame is given its id after the next_state frames of earlier elements, so the
    smallest id of consecutive elements goes down; the frames stay in the ring while the trajectory holds them"""
    from idqn_b200.sample_collection.replay_buffer import TransitionElement
    rng = np.random.default_rng(5)
    rb, ref = make_buffers(1, 3, 0.99, 2)
    drive(rb, ref, [TransitionElement(rng.integers(0, 256, (3, 2)).astype(np.uint8), 1, 1.0, t % 37 == 36, False)
                    for t in range(120)])
