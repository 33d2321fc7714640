"""ReplayBuffer(n_envs=N) without a GPU: transitions of N interleaved episodes give exactly the elements of N separate
reference buffers merged in emission order, in the element store and over the NumPy model of the frame ring (with
growth), checkpoints cover every environment's accumulator, and ``select_actions`` on the plain-function path equals
``select_action`` per environment."""
import json
import os

import numpy as np
import pytest

from oracle.replay_buffer import ReplayBufferOracle, Transition
from test_checkpoint_host import NumpyFramesIO
from test_frame_store_host import KeysOnly


class HostElements:
    """The element store's contract (_DeviceStore.put) kept in host memory."""

    def __init__(self, n_slots, shape, dtype, device):
        self.shape, self.dtype = tuple(shape), np.dtype(dtype)
        self.slots = [None] * n_slots

    def put(self, slot, el):
        self.slots[slot] = el


def interleaved(seed, n_envs, steps, max_len=9, frame_shape=(3, 2)):
    """(env, transition) pairs: each environment runs its own episodes of random lengths ending in a terminal or a
    truncation, and the environment stepped next is drawn at random"""
    from idqn_b200.sample_collection.replay_buffer import TransitionElement
    rng = np.random.default_rng(seed)
    left = [int(rng.integers(1, max_len + 1)) for _ in range(n_envs)]
    out = []
    for _ in range(steps):
        i = int(rng.integers(0, n_envs))
        left[i] -= 1
        end = left[i] == 0
        term = end and bool(rng.integers(0, 2))
        out.append((i, TransitionElement(rng.integers(0, 256, frame_shape).astype(np.uint8), int(rng.integers(0, 6)),
                                         float(rng.integers(-1, 2)), term, end)))
        if end:
            left[i] = int(rng.integers(1, max_len + 1))
    return out


def oracle_merge(drive, n_envs, stack, n, gamma):
    """elements of one reference buffer per environment, in the order the transitions emit them"""
    refs = [ReplayBufferOracle(None, 8, 10 ** 6, stack, n, gamma) for _ in range(n_envs)]
    merged = []
    for i, tr in drive:
        merged.extend(refs[i]._emit(Transition(tr.observation, tr.action, tr.reward, tr.is_terminal, tr.episode_end)))
    return merged


def assert_element(state, next_state, scalars, e):
    np.testing.assert_array_equal(state, e["state"])
    np.testing.assert_array_equal(next_state, e["next_state"])
    a, r, d, end = scalars
    assert a == e["action"] and np.float64(r).tobytes() == np.float64(e["reward"]).tobytes()
    assert bool(d) == e["is_terminal"] and bool(end) == e["episode_end"]


@pytest.mark.parametrize("n", [1, 3, 5])
@pytest.mark.parametrize("cap", [1000, 16])
def test_element_store_equals_merged_reference_buffers(monkeypatch, n, cap):
    from idqn_b200.sample_collection import replay_buffer as R
    monkeypatch.setattr(R, "_DeviceStore", HostElements)
    stack, gamma = 4, 0.9
    drive = interleaved(n * 7 + cap, 3, 400)
    merged = oracle_merge(drive, 3, stack, n, gamma)
    rb = R.ReplayBuffer(KeysOnly(), 8, cap, stack, n, gamma, compress=False, n_envs=3)
    for i, tr in drive:
        rb.add(tr, env=i)
    assert rb.add_count == len(merged) > 150
    assert len(rb._memory) == min(cap, len(merged))
    for k in rb._memory:
        el = rb._store.slots[k % cap]
        assert_element(el.state, el.next_state, (el.action, el.reward, el.is_terminal, el.episode_end), merged[k])


def frame_buffer(n_envs, stack, n, cap, gamma=0.9):
    from idqn_b200.sample_collection.replay_buffer import ReplayBuffer

    class HostFrameBuffer(ReplayBuffer):
        _frame_store_type = NumpyFramesIO

    return HostFrameBuffer(KeysOnly(), 8, cap, stack, n, gamma, compress=False, frame_store=True, n_envs=n_envs)


def check_frames(rb, merged):
    """every frame id in use lies in the ring's window and every live element is rebuilt exactly"""
    st = rb._store
    hi, F = rb._next_frame_id, st.n_frames
    live = range(max(0, rb.add_count - rb._max_capacity), rb.add_count)
    in_use = [f for k in live for f in st.rows[k % rb._max_capacity] if f >= 0]
    in_use += [f for ids in rb._env_frame_ids for f in ids if f is not None]
    assert all(hi - F <= f < hi for f in in_use)
    assert rb._lowest_frame_in_use() == min(in_use, default=hi)
    for k in live:
        s, s2 = st.stacks(k % rb._max_capacity)
        assert_element(s, s2, st.scalars[k % rb._max_capacity], merged[k])


@pytest.mark.parametrize("n,max_len,cap", [(1, 9, 64), (3, 9, 64), (5, 9, 64), (1, 2, 8), (3, 2, 8)])
def test_frame_store_rebuilds_every_live_element(n, max_len, cap):
    stack, gamma = 4, 0.9
    drive = interleaved(n * 31 + max_len, 3, 500, max_len)
    merged = oracle_merge(drive, 3, stack, n, gamma)
    rb = frame_buffer(3, stack, n, cap, gamma)
    lowest = []
    for i, tr in drive:
        rb.add(tr, env=i)
        if rb._store is not None:
            check_frames(rb, merged)
            lowest.append(rb._lowest_frame_in_use())
    assert rb.add_count == len(merged)
    assert rb._store.frame_puts == list(range(len(rb._store.frame_puts)))
    assert all(a <= b for a, b in zip(lowest, lowest[1:])), "the lowest frame id in use never decreases"
    if max_len <= 2:
        assert rb._store.grows >= 1


def test_idle_environment_pins_its_frames():
    """an environment that stops being stepped keeps its trajectory's frames: the ring grows around them"""
    from idqn_b200.sample_collection.replay_buffer import TransitionElement
    rng = np.random.default_rng(3)
    rb = frame_buffer(2, 2, 1, 8)
    tr = lambda end=False: TransitionElement(rng.integers(0, 256, (3, 2)).astype(np.uint8), 1, 1.0, False, end)
    rb.add(tr(), env=1)
    rb.add(tr(), env=1)  # env 1 emits one element and keeps its two frames in its trajectory
    pinned = [f for f in rb._env_frame_ids[1] if f is not None]
    frames = [rb._store.ring[f % rb._store.n_frames].copy() for f in pinned]
    for t in range(200):
        rb.add(tr(end=t % 5 == 4), env=0)
    assert rb._store.grows >= 1 and rb._lowest_frame_in_use() == min(pinned)
    for f, fr in zip(pinned, frames):
        np.testing.assert_array_equal(rb._store.ring[f % rb._store.n_frames], fr)


def test_env_argument_is_checked():
    from idqn_b200.sample_collection.replay_buffer import ReplayBuffer, TransitionElement
    rb = frame_buffer(3, 4, 1, 8)
    t = TransitionElement(np.zeros((3, 2), np.uint8), 0, 0.0, False)
    for bad in (-1, 3, 1.0):
        with pytest.raises(ValueError, match="env"):
            rb.add(t, env=bad)
    with pytest.raises(ValueError, match="n_envs"):
        ReplayBuffer(KeysOnly(), 8, 8, n_envs=0)


def state_of(rb):
    return (rb.add_count, rb._next_frame_id, [list(ids) for ids in rb._env_frame_ids], list(rb._live_min),
            [[(np.asarray(t.observation).tobytes(), t.action, t.reward, t.is_terminal, t.episode_end) for t in traj]
             for traj in rb._trajectories])


@pytest.mark.parametrize("n", [1, 5])
def test_checkpoint_round_trip_mid_trajectory(tmp_path, n):
    stack, cap = 4, 16
    drive = interleaved(n, 3, 400, 3)
    merged = oracle_merge(drive, 3, stack, n, 0.9)
    a = frame_buffer(3, stack, n, cap)
    cut = 0
    while cut < 250 or sum(len(t) > 0 for t in a._trajectories) < 2:  # saved with several episodes under way
        a.add(drive[cut][1], env=drive[cut][0])
        cut += 1
    assert a._store.grows >= 1
    a.save(str(tmp_path / "rb"))
    meta = json.load(open(tmp_path / "rb" / "replay.json"))
    assert meta["config"]["n_envs"] == 3 and len(meta["env_frame_ids"]) == 3
    b = frame_buffer(3, stack, n, cap)
    b.load(str(tmp_path / "rb"))
    assert state_of(b) == state_of(a)
    for i, tr in drive[cut:]:
        a.add(tr, env=i)
        b.add(tr, env=i)
        assert state_of(b) == state_of(a)
        check_frames(b, merged)
    with pytest.raises(ValueError, match="n_envs"):
        frame_buffer(2, stack, n, cap).load(str(tmp_path / "rb"))
    with pytest.raises(ValueError, match="n_envs"):
        frame_buffer(1, stack, n, cap).load(str(tmp_path / "rb"))


def test_one_environment_checkpoint_is_unchanged(tmp_path):
    """n_envs = 1 writes the files and keys it wrote before environments existed, and loads checkpoints without them"""
    a = frame_buffer(1, 4, 3, 16)
    for i, tr in interleaved(2, 1, 60, 5):
        a.add(tr)
    assert len(a._trajectory) > 0
    a.save(str(tmp_path / "rb"))
    meta = json.load(open(tmp_path / "rb" / "replay.json"))
    assert set(meta) == {"config", "add_count", "trajectory", "store", "frame_ids", "next_frame_id", "live_min"}
    assert set(meta["config"]) == {"max_capacity", "stack_size", "update_horizon", "gamma", "batch_size",
                                   "frame_store", "sampler"}
    assert sorted(os.listdir(tmp_path / "rb")) == sorted(
        ["replay.json", "frames.npy", "rows.npy", "action.npy", "reward.npy", "terminal.npy", "episode_end.npy"]
        + [f"trajectory_{f}.npy" for f in ("observation", "action", "reward", "flags")])
    b = frame_buffer(1, 4, 3, 16)
    b.load(str(tmp_path / "rb"))
    assert state_of(b) == state_of(a) and b._trajectory is b._trajectories[0] and b._frame_ids is b._env_frame_ids[0]
    with pytest.raises(ValueError, match="n_envs"):
        frame_buffer(2, 4, 3, 16).load(str(tmp_path / "rb"))


@pytest.mark.parametrize("epsilon", [0.0, 0.3, 1.0])
def test_select_actions_plain_function_equals_select_action(epsilon):
    from idqn_b200 import _prng
    from idqn_b200.sample_collection.utils import select_action, select_actions
    rng = np.random.default_rng(int(epsilon * 10))
    W = rng.standard_normal((5, 3, 6)).astype(np.float32)

    def best_action(params, state, key=None):  # a head drawn from the key, as iDQN.best_action does
        head = _prng.randint(key, 0, len(params))
        return int(np.argmax(np.asarray(state, np.float32).reshape(-1) @ params[head]))

    states = rng.integers(0, 256, (37, 3)).astype(np.float32)
    keys = _prng.split(np.asarray([7, int(epsilon * 1000)], np.uint32), 37)
    eps = lambda step: epsilon
    got = select_actions(best_action, W, states, keys, 6, eps, 11)
    want = [select_action(best_action, W, s, k, 6, eps, 11) for s, k in zip(states, keys)]
    assert got.shape == (37,) and got.tolist() == want
    with pytest.raises(ValueError):
        select_actions(best_action, W, states[:3], keys[:2], 6, eps, 11)
