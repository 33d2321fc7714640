"""ReplayBuffer(frame_store=True) on the GPU: the frame store gives the element store's samples, elements and learning
steps bit for bit -- through the image kernel, the generic kernels and the float path, across ring growth (graph
re-capture), with steps still in flight while adds reuse the frames they read -- in a fraction of the HBM."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

OBS = (84, 84)


# ---- the replay goldens and the restated reference tests with a frame store --------------------------------------

@pytest.mark.parametrize("ci", [0, 1, 2, 3])
def test_frame_store_replay_golden(golden_dir, ci):
    from idqn_b200.sample_collection import replay_buffer, samplers
    g = np.load(os.path.join(golden_dir, "replay_buffer.npz"))
    p = f"cfg{ci}_"
    stack, n, gamma, cap = g[p + "cfg"]
    rb = replay_buffer.ReplayBuffer(samplers.UniformSamplingDistribution(seed=ci), batch_size=8, max_capacity=int(cap),
                                    stack_size=int(stack), update_horizon=int(n), gamma=float(gamma), compress=False,
                                    frame_store=True)
    bi = 0
    for t in range(g[p + "obs"].shape[0]):
        rb.add(replay_buffer.TransitionElement(g[p + "obs"][t], int(g[p + "act"][t]), float(g[p + "rew"][t]),
                                               bool(g[p + "term"][t]), bool(g[p + "trunc"][t])))
        if rb.add_count and t % 10 == 9:
            b = rb.sample()
            np.testing.assert_array_equal(b.state, g[p + "b_state"][bi])
            np.testing.assert_array_equal(b.next_state, g[p + "b_next_state"][bi])
            np.testing.assert_array_equal(b.action, g[p + "b_action"][bi])
            assert b.reward.tobytes() == g[p + "b_reward"][bi].tobytes()
            np.testing.assert_array_equal(b.is_terminal, g[p + "b_is_terminal"][bi])
            bi += 1
    keys = list(rb._memory.keys())
    np.testing.assert_array_equal(keys, g[p + "keys"])
    assert rb.add_count == int(g[p + "add_count"])
    np.testing.assert_array_equal(np.stack([rb._memory[k].state for k in keys]), g[p + "state"])
    np.testing.assert_array_equal(np.stack([rb._memory[k].next_state for k in keys]), g[p + "next_state"])
    assert np.asarray([rb._memory[k].reward for k in keys]).tobytes() == g[p + "reward"].tobytes()
    assert rb._store.n_frames >= int(cap) + int(cap) // 64 + int(stack) + int(n)


def test_frame_store_ref_add_up_to_capacity():
    """reference tests/test_replay_buffer.py:51-88 (int64 observations: 8-byte values in the stacks)"""
    from idqn_b200.sample_collection import replay_buffer, samplers
    from idqn_b200.sample_collection.replay_buffer import TransitionElement
    capacity, stack = 10, 4
    rb = replay_buffer.ReplayBuffer(samplers.UniformSamplingDistribution(seed=0), batch_size=32, max_capacity=capacity,
                                    stack_size=stack, update_horizon=1, gamma=1.0, compress=False, frame_store=True)
    transitions = []
    for i in range(16):
        transitions.append(TransitionElement(np.full(OBS, i), i, i, False, False))
        rb.add(transitions[-1])
    assert len(rb._memory) == capacity
    assert list(rb._memory.keys()) == list(range(5, 5 + capacity))
    for i in range(5, 5 + capacity):
        el = rb._memory[i]
        np.testing.assert_array_equal(
            el.state, np.array([t.observation for t in transitions[i - stack + 1: i + 1]]).transpose(1, 2, 0))
        np.testing.assert_array_equal(
            el.next_state, np.array([t.observation for t in transitions[i - stack + 2: i + 2]]).transpose(1, 2, 0))
        assert el.action == transitions[i].action and el.reward == transitions[i].reward
        assert el.is_terminal == int(transitions[i].is_terminal) and el.episode_end == int(transitions[i].episode_end)


def test_frame_store_ref_nstep_and_stack_and_key_mappings():
    """reference tests/test_replay_buffer.py:90-136 and :230-299"""
    from idqn_b200.sample_collection import replay_buffer, samplers
    from idqn_b200.sample_collection.replay_buffer import TransitionElement
    mk = lambda cap, stack, n, gamma: replay_buffer.ReplayBuffer(
        samplers.UniformSamplingDistribution(seed=0), batch_size=32, max_capacity=cap, stack_size=stack,
        update_horizon=n, gamma=gamma, compress=False, frame_store=True)
    rb = mk(10, 4, 5, 1.0)
    for i in range(50):
        rb.add(TransitionElement(np.full(OBS, i), 0, 2.0, False))
    for _ in range(10):
        np.testing.assert_array_equal(rb.sample().reward, np.ones(32) * 10.0)
    rb = mk(50, 4, 5, 1.0)
    for i in range(11):
        rb.add(TransitionElement(np.full(OBS, i), 0, 0, False))
    for i in rb._memory:
        assert rb._memory[i].state.shape == OBS + (4,)
    np.testing.assert_array_equal(np.zeros(OBS + (3,)), rb._memory[0].state[:, :, :3])
    state = rb._memory[3].state
    for i in range(4):
        np.testing.assert_array_equal(np.full(OBS, i), state[:, :, i])
    capacity = 10
    rb = mk(capacity, 1, 1, 0.99)
    sampler = rb._sampling_distribution
    for i in range(capacity + 1):
        rb.add(TransitionElement(np.full(OBS, i), i, i, False, False))
    next_key = capacity
    rb.add(TransitionElement(np.full(OBS, next_key + 1), next_key + 1, next_key + 1, False, False))
    assert 0 not in sampler._key_to_index and next_key in sampler._key_to_index
    indices = np.random.default_rng(seed=0).integers(len(sampler._index_to_key), size=32)
    keys = [sampler._index_to_key[i] for i in indices]
    samples = rb.sample()
    for i, key in enumerate(keys):
        np.testing.assert_array_equal(samples.state[i, ...], np.full(OBS, key)[..., None])
        np.testing.assert_array_equal(samples.next_state[i, ...], np.full(OBS, key + 1)[..., None])
        assert samples.action[i] == key and samples.reward[i] == key
        assert samples.is_terminal[i] == 0 and samples.episode_end[i] == 0


def test_frame_store_ref_sampling_with_terminal_in_trajectory():
    """reference tests/test_replay_buffer.py:185-228"""
    from idqn_b200.sample_collection import replay_buffer, samplers
    from idqn_b200.sample_collection.replay_buffer import TransitionElement
    rb = replay_buffer.ReplayBuffer(samplers.UniformSamplingDistribution(seed=0), batch_size=2, max_capacity=10,
                                    stack_size=1, update_horizon=3, gamma=1.0, compress=False, frame_store=True)
    for i in range(rb._max_capacity):
        rb.add(TransitionElement(np.full(OBS, i), action=i * 2, reward=i, is_terminal=i == 3, episode_end=False))
    indices = np.random.default_rng(seed=0).integers(rb.add_count, size=5)
    batch = rb.sample(size=5)
    expected_states = np.array([np.full(OBS + (1,), i) if i < 3 else np.full(OBS + (1,), i + 1) for i in indices])
    np.testing.assert_array_equal(batch.state, expected_states)
    np.testing.assert_array_equal(batch.action, np.array([i * 2 if i < 3 else (i + 1) * 2 for i in indices]))
    np.testing.assert_array_equal(batch.reward, np.array([3, 6, 5, 15, 18, 21, 24])[indices])
    np.testing.assert_array_equal(batch.is_terminal, np.array([1, 1, 1, 0, 0, 0, 0])[indices])


def test_element_writes_into_a_frame_store_are_refused():
    from idqn_b200 import _lib as L
    from idqn_b200.sample_collection.replay_buffer import _FrameStore
    st = _FrameStore(4, (3, 2), np.uint8, 2, 8, 0)
    z = np.zeros((3, 2, 2), np.uint8)
    with pytest.raises(ValueError):
        L.check(st.lib.idqn_replay_put(st.h, 0, L.ptr(z), L.ptr(z), 0, 0.0, 0, 0))
    with pytest.raises(ValueError):
        st.put_element(4, [-1] * 4, 0, 0.0, False, False)  # slot out of range
    with pytest.raises(ValueError):
        st.grow(8, 0, 0)  # not larger


# ---- learning steps: element store vs frame store ------------------------------------------------------------------

def transitions(rng, n, obs, u8, episode):
    """n transitions in episodes of `episode` steps that end alternately in a terminal and a truncation"""
    out = []
    for t in range(n):
        end = t % episode == episode - 1
        term = end and (t // episode) % 2 == 0
        o = rng.integers(0, 256, obs).astype(np.uint8) if u8 else rng.standard_normal(obs).astype(np.float32)
        out.append((o, int(rng.integers(0, 4)), float(rng.integers(-1, 2)), term, end))
    return out


def twin_learners(make_agent, obs, u8, stack, cap, phases, seed=0, prioritized=False, sync_before_add=False):
    """Two agents on two buffers (element store, frame store) fed the same transitions and the same sampler stream.
    phases: [(fill, episode length, steps, adds per step)]: `fill` adds, then `steps` times one update_online_params
    step followed by that many adds.  Returns the agents, the buffers, the keys of every step and the oldest live key
    at every step."""
    from idqn_b200.sample_collection import replay_buffer, samplers
    from idqn_b200.sample_collection.replay_buffer import TransitionElement

    def sampler():
        if prioritized:
            return samplers.PrioritizedSamplingDistribution(seed=11, max_capacity=cap)
        return samplers.UniformSamplingDistribution(seed=seed)

    rbs = [replay_buffer.ReplayBuffer(sampler(), batch_size=32, max_capacity=cap, stack_size=stack, update_horizon=1,
                                      gamma=0.99, clipping=lambda x: np.clip(x, -1, 1), frame_store=fs)
           for fs in (False, True)]
    agents = [make_agent(), make_agent()]
    rng = np.random.default_rng(seed)
    keys, oldest, step = [], [], 1

    def add(trs, n):
        for _ in range(n):
            tr = TransitionElement(*next(trs))
            for rb in rbs:
                if sync_before_add:
                    torch.cuda.synchronize()
                rb.add(tr)

    for fill, episode, steps, per_step in phases:
        trs = iter(transitions(rng, fill + steps * per_step, obs, u8, episode))
        add(trs, fill)
        for _ in range(steps):
            oldest.append(max(0, rbs[1].add_count - cap))
            ks = []
            for ag, rb in zip(agents, rbs):
                assert ag.update_online_params(step, rb) is None
                ks.append(np.asarray(rb.last_keys))
                if prioritized:
                    rb.update_from_learner(ag._engine)
            np.testing.assert_array_equal(ks[0], ks[1], err_msg=f"sampled keys, step {step}")
            keys.append(ks[0])
            for ag in agents:
                ag.update_target_params(step)
            step += 1
            add(trs, per_step)
    torch.cuda.synchronize()
    return agents, rbs, keys, oldest


def assert_same_learners(a, b):
    from idqn_b200 import _lib as L
    for which in (L.ONLINE, L.TARGET, L.MU, L.NU):
        np.testing.assert_array_equal(a._engine.download_arena(which), b._engine.download_arena(which),
                                      err_msg=f"arena {which}")
    np.testing.assert_array_equal(a.cumulated_losses, b.cumulated_losses)
    np.testing.assert_array_equal(a._engine.get_count(), b._engine.get_count())


def cnn_agent(flags=0, K=2):
    from idqn_b200.networks.idqn import iDQN
    return lambda: iDQN(3, OBS + (4,), 4, K, [32, 64, 64, 512], "cnn", 3e-4, 0.99, 1, 1, 5, 3, 1.5e-4, flags=flags)


@pytest.mark.parametrize("no_img", [False, True], ids=["image-kernel", "generic-kernels"])
def test_nature_cnn_steps_are_bit_identical_across_growth(no_img):
    """K=2, uint8 84x84 frames, terminals (zero-padded stacks), FIFO wrap-around; the second phase's two-step
    episodes outgrow the ring between steps, so the captured step graph is re-captured on the new ring"""
    from idqn_b200 import _lib as L
    cap = 100
    agents, rbs, keys, _ = twin_learners(cnn_agent(L.F_NO_IMG if no_img else 0), OBS, True, 4, cap,
                                         [(160, 23, 6, 3), (0, 2, 6, 15)])
    assert rbs[1].add_count > cap, "no wrap-around"
    assert rbs[1]._store.n_frames > cap + cap // 64 + 4 + 1, "no growth"
    assert len(keys) == 12
    assert_same_learners(*agents)


def test_mlp_float_observations_are_bit_identical():
    """K=3 MLP, float32 (8,) observations, stack 1: the frame gather kernel feeds the float path"""
    from idqn_b200.networks.idqn import iDQN
    mk = lambda: iDQN(5, (8,), 4, 3, [100, 100], "fc", 3e-4, 0.99, 1, 1, 5, 3, 1e-8)
    agents, rbs, keys, _ = twin_learners(mk, (8,), False, 1, 60, [(80, 7, 6, 3), (0, 2, 6, 10)])
    assert rbs[1]._store.n_frames > 60 + 0 + 1 + 1, "no growth"
    assert len(keys) == 12
    assert_same_learners(*agents)


def test_prioritized_replay_end_to_end_with_a_frame_store():
    """the scenario of test_prioritized_replay_wired_to_the_learner_end_to_end with a frame store next to an element
    store: the same keys every step, the same tree nodes and max_recorded_priority at the end"""
    agents, rbs, keys, _ = twin_learners(cnn_agent(), OBS, True, 4, 200, [(150, 50, 12, 10)], prioritized=True)
    assert len(keys) == 12
    s0, s1 = rbs[0]._sampling_distribution, rbs[1]._sampling_distribution
    assert s0._sum_tree._nodes.tobytes() == s1._sum_tree._nodes.tobytes()
    assert s0._sum_tree.max_recorded_priority == s1._sum_tree.max_recorded_priority
    np.testing.assert_array_equal(np.asarray(s0._index_to_key), np.asarray(s1._index_to_key))
    assert_same_learners(*agents)


def test_adds_while_steps_are_in_flight_wait_for_them():
    """capacity = batch: the oldest element is sampled in most steps, and the adds right behind the step (enqueued with
    no loss read-back, not synchronised) evict it and reuse its ring slot.  The frame-store learner equals the one of a
    run that synchronises the device before every add."""
    phases = [(40, 1000, 12, 4)]
    free, _, keys, oldest = twin_learners(cnn_agent(), OBS, True, 4, 32, phases)
    assert sum(int(o) in set(k.tolist()) for o, k in zip(oldest, keys)) >= 3, "the oldest element was rarely sampled"
    synced, _, _, _ = twin_learners(cnn_agent(), OBS, True, 4, 32, phases, sync_before_add=True)
    assert_same_learners(free[1], synced[1])
    assert_same_learners(synced[0], synced[1])


def test_frame_store_footprint():
    from idqn_b200.sample_collection.replay_buffer import _DeviceStore, _FrameStore
    n, stack = 100_000, 4
    F0 = n + n // 64 + stack + 1
    _FrameStore(8, OBS, np.uint8, stack, 16, 0)  # context, library and streams set up outside the measurement
    torch.cuda.synchronize()

    def delta(make):
        free0 = torch.cuda.mem_get_info()[0]
        st = make()
        torch.cuda.synchronize()
        d = free0 - torch.cuda.mem_get_info()[0]
        del st
        torch.cuda.synchronize()
        return d

    d_frames = delta(lambda: _FrameStore(n, OBS, np.uint8, stack, F0, 0))
    d_elements = delta(lambda: _DeviceStore(n, OBS + (stack,), np.uint8, 0))
    assert d_frames <= 1.05 * (F0 * 7056 + n * (2 * stack * 8 + 14)), d_frames
    assert d_frames <= 0.15 * d_elements, (d_frames, d_elements)
