"""Checkpoints on the GPU: a training run saved and resumed in fresh objects is bit-identical to one that never stopped
(element store and frame store, uniform and prioritised sampling), the device digest of the replay store equals its
NumPy restatement, a corrupted checkpoint is refused, a save right after an enqueued step captures that step, and the
other agents round-trip."""
import gc
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

OBS = (84, 84)


class Log:
    def __init__(self):
        self.entries = []

    def log(self, d):
        self.entries.append(dict(d))


def cnn_agent(K=2):
    from idqn_b200.networks.idqn import iDQN
    return iDQN(7, OBS + (4,), 6, K, [32, 64, 64, 512], "cnn", 3e-4, 0.99, 1, 1, 20, 5, 1.5e-4)


def agent_state(agent):
    from idqn_b200 import _lib as L
    e = agent._engine
    return [e.download_arena(w) for w in (L.ONLINE, L.TARGET, L.MU, L.NU)] + [e.get_count(), agent.cumulated_losses]


def assert_same_state(a, b):
    for x, y, name in zip(agent_state(a), agent_state(b), ("online", "target", "mu", "nu", "count", "losses")):
        assert x.tobytes() == y.tobytes(), name


# ---- 1. train() resumed from its checkpoint == train() that never stopped -------------------------------------------

@pytest.mark.parametrize("frame_store", [False, True], ids=["element-store", "frame-store"])
def test_train_resumes_bit_exactly(tmp_path, frame_store):
    from idqn_b200.experiments.dqn import SyntheticAtari, train
    from idqn_b200.sample_collection.replay_buffer import ReplayBuffer
    from idqn_b200.sample_collection.samplers import UniformSamplingDistribution

    # frame store: 3-step episodes cut by the horizon use 1.5 frames per element, so the ring grows before epoch 2
    episode, horizon = (97, 3) if frame_store else (37, 1000)
    cap = 150

    def objects(p_extra):
        p = dict(n_epochs=4, n_training_steps_per_epoch=120, n_initial_samples=64, epsilon_end=0.01,
                 epsilon_duration=300, horizon=horizon, wandb=Log())
        p.update(p_extra)
        rb = ReplayBuffer(UniformSamplingDistribution(seed=1), batch_size=32, max_capacity=cap, stack_size=4,
                          update_horizon=1, gamma=0.99, checkpoint_duration=2, clipping=lambda r: np.clip(r, -1, 1),
                          frame_store=frame_store)
        return p, cnn_agent(), SyntheticAtari(n_actions=6, episode_length=episode), rb

    p, agent, env, rb = objects({})
    ret, lens = train(5, p, agent, env, rb)
    whole = dict(state=agent_state(agent), logs=p["wandb"].entries, ret=ret, lens=lens, actions=list(env.actions),
                 sample=rb.sample())
    del p, agent, env, rb
    gc.collect()

    root = str(tmp_path / "ckpt")
    p, agent, env, rb = objects({"checkpoint_dir": root, "n_epochs": 2})
    train(5, p, agent, env, rb)
    logs, actions = p["wandb"].entries, list(env.actions)
    if frame_store:
        assert rb._store.n_frames > cap + cap // 64 + 4 + 1, "the ring did not grow before the checkpoint"
    assert sorted(os.listdir(root)) == ["0", "1"]
    del p, agent, env, rb
    gc.collect()
    torch.cuda.synchronize()

    p, agent, env, rb = objects({"checkpoint_dir": root})
    ret, lens = train(5, p, agent, env, rb)
    assert sorted(os.listdir(root)) == ["2", "3"], "checkpoint_duration=2 keeps the two newest"
    for x, y, name in zip(agent_state(agent), whole["state"], ("online", "target", "mu", "nu", "count", "losses")):
        assert x.tobytes() == y.tobytes(), name
    assert logs + p["wandb"].entries == whole["logs"]
    assert (ret, lens) == (whole["ret"], whole["lens"])
    assert actions + list(env.actions) == whole["actions"]
    s = rb.sample()
    for f in ("state", "action", "reward", "next_state", "is_terminal", "episode_end"):
        assert np.asarray(getattr(s, f)).tobytes() == np.asarray(getattr(whole["sample"], f)).tobytes(), f


# ---- 2. prioritised loop with device-side priority updates ----------------------------------------------------------

def test_prioritized_loop_resumes_bit_exactly(tmp_path):
    from idqn_b200.sample_collection import replay_buffer, samplers
    from idqn_b200.sample_collection.replay_buffer import TransitionElement

    rng = np.random.default_rng(4)
    trs = []
    for t in range(150 + 24 * 10):
        end = t % 50 == 49
        trs.append(TransitionElement(rng.integers(0, 256, OBS).astype(np.uint8), int(rng.integers(0, 6)),
                                     float(rng.integers(-1, 2)), end and t % 100 == 49, end))

    def build():
        rb = replay_buffer.ReplayBuffer(samplers.PrioritizedSamplingDistribution(seed=11, max_capacity=200),
                                        batch_size=32, max_capacity=200, stack_size=4, frame_store=True)
        return cnn_agent(), rb

    def steps(agent, rb, lo, hi, keys):
        for step in range(lo, hi):
            agent.update_online_params(step, rb)
            keys.append(np.asarray(rb.last_keys))
            rb.update_from_learner(agent._engine)
            agent.update_target_params(step)
            for tr in trs[150 + (step - 1) * 10: 150 + step * 10]:
                rb.add(tr)

    agent, rb = build()
    for tr in trs[:150]:
        rb.add(tr)
    keys_whole = []
    steps(agent, rb, 1, 25, keys_whole)
    tree = rb._sampling_distribution._sum_tree
    whole = (tree._nodes.tobytes(), tree.max_recorded_priority, agent_state(agent))

    agent, rb = build()
    for tr in trs[:150]:
        rb.add(tr)
    keys = []
    steps(agent, rb, 1, 13, keys)
    agent.save(str(tmp_path / "agent"))  # no synchronisation: the last priority update may still be in flight
    rb.save(str(tmp_path / "replay"))
    del agent, rb
    gc.collect()
    agent, rb = build()
    agent.load(str(tmp_path / "agent"))
    rb.load(str(tmp_path / "replay"))
    steps(agent, rb, 13, 25, keys)
    np.testing.assert_array_equal(np.stack(keys), np.stack(keys_whole))
    tree = rb._sampling_distribution._sum_tree
    assert tree._nodes.tobytes() == whole[0]
    assert tree.max_recorded_priority == whole[1]
    for x, y in zip(agent_state(agent), whole[2]):
        assert x.tobytes() == y.tobytes()


# ---- 3. the device digest against its NumPy restatement -------------------------------------------------------------

def test_digest_matches_numpy():
    from idqn_b200 import checkpoint as ckpt
    from idqn_b200.sample_collection.replay_buffer import _DeviceStore, _FrameStore
    rng = np.random.default_rng(0)

    def numpy_digests(frames, s, s2, a, r, d, e):
        head = [ckpt.frames_digest(frames), ckpt.digest(s)] if s2 is None else [ckpt.digest(s), ckpt.digest(s2)]
        return head + [ckpt.digest(np.asarray(x)) for x in (a, r, d, e)]

    def scalars(n):
        return (rng.integers(0, 6, n).astype(np.int32), rng.standard_normal(n), rng.integers(0, 2, n).astype(np.uint8),
                rng.integers(0, 2, n).astype(np.uint8))

    # frame stores: 15-byte frames (not a multiple of 8), 84x84 frames (many blocks); ids [lo, hi) wrap the ring
    for shape, n_frames, lo, hi, n_live in (((3, 5), 10, 7, 15, 6), (OBS, 700, 400, 1000, 500)):
        frames = rng.integers(0, 256, (hi - lo,) + shape).astype(np.uint8)
        rows = rng.integers(lo, hi, (n_live, 8))
        a, r, d, e = scalars(n_live)
        got = []
        for F in (n_frames, n_frames + 3):  # the digest does not depend on the ring's size
            st = _FrameStore(n_live + 2, shape, np.uint8, 4, F, 0)
            st.write_frames(lo, frames)
            st.write_slots(0, rows, None, a, r, d, e)
            assert lo % F + (hi - lo) > F, "the ids do not wrap the ring"
            np.testing.assert_array_equal(st.read_frames(lo, hi), frames)
            back = st.read_slots(0, n_live)
            np.testing.assert_array_equal(back[0], rows)
            assert back[1] is None and back[3].tobytes() == r.tobytes()
            got.append(st.digest(n_live, lo, hi))
        assert got[0] == got[1] == numpy_digests(frames, rows, None, a, r, d, e)
        with pytest.raises(ValueError):
            st.read_frames(lo, lo + n_frames + 4)
    # element store
    st = _DeviceStore(40, OBS + (4,), np.uint8, 0)
    s, s2 = (rng.integers(0, 256, (33,) + OBS + (4,)).astype(np.uint8) for _ in range(2))
    a, r, d, e = scalars(33)
    st.write_slots(0, s[:20], s2[:20], a[:20], r[:20], d[:20], e[:20])
    st.write_slots(20, s[20:], s2[20:], a[20:], r[20:], d[20:], e[20:])
    assert st.digest(33) == numpy_digests(None, s, s2, a, r, d, e)
    back = st.read_slots(0, 33)
    for x, y in zip(back, (s, s2, a, r, d, e)):
        assert x.tobytes() == y.tobytes()


# ---- 4. a corrupted checkpoint is refused ---------------------------------------------------------------------------

def test_flipped_frame_byte_is_refused(tmp_path):
    from idqn_b200.sample_collection import replay_buffer, samplers
    from idqn_b200.sample_collection.replay_buffer import TransitionElement
    rng = np.random.default_rng(2)

    def build():
        return replay_buffer.ReplayBuffer(samplers.UniformSamplingDistribution(seed=0), batch_size=32, max_capacity=64,
                                          stack_size=4, frame_store=True)

    rb = build()
    for t in range(90):
        rb.add(TransitionElement(rng.integers(0, 256, OBS).astype(np.uint8), 1, 0.0, False, t % 30 == 29))
    rb.save(str(tmp_path))
    path = tmp_path / "frames.npy"
    with open(path, "r+b") as f:
        f.seek(os.path.getsize(path) - 1000)
        b = f.read(1)
        f.seek(-1, 1)
        f.write(bytes([b[0] ^ 0x10]))
    with pytest.raises(ValueError, match="replay digest mismatch in state/frames"):
        build().load(str(tmp_path))


# ---- 5. a save right after an enqueued step ------------------------------------------------------------------------

def test_save_after_an_enqueued_step_captures_it(tmp_path):
    from idqn_b200.sample_collection import replay_buffer, samplers
    from idqn_b200.sample_collection.replay_buffer import TransitionElement
    rng = np.random.default_rng(3)
    trs = [TransitionElement(rng.integers(0, 256, OBS).astype(np.uint8), int(rng.integers(0, 6)), 1.0, False,
                             t % 40 == 39) for t in range(100)]
    out = []
    for sync in (False, True):
        agent = cnn_agent()
        rb = replay_buffer.ReplayBuffer(samplers.UniformSamplingDistribution(seed=0), batch_size=32, max_capacity=100,
                                        stack_size=4, frame_store=True)
        for tr in trs:
            rb.add(tr)
        for step in range(1, 6):
            agent.update_online_params(step, rb)
        if sync:
            torch.cuda.synchronize()
        d = tmp_path / str(sync)
        agent.save(str(d / "agent"))
        rb.save(str(d / "replay"))
        out.append(d)
    for name in ("online", "target", "mu", "nu"):
        with np.load(out[0] / "agent" / f"{name}.npz") as x, np.load(out[1] / "agent" / f"{name}.npz") as y:
            assert sorted(x.files) == sorted(y.files)
            for k in x.files:
                assert x[k].tobytes() == y[k].tobytes(), (name, k)
    for name in ("count.npy", "cumulated_losses.npy"):
        assert np.load(out[0] / "agent" / name).tobytes() == np.load(out[1] / "agent" / name).tobytes()
    assert np.load(out[0] / "agent" / "count.npy").tolist() == [5, 5]


# ---- 6. the MLP float agent and DQN --------------------------------------------------------------------------------

@pytest.mark.parametrize("kind", ["mlp", "dqn"])
def test_other_agents_round_trip(tmp_path, kind):
    from idqn_b200.networks.dqn import DQN
    from idqn_b200.networks.idqn import iDQN
    if kind == "mlp":
        obs = (8,)
        make = lambda key, lr=3e-4: iDQN(key, obs, 4, 3, [100, 100], "fc", lr, 0.99, 1, 1, 5, 3, 1e-8)
    else:
        obs = OBS + (4,)
        make = lambda key, lr=3e-4: DQN(key, obs, 6, [32, 64, 64, 512], "cnn", lr, 0.99, 1, 1, 5, 1.5e-4)
    rng = np.random.default_rng(1)

    def batch():
        s = (rng.integers(0, 256, (32,) + obs).astype(np.uint8) if kind == "dqn"
             else rng.standard_normal((32,) + obs).astype(np.float32))
        return dict(state=s, next_state=s[::-1].copy(), action=rng.integers(0, 4, 32), reward=rng.standard_normal(32),
                    is_terminal=rng.random(32) < 0.1)

    class Fixed:
        def __init__(self, b):
            self.b = b

        def sample(self):
            return self.b

    a = make(1)
    for step in range(1, 8):
        a.update_online_params(step, Fixed(batch()))
        a.update_target_params(step)
    a.save(str(tmp_path))
    if kind == "dqn":
        with np.load(tmp_path / "online.npz") as z:
            assert z["Conv_0.kernel"].shape == (8, 8, 4, 32), "DQN keeps its leaves without the K axis"
    b = make(2)
    b.load(str(tmp_path))
    assert_same_state(a, b)
    nxt = batch()
    for ag in (a, b):
        ag.update_online_params(8, Fixed(nxt))
    assert_same_state(a, b)
    with pytest.raises(ValueError, match="learning_rate"):
        make(1, lr=1e-3).load(str(tmp_path))
