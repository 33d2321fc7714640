"""Acting for N environments on the GPU: ``select_actions`` equals ``select_action`` per environment (action, explore
decision, head) on every network path, is ordered after the learning steps enqueued before it, leaves learning
untouched, and ``train_vectorized`` over one environment is ``train``; over four it is deterministic, store-independent
and takes the learning steps its schedule implies.  A replay buffer of four environments round-trips its device
checkpoint."""
import gc

import numpy as np
import pytest
import torch

from oracle import networks as O

pytestmark = pytest.mark.gpu

OBS = (84, 84, 4)
FEATS = [32, 64, 64, 512]


def cnn_agent(K, flags=0, lr=3e-4, seed=0):
    from idqn_b200.networks.idqn import iDQN
    agent = iDQN(seed, OBS, 6, K, FEATS, "cnn", lr, 0.99, 1, 1, 8, 4, 1.5e-4, flags=flags)
    agent.params = O.init_params(np.random.default_rng(100 + K), OBS, FEATS, "cnn", 6, n_networks=K, bias_scale=0.01)
    return agent


def check_contract(agent, states, n_actions, ns=(1, 5, 32, 70), epsilons=(0.0, 0.3, 1.0)):
    from idqn_b200 import _prng
    from idqn_b200.sample_collection.utils import select_action, select_actions
    engine = agent._engine
    for eps in epsilons:
        for n in ns:
            keys = _prng.split(np.asarray([n, int(eps * 100)], np.uint32), n)
            got, explored, heads = engine.select_actions(states[:n], keys, n_actions, eps)
            for i in range(n):
                want = engine.select_action(states[i], keys[i], n_actions, eps)
                assert (int(got[i]), bool(explored[i]), int(heads[i])) == want, (eps, n, i)
            via_utils = select_actions(agent.best_action, agent.params, states[:n], keys, n_actions, lambda s: eps, 3)
            assert via_utils.tolist() == [select_action(agent.best_action, agent.params, states[i], keys[i], n_actions,
                                                        lambda s: eps, 3) for i in range(n)]
            assert via_utils.tolist() == got.tolist()
            if eps == 0.0:
                assert not explored.any()
            if eps == 1.0:
                assert explored.all()


@pytest.mark.parametrize("K", [1, 5])
@pytest.mark.parametrize("dtype", [np.uint8, np.float32], ids=["u8", "f32"])
def test_cnn_contract(K, dtype):
    agent = cnn_agent(K)
    states = np.random.default_rng(K).integers(0, 256, (70,) + OBS).astype(dtype)
    check_contract(agent, states, 6)


@pytest.mark.parametrize("flag", ["F_NO_IMG", "F_NO_GRAPH"])
def test_cnn_contract_generic_paths(flag):
    from idqn_b200 import _lib as L
    agent = cnn_agent(2, flags=getattr(L, flag))
    states = np.random.default_rng(7).integers(0, 256, (70,) + OBS).astype(np.uint8)
    check_contract(agent, states, 6, ns=(1, 5, 70))


def test_cnn_contract_fractional_float_states():
    """float observations that are not 0..255 integers take the generic float path"""
    agent = cnn_agent(2)
    states = np.random.default_rng(8).uniform(0, 255, (70,) + OBS).astype(np.float32)
    check_contract(agent, states, 6, ns=(5, 70))


def test_dqn_contract():
    from idqn_b200.networks.dqn import DQN
    agent = DQN(3, OBS, 6, FEATS, "cnn", 3e-4, 0.99, 1, 1, 8, 1.5e-4)
    states = np.random.default_rng(9).integers(0, 256, (70,) + OBS).astype(np.float32)
    check_contract(agent, states, 6)


def test_fc_and_impala_contract():
    from idqn_b200.networks.idqn import iDQN
    fc = iDQN(4, 8, 4, 3, [100, 100], "fc", 1e-3, 0.99, 1, 1, 8, 4, 1e-8)
    check_contract(fc, np.random.default_rng(10).standard_normal((70, 8)).astype(np.float32), 4)
    obs = (37, 29, 3)
    imp = iDQN(3, obs, 5, 2, [4, 6, 3, 10], "impala", 1e-3, 0.94, 1, 1, 1, 1, batch_size=8)
    check_contract(imp, np.random.default_rng(11).standard_normal((70,) + obs).astype(np.float32), 5, ns=(1, 5, 20))


def test_bad_arguments_are_refused():
    from idqn_b200 import _lib as L
    agent = cnn_agent(1)
    e = agent._engine
    states = np.zeros((3,) + OBS, np.uint8)
    keys = np.zeros((3, 2), np.uint32)
    with pytest.raises(ValueError):
        e.select_actions(states, keys[:2], 6, 0.0)
    with pytest.raises(ValueError):
        e.select_actions(states, keys, 0, 0.0)
    out = np.zeros(3, np.int32)
    with pytest.raises(ValueError):
        L.check(e.lib.idqn_select_actions(e.h, L.ptr(states), 1, -1, L.ptr(keys), 6, 0.0, L.ptr(out), None))
    a, x, h = e.select_actions(states[:0], keys[:0], 6, 0.0)
    assert len(a) == len(x) == len(h) == 0


# ---- ordering against in-flight learning steps ------------------------------------------------------------------------

def filled_buffer(seed, n=300, frame_store=False):
    from idqn_b200.sample_collection.replay_buffer import ReplayBuffer, TransitionElement
    from idqn_b200.sample_collection.samplers import UniformSamplingDistribution
    rng = np.random.default_rng(seed)
    rb = ReplayBuffer(UniformSamplingDistribution(seed=seed), batch_size=32, max_capacity=n, stack_size=4,
                      frame_store=frame_store)
    for t in range(n):
        rb.add(TransitionElement(rng.integers(0, 256, OBS[:2]).astype(np.uint8), int(rng.integers(0, 6)),
                                 float(rng.integers(-1, 2)), t % 50 == 49, t % 50 == 49))
    return rb


@pytest.mark.parametrize("path", ["replay", "submit_host"])
def test_select_actions_waits_for_enqueued_steps(path):
    from idqn_b200 import _prng
    from test_gpu_learn import make_batch
    rng = np.random.default_rng(21)
    states = rng.integers(0, 256, (32,) + OBS).astype(np.uint8)
    batches = [make_batch(np.random.default_rng(22 + i), 32, OBS, 6, True) for i in range(6)]
    runs = []
    for sync in (False, True):
        agent = cnn_agent(5, lr=3e-2)
        agent.target_params = O.init_params(np.random.default_rng(5), OBS, FEATS, "cnn", 6, n_networks=5, bias_scale=0.01)
        e = agent._engine
        rb = filled_buffer(23)
        acts = []
        for it in range(6):
            keys = _prng.split(np.asarray([it, 1], np.uint32), 32)
            if path == "replay":
                rb.learn_step_on(e)
            else:
                e.submit_host(batches[it])
            if sync:
                torch.cuda.synchronize()
            acts.append(e.select_actions(states, keys, 6, 0.0)[0])
            if path == "submit_host":
                e.submit_host(batches[(it + 3) % 6])  # a second batch in flight, the two staging slots alternating
        runs.append(np.stack(acts))
        del agent, rb
        gc.collect()
    np.testing.assert_array_equal(runs[0], runs[1])
    assert len({a.tobytes() for a in runs[0]}) > 1, "the learning steps did not change a single greedy action"


def agent_state(agent):
    from idqn_b200 import _lib as L
    e = agent._engine
    return [e.download_arena(w) for w in (L.ONLINE, L.TARGET, L.MU, L.NU)] + [e.get_count(), agent.cumulated_losses]


def assert_same_state(a, b):
    for x, y, name in zip(agent_state(a), agent_state(b), ("online", "target", "mu", "nu", "count", "losses")):
        assert np.asarray(x).tobytes() == np.asarray(y).tobytes(), name


def test_acting_leaves_learning_untouched():
    from idqn_b200 import _prng
    states = np.random.default_rng(31).integers(0, 256, (40,) + OBS).astype(np.uint8)
    agents = []
    for act in (False, True):
        agent = cnn_agent(5)
        rb = filled_buffer(32)
        for step in range(1, 21):
            agent.update_online_params(step, rb)
            if act:
                agent._engine.select_actions(states[: step * 2], _prng.split(step, step * 2), 6, 0.3)
            agent.update_target_params(step)
        agents.append(agent)
    assert_same_state(*agents)


# ---- train_vectorized ---------------------------------------------------------------------------------------------------

class Log:
    def __init__(self):
        self.entries = []

    def log(self, d):
        self.entries.append(dict(d))


def run_loop(vectorized, n_envs, frame_store, sampler="uniform", seed=5, K=2, utd=1):
    from idqn_b200.experiments.dqn import SyntheticAtari, train, train_vectorized
    from idqn_b200.networks.idqn import iDQN
    from idqn_b200.sample_collection.replay_buffer import ReplayBuffer
    from idqn_b200.sample_collection.samplers import PrioritizedSamplingDistribution, UniformSamplingDistribution
    s = UniformSamplingDistribution(seed=1) if sampler == "uniform" else PrioritizedSamplingDistribution(1, 300)
    kw = dict(n_envs=n_envs) if vectorized else {}
    rb = ReplayBuffer(s, batch_size=32, max_capacity=300, stack_size=4, clipping=lambda r: np.clip(r, -1, 1),
                      frame_store=frame_store, **kw)
    agent = iDQN(7, OBS, 6, K, FEATS, "cnn", 3e-4, 0.99, 1, utd, 20, 5, 1.5e-4)
    envs = [SyntheticAtari(n_actions=6, episode_length=23 + 7 * i, seed=i) for i in range(n_envs)]
    p = dict(n_epochs=2, n_training_steps_per_epoch=90, n_initial_samples=50, epsilon_end=0.01, epsilon_duration=150,
             horizon=1000, wandb=Log())
    if vectorized:
        ret, lens = train_vectorized(seed, p, agent, envs, rb)
    else:
        ret, lens = train(seed, p, agent, envs[0], rb)
    st = rb._store
    n_live = min(rb.add_count, rb._max_capacity)
    lo, hi = (rb._lowest_frame_in_use(), rb._next_frame_id) if frame_store else (0, 0)
    return dict(state=agent_state(agent), logs=p["wandb"].entries, ret=ret, lens=lens,
                actions=[list(e.actions) for e in envs], digest=st.digest(n_live, lo, hi), last_keys=rb.last_keys,
                count=np.asarray(agent._engine.get_count()))


def same_run(a, b, digest=True):
    for x, y, name in zip(a["state"], b["state"], ("online", "target", "mu", "nu", "count", "losses")):
        assert np.asarray(x).tobytes() == np.asarray(y).tobytes(), name
    assert a["actions"] == b["actions"] and a["logs"] == b["logs"] and (a["ret"], a["lens"]) == (b["ret"], b["lens"])
    assert np.asarray(a["last_keys"]).tolist() == np.asarray(b["last_keys"]).tolist()
    if digest:
        assert a["digest"] == b["digest"]


@pytest.mark.parametrize("frame_store", [False, True], ids=["element-store", "frame-store"])
def test_one_environment_is_train(frame_store):
    same_run(run_loop(True, 1, frame_store), run_loop(False, 1, frame_store))


@pytest.mark.parametrize("sampler", ["uniform", "prioritized"])
def test_four_environments(sampler):
    elem = run_loop(True, 4, False, sampler, utd=2)
    frames = run_loop(True, 4, True, sampler, utd=2)
    same_run(elem, frames, digest=False)  # the two stores hash different arrays
    same_run(frames, run_loop(True, 4, True, sampler, utd=2))
    n_steps = sum(len(a) for a in elem["actions"])
    assert n_steps == 2 * 92  # two epochs of 90 environment steps, rounded up to whole iterations of 4
    assert all(len(a) == n_steps // 4 for a in elem["actions"])
    assert elem["count"].tolist() == [sum(1 for s in range(51, n_steps + 1) if s % 2 == 0)] * 2
    assert [d["epoch"] for d in elem["logs"] if "epoch" in d] == [0, 1]
    finished = sum(len(l) for l in elem["lens"])
    assert finished == sum(len(a) // (23 + 7 * i) for i, a in enumerate(elem["actions"]))


def test_train_vectorized_refuses_checkpoints_and_mismatched_buffers():
    from idqn_b200.experiments.dqn import SyntheticAtari, train_vectorized
    from idqn_b200.sample_collection.replay_buffer import ReplayBuffer
    from idqn_b200.sample_collection.samplers import UniformSamplingDistribution
    envs = [SyntheticAtari(), SyntheticAtari(seed=1)]
    rb = ReplayBuffer(UniformSamplingDistribution(seed=1), 32, 100, n_envs=2)
    with pytest.raises(ValueError, match="checkpoint"):
        train_vectorized(0, {"checkpoint_dir": "x"}, None, envs, rb)
    with pytest.raises(ValueError, match="n_envs"):
        train_vectorized(0, {}, None, envs[:1], rb)


# ---- device checkpoint of a four-environment frame store ------------------------------------------------------------------

def test_four_environment_frame_store_round_trips(tmp_path):
    from idqn_b200.sample_collection.replay_buffer import ReplayBuffer, TransitionElement
    from idqn_b200.sample_collection.samplers import UniformSamplingDistribution
    rng = np.random.default_rng(41)
    drive = []
    for t in range(600):
        i = int(rng.integers(0, 4))
        end = rng.random() < 0.1
        drive.append((i, TransitionElement(rng.integers(0, 256, OBS[:2]).astype(np.uint8), int(rng.integers(0, 6)),
                                           float(rng.integers(-1, 2)), end and rng.random() < 0.5, end)))

    def make():
        return ReplayBuffer(UniformSamplingDistribution(seed=3), batch_size=32, max_capacity=200, stack_size=4,
                            update_horizon=3, frame_store=True, n_envs=4)

    a = make()
    for i, tr in drive[:400]:
        a.add(tr, env=i)
    assert sum(len(t) > 0 for t in a._trajectories) >= 2
    a.save(str(tmp_path / "rb"))
    b = make()
    b.load(str(tmp_path / "rb"))  # recomputes the device digests and compares them with the saved ones
    for i, tr in drive[400:]:
        a.add(tr, env=i)
        b.add(tr, env=i)
    lo, hi = a._lowest_frame_in_use(), a._next_frame_id
    assert (b._lowest_frame_in_use(), b._next_frame_id) == (lo, hi)
    assert a._store.digest(200, lo, hi) == b._store.digest(200, lo, hi)
    sa, sb = a.sample(), b.sample()
    for f in ("state", "action", "reward", "next_state", "is_terminal", "episode_end"):
        assert np.asarray(getattr(sa, f)).tobytes() == np.asarray(getattr(sb, f)).tobytes(), f
