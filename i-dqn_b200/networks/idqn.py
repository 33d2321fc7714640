"""``iDQN`` — drop-in for slimdqn/networks/idqn.py of the reference, with every tensor resident on one B200
and the whole learning step (K online + K target forwards, iterated Bellman loss, backward, Adam) running as
one CUDA graph inside libidqn_b200.so.

Same constructor, attributes and methods as the reference class (idqn.py:28-134).  ``params`` /
``target_params`` / ``optimizer_state`` are live device views (``_engine.Tree``); handing them back to this
agent's methods moves no data.  Host pytrees (nested dicts of numpy arrays, flax layout, leading K axis) are
accepted everywhere the reference accepts a pytree and make the call pure-functional, as in the reference."""
from __future__ import annotations

import os
from typing import Any, Dict, Optional, Tuple

import numpy as np

from .. import _lib as L
from .. import _prng
from .. import checkpoint as ckpt
from ._engine import EmptyState, Engine, ScaleByAdamState, Tree, CountView, _get
from .architectures.dqn import DQNNet


def _engine_of(tree) -> Optional[Engine]:
    return tree._engine_ref() if isinstance(tree, Tree) else None


def shift_params(params):
    """idqn.py:13-17 — params[k] <- params[k+1] for k < K-1 (in place for device views)."""
    eng = _engine_of(params)
    if eng is not None:
        if params._which != L.ONLINE:
            raise ValueError("shift_params expects the online parameters")
        eng.shift_params()
        return params
    return _map(lambda a: np.concatenate([np.asarray(a)[1:], np.asarray(a)[-1:]], axis=0), params)


def sync_target_params(params, target_params):
    """idqn.py:20-24 — target[k] <- params[k-1] for k >= 1 (in place for device views)."""
    eng, eng_t = _engine_of(params), _engine_of(target_params)
    if eng is not None and eng is eng_t:
        eng.sync_target()
        return target_params
    params = params.to_host() if eng is not None else params
    target_params = target_params.to_host() if eng_t is not None else target_params
    return _map2(lambda p, t: np.concatenate([np.asarray(t)[:1], np.asarray(p)[:-1]], axis=0), params, target_params)


def _map(fn, tree):
    if isinstance(tree, dict):
        return {k: _map(fn, v) for k, v in tree.items()}
    return fn(tree)


def _map2(fn, a, b):
    if isinstance(a, dict):
        return {k: _map2(fn, a[k], b[k]) for k in a}
    return fn(a, b)


class iDQN:
    def __init__(
        self,
        key,
        observation_dim,
        n_actions,
        n_networks: int,
        features: list,
        architecture_type: str,
        learning_rate: float,
        gamma: float,
        update_horizon: int,
        update_to_data: int,
        target_update_frequency: int,
        target_sync_frequency: int,
        adam_eps: float = 1e-8,
        *,
        batch_size: int = 32,
        device: int = 0,
        flags: int = 0,
    ):
        self.n_networks = int(n_networks)
        self.network = DQNNet(features, architecture_type, n_actions)
        self._squeeze = False
        self._ctor = dict(observation_dim=observation_dim, n_actions=n_actions, features=features,
                          architecture_type=architecture_type, learning_rate=learning_rate, gamma=gamma,
                          update_horizon=update_horizon, adam_eps=adam_eps, batch_size=batch_size, device=device,
                          flags=flags)
        self._engine = self._make_engine()
        self._scratch: Optional[Engine] = None
        # K independently initialised heads (idqn.py:48-50); target_params = params (idqn.py:56)
        obs = tuple(int(d) for d in np.atleast_1d(observation_dim))
        keys = _prng.split(key, self.n_networks)
        heads = [self.network.init(k, np.zeros(obs, np.float32)) for k in keys]
        self._engine.upload_tree(L.ONLINE, _map_stack(heads))
        self._engine.copy_online_to_target()

        self.gamma = gamma
        self.update_horizon = update_horizon
        self.update_to_data = update_to_data
        self.target_update_frequency = target_update_frequency
        self.target_sync_frequency = target_sync_frequency

    def _make_engine(self) -> Engine:
        c = self._ctor
        return Engine(c["observation_dim"], c["n_actions"], self.n_networks, c["features"], c["architecture_type"],
                      c["learning_rate"], c["gamma"], c["update_horizon"], c["adam_eps"], batch_size=c["batch_size"],
                      device=c["device"], flags=c["flags"])

    # ---- state (live device views) -------------------------------------------------------------------
    def _view(self, which: int) -> Tree:
        # live views are stateless handles on an arena: built once (the acting path reads agent.params every environment step)
        cache = self.__dict__.setdefault("_views", {})
        v = cache.get((which, self._squeeze))
        if v is None or v._engine_ref() is not self._engine:
            v = cache[(which, self._squeeze)] = Tree(self._engine, which, self._squeeze)
        return v

    @property
    def params(self) -> Tree:
        return self._view(L.ONLINE)

    @params.setter
    def params(self, value):
        if not (isinstance(value, Tree) and value.is_view_of(self._engine, L.ONLINE)):
            self._engine.upload_tree(L.ONLINE, _host(value), squeezed=self._squeeze)

    @property
    def target_params(self) -> Tree:
        return self._view(L.TARGET)

    @target_params.setter
    def target_params(self, value):
        if isinstance(value, Tree) and value.is_view_of(self._engine, L.ONLINE):
            self._engine.copy_online_to_target()
        elif not (isinstance(value, Tree) and value.is_view_of(self._engine, L.TARGET)):
            self._engine.upload_tree(L.TARGET, _host(value), squeezed=self._squeeze)

    @property
    def optimizer_state(self):
        e = self._engine
        return (ScaleByAdamState(CountView(e, self._squeeze), self._view(L.MU), self._view(L.NU)), EmptyState())

    @optimizer_state.setter
    def optimizer_state(self, value):
        self._load_opt_state(self._engine, value)

    @property
    def cumulated_losses(self) -> np.ndarray:
        """idqn.py:63,72 — kept on the device; reading it is the only host sync."""
        return self._engine.cumulated_losses(reset=False)

    def gradients(self) -> Dict[str, Any]:
        """d loss_k / d params[k] of the most recent step (parity/debug aid; not in the reference)."""
        return self._engine.download_tree(L.GRAD, squeezed=self._squeeze)

    # ---- update_online_params / update_target_params (idqn.py:65-94) -----------------------------------
    def update_online_params(self, step: int, replay_buffer):
        if step % self.update_to_data == 0:
            learn = getattr(replay_buffer, "learn_step_on", None)
            if learn is not None and learn(self._engine):  # device-resident replay: gather + step, no host hop
                return
            batch_samples = replay_buffer.sample()
            self._engine.learn_host(batch_samples, want_losses=False)

    def update_target_params(self, step: int):
        if step % self.target_update_frequency == 0:
            # target_params[k] <- params[k], then the window shift params[k] <- params[k+1]  (idqn.py:75-80)
            self._engine.copy_online_to_target()
            self._engine.shift_params()

            cumulated = self._engine.cumulated_losses(reset=True)
            denom = self.target_update_frequency / self.update_to_data
            logs = {"loss": np.mean(cumulated) / denom}
            for idx_network in range(self.n_networks):
                logs[f"networks/{idx_network}_loss"] = cumulated[idx_network] / denom
            return True, logs

        if step % self.target_sync_frequency == 0:  # idqn.py:91-92
            self._engine.sync_target()

        return False, {}

    # ---- learn_on_batch (idqn.py:96-109) -------------------------------------------------------------
    def learn_on_batch(self, params, params_target, optimizer_state, batch_samples):
        """One gradient step of all K heads on one shared batch -> (params, optimizer_state, losses[K]).

        With this agent's own device views the step runs in place on the resident state and the same views
        are returned.  With host pytrees the call is pure: it runs on a scratch engine and returns new host
        pytrees, leaving the agent untouched."""
        own = (isinstance(params, Tree) and params.is_view_of(self._engine, L.ONLINE)
               and isinstance(params_target, Tree) and params_target.is_view_of(self._engine, L.TARGET))
        if own:
            self._engine.set_loss_accumulation(False)  # idqn.py:72: only update_online_params feeds cumulated_losses
            try:
                losses = self._engine.learn_host(batch_samples)
            finally:
                self._engine.set_loss_accumulation(True)
            return self.params, self.optimizer_state, self._out_loss(losses)
        eng = self._scratch_engine()
        eng.upload_tree(L.ONLINE, _host(params), squeezed=self._squeeze)
        eng.upload_tree(L.TARGET, _host(params_target), squeezed=self._squeeze)
        self._load_opt_state(eng, optimizer_state)
        losses = eng.learn_host(batch_samples)
        new_params = eng.download_tree(L.ONLINE, squeezed=self._squeeze)
        count = eng.get_count()
        new_state = (ScaleByAdamState(count[0] if self._squeeze else count,
                                      eng.download_tree(L.MU, squeezed=self._squeeze),
                                      eng.download_tree(L.NU, squeezed=self._squeeze)), EmptyState())
        return new_params, new_state, self._out_loss(losses)

    def last_scratch_gradients(self):
        """Gradients of the last pure-functional ``learn_on_batch`` call (parity aid)."""
        return self._scratch_engine().download_tree(L.GRAD, squeezed=self._squeeze)

    def _out_loss(self, losses):
        return losses

    def _scratch_engine(self) -> Engine:
        if self._scratch is None:
            self._scratch = self._make_engine()
        return self._scratch

    def _load_opt_state(self, eng: Engine, state):
        adam = state[0] if isinstance(state, tuple) and not hasattr(state, "mu") else state
        count, mu, nu = _get(adam, "count"), _get(adam, "mu"), _get(adam, "nu")
        if isinstance(mu, Tree) and mu.is_view_of(eng, L.MU):
            return
        eng.upload_tree(L.MU, _host(mu), squeezed=self._squeeze)
        eng.upload_tree(L.NU, _host(nu), squeezed=self._squeeze)
        eng.set_count(np.asarray(count))

    # ---- single-sample helpers (idqn.py:111-124); params carry NO K axis here, as in the reference -----
    def loss_on_batch(self, params, params_target, samples):
        s = np.asarray(_get(samples, "state"))
        losses = [self.loss(params, params_target, _index_sample(samples, i)) for i in range(s.shape[0])]
        return np.float32(np.mean(np.asarray(losses, np.float32)))

    def loss(self, params, params_target, sample):
        target = self.compute_target(params_target, sample)
        q_value = self.network.apply(params, _get(sample, "state"), self._ctor["device"])[int(_get(sample, "action"))]
        return np.square(np.float32(q_value) - target)

    def compute_target(self, params, sample):
        q_next = self.network.apply(params, _get(sample, "next_state"), self._ctor["device"])
        coef = np.float32(1 - int(_get(sample, "is_terminal"))) * np.float32(self.gamma ** self.update_horizon)
        return np.float32(_get(sample, "reward")) + coef * np.max(q_next)

    # ---- best_action (idqn.py:126-131) ----------------------------------------------------------------
    def best_action(self, params, state, key=None, idx_params: Optional[int] = None):
        """argmax_a Q(params[idx], state) with idx = jax.random.randint(key, (), 0, K) (restated, _prng.py);
        pass ``idx_params`` to pin the head explicitly."""
        if idx_params is None:
            idx_params = _prng.randint(key, 0, self.n_networks) if key is not None else 0
        if isinstance(params, Tree) and params._engine_ref() is self._engine:
            return self._engine.best_action(params._which, int(idx_params), state)
        head = _host(params) if self._squeeze else _map(lambda a: np.asarray(a)[idx_params], _host(params))
        return int(np.argmax(self.network.apply(head, state, self._ctor["device"])))

    def get_model(self):
        """idqn.py:133-134 — host numpy copy in the flax layout, so the pickles stay interchangeable."""
        return {"params": self._engine.download_tree(L.ONLINE, squeezed=self._squeeze)}

    # ---- checkpoint (no reference counterpart: the reference only pickles get_model()) --------------------------------
    _TREES = (("online", L.ONLINE), ("target", L.TARGET), ("mu", L.MU), ("nu", L.NU))

    def _checkpoint_meta(self) -> dict:
        """What a checkpoint must agree on: the model constructor fields and the schedule (not device / flags)."""
        c = self._ctor
        return {"class": type(self).__name__, "observation_dim": [int(d) for d in np.atleast_1d(c["observation_dim"])],
                "n_actions": int(c["n_actions"]), "n_networks": self.n_networks,
                "features": [int(f) for f in c["features"]], "architecture_type": c["architecture_type"],
                "learning_rate": float(c["learning_rate"]), "gamma": float(c["gamma"]),
                "update_horizon": int(c["update_horizon"]), "adam_eps": float(c["adam_eps"]),
                "batch_size": int(c["batch_size"]), "update_to_data": int(self.update_to_data),
                "target_update_frequency": int(self.target_update_frequency),
                "target_sync_frequency": int(getattr(self, "target_sync_frequency", self.target_update_frequency))}

    def save(self, directory: str) -> None:
        """Online and target parameters and the Adam moments in the flax layout (one .npz each, leaves named
        "Module.kind"), Adam's count and the device loss sums.  Waits for learner steps still in flight."""
        os.makedirs(directory, exist_ok=True)
        e = self._engine
        for name, which in self._TREES:
            leaves = {}
            for i, info in enumerate(e.leaves):
                a = e.download_leaf(which, i)
                leaves[info["module"].replace("/", ".") + "." + info["kind"]] = a[0] if self._squeeze else a
            np.savez(os.path.join(directory, name + ".npz"), **leaves)
        np.save(os.path.join(directory, "count.npy"), e.get_count())
        np.save(os.path.join(directory, "cumulated_losses.npy"), e.cumulated_losses(reset=False))
        ckpt.write_json(os.path.join(directory, "agent.json"), self._checkpoint_meta())

    def load(self, directory: str) -> None:
        """Restore what ``save`` wrote; ValueError naming the first field in which the checkpoint's agent differs."""
        saved = ckpt.read_json(os.path.join(directory, "agent.json"))
        for k, v in self._checkpoint_meta().items():
            if saved.get(k) != v:
                raise ValueError(f"agent checkpoint has {k}={saved.get(k)!r}, this agent {v!r}")
        e = self._engine
        for name, which in self._TREES:
            with np.load(os.path.join(directory, name + ".npz")) as z:
                for i, info in enumerate(e.leaves):
                    a = z[info["module"].replace("/", ".") + "." + info["kind"]]
                    e.upload_leaf(which, i, a[None] if self._squeeze else a)  # the bf16 planes are rebuilt from these
        e.set_count(np.load(os.path.join(directory, "count.npy")))
        sums = np.ascontiguousarray(np.load(os.path.join(directory, "cumulated_losses.npy")), np.float64)
        if sums.shape != (e.K,):
            raise ValueError(f"agent checkpoint has {sums.shape[0]} loss sums, this agent {e.K} heads")
        L.check(e.lib.idqn_write_cumulated_losses(e.h, L.ptr(sums)))


def _host(tree):
    return tree.to_host() if hasattr(tree, "to_host") else tree


def _map_stack(trees):
    t0 = trees[0]
    if isinstance(t0, dict):
        return {k: _map_stack([t[k] for t in trees]) for k in t0}
    return np.stack(trees)


def _index_sample(samples, i):
    names = ("state", "action", "reward", "next_state", "is_terminal")
    return {n: np.asarray(_get(samples, n))[i] for n in names}
