"""Acting helpers — host-side mirror of slimdqn/sample_collection/utils.py (``select_action`` :8-15,
``collect_single_sample`` :18-40).  SURVEY §8(f) N1: outside the accelerated path (env-bound); kept so the
reference training loop runs unchanged against this package.  PRNG semantics: ``idqn_b200._prng``."""
from __future__ import annotations

import numpy as np

from .. import _prng
from .replay_buffer import ReplayBuffer, TransitionElement


def select_action(best_action_fn, params, state, key, n_actions, epsilon_fn, n_training_steps):
    agent = getattr(best_action_fn, "__self__", None)
    engine = getattr(agent, "_engine", None)
    if engine is not None and getattr(params, "_engine_ref", lambda: None)() is engine and getattr(params, "_which", None) == 0 \
            and getattr(agent, "n_networks", 0) == engine.K and not getattr(agent, "_squeeze", False):
        # the agent's own live parameters: draws + (on a greedy step) the forward pass in one call into the library
        return engine.select_action(state, key, n_actions, epsilon_fn(n_training_steps))[0]
    uniform_key, action_key, kwargs_key = _prng.split(key, 3)
    if _prng.uniform(uniform_key) <= epsilon_fn(n_training_steps):  # utils.py:12
        return _prng.randint(action_key, 0, n_actions)
    return best_action_fn(params, state, key=kwargs_key)  # only the taken branch is evaluated


def select_actions(best_action_fn, params, states, keys, n_actions, epsilon_fn, n_training_steps) -> np.ndarray:
    """``select_action`` for N environments: ``out[i] == select_action(best_action_fn, params, states[i], keys[i], ...)``.
    For the agent's own live online parameters (iDQN, and DQN, whose head draw ``randint(., 0, 1)`` is always 0) the
    draws and the greedy forward passes of all N environments run in one call into the library; anything else is the
    per-environment loop."""
    agent = getattr(best_action_fn, "__self__", None)
    engine = getattr(agent, "_engine", None)
    if len(states) != len(keys):
        raise ValueError(f"{len(states)} states but {len(keys)} keys")
    if engine is not None and getattr(params, "_engine_ref", lambda: None)() is engine and getattr(params, "_which", None) == 0 \
            and (engine.K == 1 if getattr(agent, "_squeeze", False) else getattr(agent, "n_networks", 0) == engine.K):
        return engine.select_actions(states, keys, n_actions, epsilon_fn(n_training_steps))[0]
    return np.asarray([select_action(best_action_fn, params, s, k, n_actions, epsilon_fn, n_training_steps)
                       for s, k in zip(states, keys)], np.int32).reshape(len(keys))


def collect_single_sample(key, env, agent, rb: ReplayBuffer, p, epsilon_schedule, n_training_steps: int):
    action = int(select_action(agent.best_action, agent.params, env.state, key, env.n_actions, epsilon_schedule,
                               n_training_steps))
    obs = env.observation
    reward, absorbing = env.step(action)
    episode_end = absorbing or env.n_steps >= p["horizon"]
    rb.add(TransitionElement(observation=obs, action=action,
                             reward=reward if rb._clipping is None else rb._clipping(reward),
                             is_terminal=absorbing, episode_end=episode_end))
    if episode_end:
        env.reset()
    return reward, episode_end
