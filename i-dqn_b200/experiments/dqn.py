"""``train`` — the reference's only driver (experiments/base/dqn.py:12-69) over the B200 agent, with the learning step
overlapped with environment stepping.

Same signature, same control flow, same bookkeeping as the reference.  What differs is *when the host waits*:

* ``agent.update_online_params(step, rb)`` only ENQUEUES the step (sample keys -> CUDA graph of the whole learn_on_batch)
  and returns; the host goes straight on to the next ``collect_single_sample`` -- environment step, replay ``add``,
  the three PRNG draws -- while the GPU computes.  The reference gets the same overlap from jax's asynchronous dispatch
  (idqn.py:72 accumulates device futures).
* losses are summed on the device (``cumulated_losses``) and read only at a T-update (idqn.py:82-87), the one host
  synchronisation per ``target_update_frequency`` learning steps besides the 4-byte action of a greedy acting step.
* ``update_to_data`` > 1 (idqn.py:66): the learner runs every ``update_to_data``-th environment step, so up to that many
  acting steps hide behind one learning step.

``p`` needs: n_epochs, n_training_steps_per_epoch, n_initial_samples, epsilon_end, epsilon_duration, horizon; optional
``wandb`` (anything with ``.log(dict)``), ``save`` (callable(p, returns, lengths, model), the reference's save_data) and
``checkpoint_dir``: after every epoch ``<checkpoint_dir>/<epoch>/`` receives the agent, the replay buffer (with its
sampler) and the loop state, and ``train`` resumes from the newest complete checkpoint there.  Only the newest
``rb._checkpoint_duration`` checkpoints are kept.  An epoch ends right after an episode ended, so the environment has
just been reset and nothing of it is saved: ``env`` stays the caller's object (its own random state is not restored).
"""
from __future__ import annotations

import os

import numpy as np

from .. import _prng
from .. import checkpoint as ckpt
from ..sample_collection.replay_buffer import TransitionElement
from ..sample_collection.utils import collect_single_sample, select_actions


def linear_schedule(init_value: float, end_value: float, transition_steps: int):
    """optax.linear_schedule(init, end, steps) (experiments/base/dqn.py:19): init + (end - init) * clip(count / steps, 0, 1)."""

    def schedule(count):
        if transition_steps <= 0:
            return init_value
        frac = min(max(count / transition_steps, 0.0), 1.0)
        return (init_value - end_value) * (1.0 - frac) + end_value  # optax's polynomial_schedule form, power 1

    return schedule


def train(key, p: dict, agent, env, rb):
    epsilon_schedule = linear_schedule(1.0, p["epsilon_end"], p["epsilon_duration"])
    log = p["wandb"].log if p.get("wandb") is not None else (lambda d: None)

    n_training_steps = 0
    env.reset()
    episode_returns_per_epoch = [[0]]
    episode_lengths_per_epoch = [[0]]
    first_epoch = 0
    root = p.get("checkpoint_dir")
    if root is not None and (latest := ckpt.latest_checkpoint(root)) is not None:
        ckpt.verify(latest)
        agent.load(os.path.join(latest, "agent"))
        rb.load(os.path.join(latest, "replay"))
        loop = ckpt.read_json(os.path.join(latest, "loop.json"))
        first_epoch, n_training_steps = loop["next_epoch"], loop["n_training_steps"]
        key = np.asarray(loop["key"], np.uint32)
        episode_returns_per_epoch, episode_lengths_per_epoch = loop["returns"], loop["lengths"]
        if len(episode_returns_per_epoch) == first_epoch:  # saved after what was then the last epoch
            episode_returns_per_epoch.append([0])
            episode_lengths_per_epoch.append([0])

    for idx_epoch in range(first_epoch, p["n_epochs"]):
        n_training_steps_epoch = 0
        has_reset = False

        while n_training_steps_epoch < p["n_training_steps_per_epoch"] or not has_reset:
            key, exploration_key = _prng.split(key)
            reward, has_reset = collect_single_sample(exploration_key, env, agent, rb, p, epsilon_schedule, n_training_steps)

            n_training_steps_epoch += 1
            n_training_steps += 1

            episode_returns_per_epoch[idx_epoch][-1] += reward
            episode_lengths_per_epoch[idx_epoch][-1] += 1
            if has_reset and n_training_steps_epoch < p["n_training_steps_per_epoch"]:
                episode_returns_per_epoch[idx_epoch].append(0)
                episode_lengths_per_epoch[idx_epoch].append(0)

            if n_training_steps > p["n_initial_samples"]:
                agent.update_online_params(n_training_steps, rb)  # enqueued; the next acting step overlaps it
                target_updated, logs = agent.update_target_params(n_training_steps)
                if target_updated:
                    log({"n_training_steps": n_training_steps, **logs})

        avg_return = np.mean(episode_returns_per_epoch[idx_epoch])
        avg_length_episode = np.mean(episode_lengths_per_epoch[idx_epoch])
        log({"epoch": idx_epoch, "n_training_steps": n_training_steps, "avg_return": avg_return,
             "avg_length_episode": avg_length_episode})
        if idx_epoch < p["n_epochs"] - 1:
            episode_returns_per_epoch.append([0])
            episode_lengths_per_epoch.append([0])
        if p.get("save") is not None:
            p["save"](p, episode_returns_per_epoch, episode_lengths_per_epoch, agent.get_model())
        if root is not None:
            tmp = ckpt.begin(root, str(idx_epoch))
            agent.save(os.path.join(tmp, "agent"))  # waits for the learner steps still in flight
            rb.save(os.path.join(tmp, "replay"))
            ckpt.write_json(os.path.join(tmp, "loop.json"), {
                "next_epoch": idx_epoch + 1, "n_training_steps": n_training_steps,
                "key": [int(k) for k in _prng.as_key(key)],
                "returns": episode_returns_per_epoch, "lengths": episode_lengths_per_epoch})
            ckpt.commit(root, str(idx_epoch), keep=rb._checkpoint_duration)
    return episode_returns_per_epoch, episode_lengths_per_epoch


def train_vectorized(key, p: dict, agent, envs, rb):
    """``train`` over N environments that act together: each iteration draws N + 1 keys, chooses all N actions in one
    ``select_actions`` call, then steps the environments in order, each step followed by ``train``'s body (replay ``add``
    into that environment's accumulator, reset on episode end, the learner past ``n_initial_samples``).  The learner
    still runs after every environment step, so ``update_to_data`` and the target schedule count environment steps.

    ``rb`` must have been built with ``n_envs=len(envs)``.  With one environment this is ``train`` exactly (the same
    keys, actions, epochs, returns and logs).  With more, an epoch ends at the first iteration boundary after at least
    ``n_training_steps_per_epoch`` environment steps; an episode's return and length go to the epoch in which it ended,
    and episodes still running carry over.  ``p["checkpoint_dir"]`` is refused: environments cannot be saved mid-episode."""
    if p.get("checkpoint_dir") is not None:
        raise ValueError("train_vectorized does not checkpoint (environments cannot be saved mid-episode): "
                         "remove p['checkpoint_dir']")
    n_envs = len(envs)
    if n_envs < 1 or getattr(rb, "_n_envs", 1) != n_envs:
        raise ValueError(f"train_vectorized needs a ReplayBuffer with n_envs={n_envs}, got {getattr(rb, '_n_envs', 1)}")
    epsilon_schedule = linear_schedule(1.0, p["epsilon_end"], p["epsilon_duration"])
    log = p["wandb"].log if p.get("wandb") is not None else (lambda d: None)
    single = n_envs == 1

    n_training_steps = 0
    for env in envs:
        env.reset()
    # one environment: train's lists (the running episode is the last entry); several: finished episodes only
    episode_returns_per_epoch = [[0]] if single else [[]]
    episode_lengths_per_epoch = [[0]] if single else [[]]
    running_return, running_length = [0.0] * n_envs, [0] * n_envs

    for idx_epoch in range(p["n_epochs"]):
        n_training_steps_epoch = 0
        has_reset = False

        while n_training_steps_epoch < p["n_training_steps_per_epoch"] or (single and not has_reset):
            key, *env_keys = _prng.split(key, n_envs + 1)
            actions = select_actions(agent.best_action, agent.params, [env.state for env in envs], env_keys,
                                     envs[0].n_actions, epsilon_schedule, n_training_steps)
            for i, env in enumerate(envs):
                action = int(actions[i])
                obs = env.observation
                reward, absorbing = env.step(action)
                has_reset = absorbing or env.n_steps >= p["horizon"]
                rb.add(TransitionElement(observation=obs, action=action,
                                         reward=reward if rb._clipping is None else rb._clipping(reward),
                                         is_terminal=absorbing, episode_end=has_reset), env=i)
                if has_reset:
                    env.reset()

                n_training_steps_epoch += 1
                n_training_steps += 1

                if single:
                    episode_returns_per_epoch[idx_epoch][-1] += reward
                    episode_lengths_per_epoch[idx_epoch][-1] += 1
                    if has_reset and n_training_steps_epoch < p["n_training_steps_per_epoch"]:
                        episode_returns_per_epoch[idx_epoch].append(0)
                        episode_lengths_per_epoch[idx_epoch].append(0)
                else:
                    running_return[i] += reward
                    running_length[i] += 1
                    if has_reset:
                        episode_returns_per_epoch[idx_epoch].append(running_return[i])
                        episode_lengths_per_epoch[idx_epoch].append(running_length[i])
                        running_return[i], running_length[i] = 0.0, 0

                if n_training_steps > p["n_initial_samples"]:
                    agent.update_online_params(n_training_steps, rb)
                    target_updated, logs = agent.update_target_params(n_training_steps)
                    if target_updated:
                        log({"n_training_steps": n_training_steps, **logs})

        finished = episode_returns_per_epoch[idx_epoch]
        avg_return = np.mean(finished) if finished else float("nan")  # several environments: maybe none ended
        avg_length_episode = np.mean(episode_lengths_per_epoch[idx_epoch]) if finished else float("nan")
        log({"epoch": idx_epoch, "n_training_steps": n_training_steps, "avg_return": avg_return,
             "avg_length_episode": avg_length_episode})
        if idx_epoch < p["n_epochs"] - 1:
            episode_returns_per_epoch.append([0] if single else [])
            episode_lengths_per_epoch.append([0] if single else [])
        if p.get("save") is not None:
            p["save"](p, episode_returns_per_epoch, episode_lengths_per_epoch, agent.get_model())
    return episode_returns_per_epoch, episode_lengths_per_epoch


class SyntheticAtari:
    """A stand-in environment with the interface the loop uses (reference: slimdqn/environments/atari.py): 84x84 uint8
    frames, a 4-frame ``state`` as float32 holding 0..255 (atari.py:43-45), ``observation`` = newest frame, a fixed
    host cost per ``step`` and episodes of ``episode_length`` steps.  Used by the tests and the overlap measurement; the
    real ALE wrapper is outside the scope of this package (SURVEY §2)."""

    def __init__(self, n_actions: int = 6, episode_length: int = 97, seed: int = 0, step_cost_s: float = 0.0):
        self.n_actions, self.episode_length, self.step_cost_s = n_actions, episode_length, step_cost_s
        self._rng = np.random.default_rng(seed)
        self._frames = self._rng.integers(0, 256, (64, 84, 84), dtype=np.uint8)
        self.actions = []
        self.reset()

    def reset(self):
        self.n_steps = 0
        self._stack = np.zeros((84, 84, 4), np.uint8)
        self._push(self._frames[0])

    def _push(self, frame):
        self._stack = np.concatenate([self._stack[..., 1:], frame[..., None]], axis=-1)

    @property
    def observation(self):
        return self._stack[..., -1]

    @property
    def state(self):
        return self._stack.astype(np.float32)

    def step(self, action: int):
        import time
        if self.step_cost_s > 0:  # emulator time: the host is busy, the GPU keeps learning
            t_end = time.perf_counter() + self.step_cost_s
            while time.perf_counter() < t_end:
                pass
        self.actions.append(int(action))
        self.n_steps += 1
        self._push(self._frames[(self.n_steps * 7 + int(action)) % len(self._frames)])
        reward = float((action + self.n_steps) % 3 - 1)
        absorbing = self.n_steps >= self.episode_length
        return reward, absorbing
