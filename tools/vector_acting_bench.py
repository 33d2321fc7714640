"""Acting for N environments (select_actions) on one GPU, in one process:

- acting latency of a K=5 NatureCNN agent at epsilon 0 for N in {1, 4, 8, 16, 32, 64}: median wall time of one
  select_actions call (it ends in a stream synchronise) over `calls` calls, against N sequential select_action calls
  on the same states and keys;
- environment steps/s of train_vectorized with SyntheticAtari environments (in the style of tools/train_overlap.py) for
  N in {1, 8, 32}, update_to_data in {1, 4} and an emulator costing 0 or 150 us of host time per step: one warm-up epoch,
  then `env_steps` timed environment steps.

Writes one JSON file (--out) with the card name and power limit read in the same run."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from frame_store_bench import card  # noqa: E402

OBS, FEATS, A, K = (84, 84, 4), [32, 64, 64, 512], 6, 5


def acting(calls):
    import torch
    from idqn_b200 import _prng
    from idqn_b200.networks.idqn import iDQN
    from idqn_b200.sample_collection.utils import select_action, select_actions
    agent = iDQN(5, OBS, A, K, FEATS, "cnn", 3e-4, 0.99, 1, 1, 200, 10, 1.5e-4)
    eps = lambda step: 0.0
    rng = np.random.default_rng(0)
    rows = []
    for n in (1, 4, 8, 16, 32, 64):
        states = rng.integers(0, 256, (n,) + OBS).astype(np.float32)  # atari.py:43-45: float32 holding 0..255
        keys = _prng.split(n, n)
        vec, seq = [], []
        for it in range(calls + 20):  # the first 20 of each: graph capture, warm-up
            t0 = time.perf_counter()
            got = select_actions(agent.best_action, agent.params, states, keys, A, eps, 0)
            t1 = time.perf_counter()
            want = [select_action(agent.best_action, agent.params, s, k, A, eps, 0) for s, k in zip(states, keys)]
            t2 = time.perf_counter()
            if it >= 20:
                vec.append(t1 - t0)
                seq.append(t2 - t1)
            assert got.tolist() == want
        torch.cuda.synchronize()
        row = {"n_envs": n, "select_actions_us": float(np.median(vec) * 1e6),
               "sequential_select_action_us": float(np.median(seq) * 1e6)}
        row["speedup"] = row["sequential_select_action_us"] / row["select_actions_us"]
        print(row, flush=True)
        rows.append(row)
    return rows


def loop(env_steps):
    import torch
    from idqn_b200.experiments.dqn import SyntheticAtari, train_vectorized
    from idqn_b200.networks.idqn import iDQN
    from idqn_b200.sample_collection.replay_buffer import ReplayBuffer
    from idqn_b200.sample_collection.samplers import UniformSamplingDistribution
    rows = []
    for n in (1, 8, 32):
        for utd in (1, 4):
            for cost in (0.0, 150.0):
                agent = iDQN(5, OBS, A, K, FEATS, "cnn", 3e-4, 0.99, 1, utd, 200, 10, 1.5e-4)
                rb = ReplayBuffer(UniformSamplingDistribution(seed=1), batch_size=32, max_capacity=8192, stack_size=4,
                                  clipping=lambda r: np.clip(r, -1, 1), n_envs=n)
                envs = [SyntheticAtari(episode_length=500 + 13 * i, seed=i, step_cost_s=cost * 1e-6) for i in range(n)]
                # epsilon 1 on step 0 only, then 0.01: almost every step is greedy
                p = dict(n_epochs=1, n_training_steps_per_epoch=600, n_initial_samples=100, epsilon_end=0.01,
                         epsilon_duration=1, horizon=10 ** 6)
                train_vectorized(3, p, agent, envs, rb)  # warm-up epoch (graph capture, allocator)
                for e in envs:
                    e.actions.clear()
                p = dict(p, n_training_steps_per_epoch=env_steps, n_initial_samples=0)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                train_vectorized(4, p, agent, envs, rb)
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                steps = sum(len(e.actions) for e in envs)
                row = {"n_envs": n, "update_to_data": utd, "emulator_us": cost, "env_steps": steps,
                       "env_steps_per_s": steps / dt, "us_per_env_step": dt / steps * 1e6}
                print(row, flush=True)
                rows.append(row)
                del agent, rb
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_vector_acting.json"))
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--env-steps", type=int, default=3000)
    args = ap.parse_args()
    out = {"card": card(), "K": K, "epsilon": 0.0, "calls": args.calls}
    out["acting"] = acting(args.calls)
    out["loop"] = loop(args.env_steps)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
