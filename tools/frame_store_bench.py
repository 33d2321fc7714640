"""Element store vs frame store (ReplayBuffer(frame_store=True)) on one GPU, in one process:

- resident NatureCNN K=5 learning steps/s (the workload of bench.py: batch 32, 84x84x4 uint8, A=6, T=200, D=10,
  4096 elements filled from 4200 random frames with 1 % terminals), CUDA events around `steps` steps after `warmup`,
  the two stores alternated three times; both buffers draw the same key stream (same sampler seed, same adds);
- rb.add latency of both stores (host clock around each call; every add ends in a stream synchronise);
- HBM of the stores from torch.cuda.mem_get_info around their creation: a 1M-element frame store measured, the element
  store measured at 100k elements (its 1M figure is 10x that, computed: 56 GB does not fit next to the rest).

Writes one JSON file (--out) with the card name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

OBS, FEATS, A, K, B = (84, 84, 4), [32, 64, 64, 512], 6, 5, 32
LR, GAMMA, EPS, T_FREQ, D_FREQ = 3e-4, 0.99, 1.5e-4, 200, 10


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, check=True)
    name, power = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--adds", type=int, default=2000)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_frame_store.json"))
    args = ap.parse_args()

    import torch

    from idqn_b200.networks.idqn import iDQN
    from idqn_b200.sample_collection.replay_buffer import ReplayBuffer, TransitionElement, _DeviceStore, _FrameStore
    from idqn_b200.sample_collection.samplers import UniformSamplingDistribution

    assert torch.cuda.is_available(), "needs a CUDA device"
    out = {"card": card(), "steps": args.steps, "warmup": args.warmup}

    # ---- HBM footprint ---------------------------------------------------------------------------------------------
    def hbm(make):
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        st = make()
        torch.cuda.synchronize()
        d = free0 - torch.cuda.mem_get_info()[0]
        del st
        torch.cuda.synchronize()
        return d

    hbm(lambda: _FrameStore(8, OBS[:2], np.uint8, 4, 16, 0))  # library / context set-up outside the measurement
    f0 = lambda n: n + n // 64 + 4 + 1
    out["hbm_bytes"] = {
        "frame_store_1m_measured": hbm(lambda: _FrameStore(1_000_000, OBS[:2], np.uint8, 4, f0(1_000_000), 0)),
        "frame_store_100k_measured": hbm(lambda: _FrameStore(100_000, OBS[:2], np.uint8, 4, f0(100_000), 0)),
        "element_store_100k_measured": hbm(lambda: _DeviceStore(100_000, OBS, np.uint8, 0)),
    }
    out["hbm_bytes"]["element_store_1m_computed_from_100k"] = 10 * out["hbm_bytes"]["element_store_100k_measured"]

    # ---- buffers and agents ----------------------------------------------------------------------------------------
    rng = np.random.default_rng(0)
    frames = rng.integers(0, 256, (4200 + args.adds, 84, 84), dtype=np.uint8)
    acts, rews = rng.integers(0, A, len(frames)), rng.integers(-1, 2, len(frames))
    terms = rng.random(len(frames)) < 0.01
    stores = {}
    for name, fs in (("element", False), ("frame", True)):
        rb = ReplayBuffer(UniformSamplingDistribution(seed=0), batch_size=B, max_capacity=4096, stack_size=4,
                          clipping=lambda r: np.clip(r, -1, 1), frame_store=fs)
        for t in range(4200):
            rb.add(TransitionElement(frames[t], int(acts[t]), float(rews[t]), bool(terms[t]), False))
        agent = iDQN(0, OBS, A, K, FEATS, "cnn", LR, GAMMA, 1, 1, T_FREQ, D_FREQ, EPS)
        stores[name] = {"rb": rb, "agent": agent, "step": 1, "keys": []}

    def run(s, n, record):
        agent, rb = s["agent"], s["rb"]
        for _ in range(n):
            agent.update_online_params(s["step"], rb)
            agent.update_target_params(s["step"])
            if record:
                s["keys"].append(np.asarray(rb.last_keys))
            s["step"] += 1

    rates = {"element": [], "frame": []}
    for rep in range(3):
        for name, s in stores.items():
            stream = torch.cuda.ExternalStream(int(s["agent"]._engine.lib.idqn_stream(s["agent"]._engine.h)))
            run(s, args.warmup, False)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            run(s, args.steps, rep == 0)
            e1.record(stream)
            torch.cuda.synchronize()
            rates[name].append(args.steps / (e0.elapsed_time(e1) / 1e3))
    same_keys = all(np.array_equal(a, b) for a, b in zip(stores["element"]["keys"], stores["frame"]["keys"]))
    med = {k: float(np.median(v)) for k, v in rates.items()}
    out["resident_steps_per_s"] = {"element": rates["element"], "frame": rates["frame"], "median": med,
                                   "frame_over_element": med["frame"] / med["element"],
                                   "same_sampled_keys": bool(same_keys)}
    out["resident_how"] = ("CUDA events on the learner stream around update_online_params + update_target_params "
                           "(T=200, D=10); alternated element, frame x3 in one process; first repetition's keys compared")

    # ---- rb.add latency ----------------------------------------------------------------------------------------------
    lat = {}
    for name, s in stores.items():
        rb, ts = s["rb"], []
        torch.cuda.synchronize()
        for t in range(4200, 4200 + args.adds):
            t0 = time.perf_counter()
            rb.add(TransitionElement(frames[t], int(acts[t]), float(rews[t]), bool(terms[t]), False))
            ts.append(time.perf_counter() - t0)
        ts = np.asarray(ts) * 1e6
        lat[name] = {"mean_us": float(ts.mean()), "median_us": float(np.median(ts)), "p99_us": float(np.percentile(ts, 99))}
    out["add_latency"] = lat
    out["frame_store_n_frames"] = stores["frame"]["rb"]._store.n_frames

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
