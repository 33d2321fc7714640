"""Save and load of a full-size checkpoint on one GPU, in one process: the configuration tools/frame_store_bench.py fills,
at 1 M elements -- a filled 1 M-element Atari frame store (84x84 uint8 frames, stack 4), a 1 M prioritised sampler and a
K=5 NatureCNN agent.

Records:
- save and load wall time (host clock; every transfer ends in a stream synchronise), total and split into device transfer
  (time inside the store's bulk read/write calls and the agent's downloads/uploads) and the rest (file reads and writes,
  fsync, host bookkeeping);
- the checkpoint's bytes on disk;
- the device digest of the store: CUDA events on the store's stream around idqn_replay_digest, median of 5;
- the peak growth of the process's resident set during save and during load (sampled every 5 ms);
- the card name and power limit, read in the same run.

Writes one JSON file (--out).  The checkpoint goes to a temporary directory (--dir) and is deleted afterwards."""
import argparse
import json
import os
import shutil
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

OBS, FEATS, A, K, B = (84, 84, 4), [32, 64, 64, 512], 6, 5, 32
LR, GAMMA, EPS, T_FREQ, D_FREQ = 3e-4, 0.99, 1.5e-4, 200, 10


def rss_bytes() -> int:
    with open("/proc/self/statm") as f:
        return int(f.read().split()[1]) * os.sysconf("SC_PAGE_SIZE")


class PeakRSS:
    """Largest resident set seen while the block runs, minus the one at its start."""

    def __enter__(self):
        self.base = self.peak = rss_bytes()
        self._stop = threading.Event()
        self._t = threading.Thread(target=self._poll, daemon=True)
        self._t.start()
        return self

    def _poll(self):
        while not self._stop.wait(0.005):
            self.peak = max(self.peak, rss_bytes())

    def __exit__(self, *exc):
        self._stop.set()
        self._t.join()
        self.peak = max(self.peak, rss_bytes())
        self.growth = self.peak - self.base


class Timed:
    """Wraps methods of an object and adds the wall time spent inside them to `total`."""

    def __init__(self):
        self.total = 0.0

    def wrap(self, obj, *names):
        for name in names:
            fn = getattr(obj, name)

            def timed(*a, _fn=fn, **k):
                t0 = time.perf_counter()
                try:
                    return _fn(*a, **k)
                finally:
                    self.total += time.perf_counter() - t0
            setattr(obj, name, timed)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--elements", type=int, default=1_000_000)
    ap.add_argument("--dir", default=None, help="parent of the temporary checkpoint directory")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_checkpoint.json"))
    args = ap.parse_args()

    import torch

    from frame_store_bench import card
    from idqn_b200 import checkpoint as ckpt
    from idqn_b200.networks.idqn import iDQN
    from idqn_b200.sample_collection.replay_buffer import ReplayBuffer, TransitionElement
    from idqn_b200.sample_collection.samplers import PrioritizedSamplingDistribution

    assert torch.cuda.is_available(), "needs a CUDA device"
    n = args.elements
    out = {"card": card(), "elements": n}

    def build():
        rb = ReplayBuffer(PrioritizedSamplingDistribution(seed=0, max_capacity=n), batch_size=B, max_capacity=n,
                          stack_size=4, clipping=lambda r: np.clip(r, -1, 1), frame_store=True)
        return iDQN(0, OBS, A, K, FEATS, "cnn", LR, GAMMA, 1, 1, T_FREQ, D_FREQ, EPS), rb

    # ---- fill: n elements in 1000-step episodes, frames drawn from a pool of distinct random frames ------------------
    agent, rb = build()
    rng = np.random.default_rng(0)
    pool = rng.integers(0, 256, (4099, 84, 84), dtype=np.uint8)
    acts, rews = rng.integers(0, A, 8192), rng.integers(-1, 2, 8192)
    t0 = time.perf_counter()
    t = 0
    while rb.add_count < n:
        rb.add(TransitionElement(pool[t % len(pool)], int(acts[t % 8192]), float(rews[t % 8192]), t % 1000 == 999,
                                 t % 1000 == 999))
        t += 1
    out["fill_s"] = time.perf_counter() - t0
    for step in range(1, 51):  # some learning steps and priority updates, the last one left in flight
        agent.update_online_params(step, rb)
        rb.update_from_learner(agent._engine)
        agent.update_target_params(step)
    st = rb._store
    lo, hi = rb._lowest_frame_in_use(), rb._next_frame_id
    out["store"] = {"n_frames": st.n_frames, "live_frames": hi - lo, "frame_bytes": st.frame_bytes}

    # ---- digest --------------------------------------------------------------------------------------------------------
    stream = torch.cuda.ExternalStream(int(st.lib.idqn_replay_stream(st.h)))
    ms = []
    for _ in range(6):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        st.digest(n, lo, hi)
        e1.record(stream)
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    digest_bytes = (hi - lo) * ((st.frame_bytes + 7) // 8 * 8) + n * (8 * 8 + 14)
    med = float(np.median(ms[1:]))
    out["digest"] = {"ms": ms[1:], "median_ms": med, "bytes": digest_bytes, "GB_per_s": digest_bytes / med / 1e6,
                     "how": "CUDA events on the store's stream around idqn_replay_digest (allocation, memset, kernel, "
                            "48-byte read-back); first call dropped, median of 5"}

    # ---- save ------------------------------------------------------------------------------------------------------------
    parent = tempfile.mkdtemp(dir=args.dir)
    try:
        dev = Timed()
        dev.wrap(st, "read_frames", "read_slots")
        dev.wrap(agent._engine, "download_leaf", "get_count", "cumulated_losses")
        dig = Timed()
        dig.wrap(st, "digest")
        with PeakRSS() as rss:
            t0 = time.perf_counter()
            tmp = ckpt.begin(parent, "0")
            agent.save(os.path.join(tmp, "agent"))
            rb.save(os.path.join(tmp, "replay"))
            path = ckpt.commit(parent, "0")
            total = time.perf_counter() - t0
        size = sum(os.path.getsize(os.path.join(d, f)) for d, _, fs in os.walk(path) for f in fs)
        out["save"] = {"total_s": total, "device_transfer_s": dev.total, "digest_s": dig.total,
                       "file_io_and_host_s": total - dev.total - dig.total, "peak_rss_growth_bytes": rss.growth}
        out["checkpoint_bytes"] = size

        # ---- load into fresh objects ---------------------------------------------------------------------------------
        agent2, rb2 = build()
        torch.cuda.synchronize()
        dev = Timed()
        dev.wrap(agent2._engine, "upload_leaf", "set_count")
        dig = Timed()
        orig = type(rb2)._frame_store_type

        def store_type(*a, **k):  # time the bulk writes of the store the load creates
            s = orig(*a, **k)
            dev.wrap(s, "write_frames", "write_slots")
            dig.wrap(s, "digest")
            return s
        rb2._frame_store_type = store_type
        with PeakRSS() as rss:
            t0 = time.perf_counter()
            ckpt.verify(path)
            agent2.load(os.path.join(path, "agent"))
            rb2.load(os.path.join(path, "replay"))
            total = time.perf_counter() - t0
        out["load"] = {"total_s": total, "device_transfer_s": dev.total, "digest_s": dig.total,
                       "file_io_and_host_s": total - dev.total - dig.total, "peak_rss_growth_bytes": rss.growth}
        k1, k2 = rb._sampling_distribution.sample(B), rb2._sampling_distribution.sample(B)
        out["resumed_sampler_draws_same_keys"] = bool(np.array_equal(k1, k2))
        out["split_how"] = ("device_transfer: wall time inside the store's bulk read/write calls and the agent's "
                            "per-leaf downloads/uploads (each ends in a stream synchronise); digest: inside "
                            "idqn_replay_digest; file_io_and_host: the rest (file writes/reads, fsync, numpy)")
    finally:
        shutil.rmtree(parent, ignore_errors=True)

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
