#!/usr/bin/env python
"""Benchmark of the i-DQN learning step (BASELINE.json metric: gradient steps/s, NatureCNN K=5, batch 32).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Ours, N GPUs: one process per GPU (torchrun for N>1); each rank owns 5 heads of one 5N-head i-DQN chain
(weak scaling, head-sharded; the only cross-GPU traffic is the neighbour target exchange every D / T steps, a kernel
storing into the neighbour's memory over NVLink).
`value`     : steps/s with the replay store resident in HBM (sampler indices are the only H2D traffic);
`e2e`       : steps/s through the host-buffer C-ABI call (H2D of the batch + D2H of the losses every step);
`strong_k8` : BASELINE configs[3] -- ONE K=8 chain sharded ceil(8/N) heads per GPU, chain steps/s, next to the K=8 rate of a
              single GPU measured in the same run (speed-up and efficiency follow from the two);
`sharded_parity` (N>1): the sharded K=8 chain against the unsharded K=8 agent, bit for bit, on every rank.
Reference: the CPU oracle restatement of the reference's learn_on_batch (jax is not installable here; if `import jax`
ever succeeds the reference's own slimdqn.networks.idqn.iDQN.learn_on_batch is timed instead) on the host cores of the
box (`--impl reference`, and the `cpu_baseline` leg of the default run)."""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

OBS, FEATS, A, B, HEADS_PER_GPU = (84, 84, 4), [32, 64, 64, 512], 6, 32, 5
LR, GAMMA, EPS, T_FREQ, D_FREQ = 3e-4, 0.99, 1.5e-4, 200, 10
P_HEAD = 4_046_502
F_MAC, DG_MAC, WG_MAC = 16_006_144, 12_393_472, 16_006_144  # SURVEY §8(d)
FLOP_PER_HEAD_STEP = B * 2 * (2 * F_MAC + DG_MAC + WG_MAC)
BYTES_PER_HEAD_STEP = 7 * P_HEAD * 4
BATCH_BYTES = B * (2 * 28224 + 9)
METRIC = "i-DQN grad steps/sec (NatureCNN K=5, batch 32)"


def config(n_gpus: int) -> dict:
    """The same `config` object in both arms (the driver compares the two JSON lines)."""
    return {"workload": (f"Atari NatureCNN i-DQN, {HEADS_PER_GPU} heads per GPU ({HEADS_PER_GPU * n_gpus} total, head-sharded), "
                         "batch 32, 84x84x4 uint8, A=6, T=200, D=10, uniform replay"),
            "heads_total": HEADS_PER_GPU * n_gpus,
            "l2": "inputs larger than L2: working set per step (5 arenas x 81 MB per GPU + 231 MB replay) exceeds the 126 MB L2; no flush"}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm=float(p["hbm_gbs"]), tf_burst=float(p["bf16_tflops"]), tf_sus=float(p["bf16_tflops_sustained"]),
                    src="measured")
    except Exception:
        return dict(hbm=6650.0, tf_burst=1590.0, tf_sus=1400.0, src="fallback")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (pynvml, 50 ms period)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.max_mhz = index, False, [], set(), None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                     "sw_power_cap": 0x4, "hw_power_brake": 0x80}
            while not self.stop_flag:
                self.sm.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for n, bit in names.items():
                    if r & bit:
                        self.reasons.add(n)
                time.sleep(0.05)
        except Exception as e:  # pragma: no cover
            self.reasons.add(f"unavailable:{type(e).__name__}")

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.sm)}


def synthetic_batch(rng):
    return dict(state=rng.integers(0, 256, (B,) + OBS, dtype=np.uint8),
                next_state=rng.integers(0, 256, (B,) + OBS, dtype=np.uint8),
                action=rng.integers(0, A, B).astype(np.int32),
                reward=rng.integers(-1, 2, B).astype(np.float32), is_terminal=(rng.random(B) < 0.1))


# ------------------------------------------------------------------------------------------------------
def jax_reference_rate(n_heads: int, max_steps: int, warmup: int):
    """If jax/flax/optax ever become importable: the reference's OWN learn_on_batch (slimdqn/networks/idqn.py:96-109)
    on JAX_PLATFORMS=cpu.  Returns None when they are not (the case in this image)."""
    try:
        os.environ.setdefault("JAX_PLATFORMS", "cpu")
        import jax  # noqa: F401
        sys.path.insert(0, os.environ.get("IDQN_REFERENCE_PATH", os.path.join(ROOT, "baseline", "_ref")))
        from slimdqn.networks.idqn import iDQN as RefIDQN
    except Exception:
        return None
    agent = RefIDQN(jax.random.PRNGKey(0), OBS, A, n_heads, FEATS, "cnn", LR, GAMMA, 1, 1, T_FREQ, D_FREQ, EPS)
    from slimdqn.sample_collection.replay_buffer import ReplayElement
    b = synthetic_batch(np.random.default_rng(0))
    batch = ReplayElement(state=b["state"], action=b["action"], reward=b["reward"], next_state=b["next_state"],
                          is_terminal=b["is_terminal"], episode_end=b["is_terminal"])
    p, o = agent.params, agent.optimizer_state
    for _ in range(warmup):
        p, o, l = agent.learn_on_batch(p, agent.target_params, o, batch)
        jax.block_until_ready(l)
    times = []
    for _ in range(max_steps):
        t0 = time.perf_counter()
        p, o, l = agent.learn_on_batch(p, agent.target_params, o, batch)
        jax.block_until_ready(l)
        times.append(time.perf_counter() - t0)
    return 1.0 / float(np.median(times)), len(times), os.cpu_count()


def cpu_reference_rate(n_heads: int, min_seconds: float, max_steps: int, warmup: int = 1, threads: int = 0):
    """steps/s of the CPU oracle restatement of learn_on_batch (fp32).  threads = 0: every host core."""
    import torch
    from oracle import networks as O

    # torchrun exports OMP_NUM_THREADS=1: set the thread count explicitly (round-1 N>=2 reference lines ran on one thread)
    torch.set_num_threads(threads if threads > 0 else (os.cpu_count() or 1))
    rng = np.random.default_rng(0)
    params = O.init_params(rng, OBS, FEATS, "cnn", A, n_networks=n_heads)
    target = O.init_params(np.random.default_rng(1000), OBS, FEATS, "cnn", A, n_networks=n_heads)
    learner = O.CpuLearner(params, target, "cnn", GAMMA, 1, LR, EPS)
    batch = synthetic_batch(rng)
    for _ in range(warmup):
        learner.step(batch)
    times = []
    t_start = time.perf_counter()
    # min_seconds > 0: a time-bounded sample (cpu_baseline leg); otherwise exactly max_steps steps (reference arm)
    while len(times) < max_steps and (min_seconds <= 0 or time.perf_counter() - t_start < min_seconds or len(times) < 3):
        t0 = time.perf_counter()
        learner.step(batch)
        times.append(time.perf_counter() - t0)
    return 1.0 / float(np.median(times)), len(times), torch.get_num_threads()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_heads = HEADS_PER_GPU * args.gpus
    steps = max(1, min(args.steps, 100))  # bounded sample: at most 100 CPU steps (40 ms .. 0.4 s each at N = 1..8)
    warm = args.warmup
    jx = jax_reference_rate(n_heads, steps, warm)
    if jx is not None:
        rate, n, threads = jx
        kind, sample = "reference", f"{n} learn_on_batch steps of slimdqn.networks.idqn.iDQN on JAX_PLATFORMS=cpu"
    else:
        rate, n, threads = cpu_reference_rate(n_heads, min_seconds=0.0, max_steps=steps, warmup=min(warm, 3))
        kind, sample = "port", f"{n} full learn_on_batch steps of the torch-CPU fp32 oracle (jax not installable)"
    value = rate * args.gpus  # same head-normalised unit as our arm (steps/s of a K=5 agent)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value,
        "unit": "steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 / rate,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config(args.gpus),
        "timed_steps": n, "untimed_warmup": min(warm, 3),
        "cpu_baseline": {"value": value, "unit": "steps/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------------------
def source_sha() -> str:
    """Hash of the kernel sources: profiles/ncu_traffic.json is only trusted for the sources it was captured from."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "i-dqn_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh")):
            with open(os.path.join(d, f), "rb") as fh:
                h.update(fh.read())
    return h.hexdigest()[:16]


DUMP_SAMPLE = 65536  # entries kept per head of a larger leaf (only Dense_0/kernel, 3.96 M per head, at the bench sizes)


def dump_outputs(agent, L, out_dir):
    """Writes what the timed resident path leaves its caller after its last step, one DIR/<name>.npy per array: the
    online and target parameters, the Adam moments and step counts, the device-side loss sums (idqn.py:63,72) and the
    |TD| of the last step per head and sample.  A leaf larger than DUMP_SAMPLE entries per head is reduced to a fixed,
    seeded sample of its entries, the same ones in every tree: about 12 MB in all at K = 5."""
    eng = agent._engine
    os.makedirs(out_dir, exist_ok=True)
    out = {"cumulated_losses": agent.cumulated_losses, "td_abs": eng.td_abs(),
           "optimizer_state.count": eng.get_count().astype(np.float64)}
    for i, info in enumerate(eng.leaves):
        pick = None
        if info["size"] > DUMP_SAMPLE:
            pick = np.sort(np.random.default_rng(i).choice(info["size"], DUMP_SAMPLE, replace=False))
        leaf = info["module"].replace("/", ".") + "." + info["kind"]
        for tree, which in (("params", L.ONLINE), ("target_params", L.TARGET), ("optimizer_state.mu", L.MU),
                            ("optimizer_state.nu", L.NU)):
            a = eng.download_leaf(which, i)
            out[f"{tree}.{leaf}"] = a if pick is None else a.reshape(eng.K, -1)[:, pick]
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args):
    import torch
    import torch.distributed as dist

    from idqn_b200 import _lib as L
    from idqn_b200.networks.idqn import iDQN, _map_stack
    from idqn_b200.networks.architectures.dqn import DQNNet
    from idqn_b200.parallel import head_partition, make_sharded_idqn
    from idqn_b200.sample_collection.replay_buffer import ReplayBuffer, TransitionElement
    from idqn_b200.sample_collection.samplers import UniformSamplingDistribution

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    net = DQNNet(FEATS, "cnn", A)

    def make_agent(k_total, T=T_FREQ, D=D_FREQ, flags=0):
        """k_total-head chain over all ranks (this rank's shard) with an independent target draw (theta_bar != theta)."""
        if world > 1:
            ag = make_sharded_idqn(0, OBS, A, k_total, FEATS, "cnn", LR, GAMMA, 1, 1, T, D, EPS, rank=rank,
                                   world_size=world, device=local, flags=flags)
            start = ag.head_offset
        else:
            ag = iDQN(0, OBS, A, k_total, FEATS, "cnn", LR, GAMMA, 1, 1, T, D, EPS, device=local, flags=flags)
            start = 0
        e = ag._engine
        e.upload_tree(L.TARGET, _map_stack([net.init(1000 + start + k, np.zeros(OBS, np.float32)) for k in range(e.K)]))
        return ag

    k_total = HEADS_PER_GPU * world
    agent = make_agent(k_total, flags=args.flags)
    eng = agent._engine

    # device-resident replay: 4096 synthetic stacked elements = 231 MB (> 126 MB L2), same content on every rank
    rb = ReplayBuffer(UniformSamplingDistribution(seed=0), batch_size=B, max_capacity=4096, stack_size=4,
                      clipping=lambda r: np.clip(r, -1, 1), device=local)
    rng = np.random.default_rng(0)
    frames = rng.integers(0, 256, (4200, 84, 84), dtype=np.uint8)
    for t in range(4200):
        rb.add(TransitionElement(frames[t], int(rng.integers(0, A)), float(rng.integers(-1, 2)),
                                 bool(rng.random() < 0.01), False))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(engine, fn, steps, warmup, first_step, drain=None, clocks=False):
        stream = torch.cuda.ExternalStream(int(engine.lib.idqn_stream(engine.h)), device=f"cuda:{local}")
        step = first_step
        for _ in range(warmup):
            fn(step)
            step += 1
        if drain:
            drain()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sampler = ClockSampler(local) if clocks else None
        if sampler:
            sampler.start()
        t0 = time.perf_counter()
        e0.record(stream)
        for _ in range(steps):
            fn(step)
            step += 1
        if drain:
            drain()  # the last step's losses are read inside the timed region
        e1.record(stream)
        barrier()
        wall = time.perf_counter() - t0
        if sampler:
            sampler.stop_flag = True
            sampler.join()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=f"cuda:{local}")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, wall, (sampler.summary() if sampler else None), step

    # (1) resident path: sampler -> device gather -> step (+ the T/D target events of the schedule)
    def resident_step(step):
        agent.update_online_params(step, rb)
        agent.update_target_params(step)

    ms, wall, clocks, nxt = timed(eng, resident_step, args.steps, args.warmup, 1, clocks=True)
    steps_per_s = args.steps / (ms / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(agent, L, args.dump_outputs)

    # (2) end to end through the host-buffer C-ABI call: pinned host batch -> H2D -> step -> D2H losses
    pool = []
    for i in range(8):
        b = synthetic_batch(np.random.default_rng(100 + i))
        pinned = {k: torch.from_numpy(np.ascontiguousarray(v.astype(np.uint8) if v.dtype == bool else v)).pin_memory()
                  for k, v in b.items()}
        pool.append({k: t.numpy() for k, t in pinned.items()} | {"_keep": pinned})

    # (2a) pipelined the way the reference's own call is (async dispatch): submit enqueues the pinned H2D copies of
    # this step on the copy stream + the step, the losses of the previous step are read back (D2H) right after
    pending = [None]
    loss_log = []

    def e2e_step(step):
        b = pool[step % len(pool)]
        t = eng.submit_host(b)
        if pending[0] is not None:
            loss_log.append(eng.wait_losses(pending[0]))
        pending[0] = t
        agent.update_target_params(step)

    def e2e_drain():
        if pending[0] is not None:
            loss_log.append(eng.wait_losses(pending[0]))
            pending[0] = None

    e2e_steps = args.steps
    ms_e2e, _, _, nxt = timed(eng, e2e_step, e2e_steps, args.warmup, nxt, drain=e2e_drain)
    e2e_rate = e2e_steps / (ms_e2e / 1e3)
    assert len(loss_log) >= e2e_steps and all(np.isfinite(l).all() for l in loss_log)

    # (2b) the call a user of the reference makes: agent.update_online_params(step, replay_buffer) with a HOST replay buffer
    # (rb.sample() hands over a host batch, idqn.py:65-72) + update_target_params; losses stay on the device until a
    # T-update reads their sum (idqn.py:82-87), exactly like the reference's device futures
    class HostBuffer:
        def __init__(self):
            self.i = 0

        def sample(self):
            self.i += 1
            return pool[self.i % len(pool)]

    host_rb = HostBuffer()

    def dropin_step(step):
        agent.update_online_params(step, host_rb)
        agent.update_target_params(step)

    ms_drop, _, _, nxt = timed(eng, dropin_step, e2e_steps, args.warmup, nxt)
    dropin_rate = e2e_steps / (ms_drop / 1e3)

    # (2c) strictly serial: H2D, step and D2H of this step's losses one after the other (learn_on_batch returning losses)
    def e2e_sync_step(step):
        eng.learn_host(pool[step % len(pool)], want_losses=True)
        agent.update_target_params(step)

    serial_steps = max(args.steps // 2, 5)
    ms_sync, _, _, nxt = timed(eng, e2e_sync_step, serial_steps, 3, nxt)
    e2e_sync_rate = serial_steps / (ms_sync / 1e3)

    # (2d) configs[4]: the resident step fed by the prioritised sampler -- 1 M-leaf float64 SumTree on the device, new
    # elements inserted at max_recorded_priority, |TD| priorities written back after every step (rb.update)
    prio = None
    if world == 1 and not args.no_prioritized:
        prio = prioritized_leg(agent, frames, timed, eng, args, nxt, local)

    # (3) live per-kernel timing (CUDA events after every launch, un-graphed) for the roofline of the top kernel
    acc = profile_kernels(eng, L)
    kernels_per_step = int(eng.lib.idqn_kernels_per_step(eng.h))  # the replay gather is part of the step's first kernel
    top = max(acc, key=acc.get)
    pk = peaks()
    rl = kernel_roofline(top, acc[top], eng.K, pk)
    rl["traffic"] = None
    try:  # per-launch DRAM bytes of this kernel from the committed ncu --set full capture (K = 5 per GPU)
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            tj = json.load(f)
        if tj.get("source_sha") != source_sha():
            rl["traffic_note"] = "profiles/ncu_traffic.json was captured from other kernel sources: not used"
        elif tj.get(top) and eng.K == HEADS_PER_GPU:
            rl["traffic"] = tj[top]
            rl["algorithmic_bytes"] = int(round(rl["achieved"] * acc[top] * 1e6)) if rl.get("achieved") else None
    except Exception:
        pass
    rl["kernel"] = top
    rl["peak_source"] = pk["src"]
    ctas = int(eng.lib.idqn_dense_update_ctas(eng.h))
    rl["how"] = ("CUDA events around every launch of an un-graphed step (idqn_profile_step), same grids as the graph-replayed step: "
                 + (f"this kernel on {ctas} CTAs, the share of the machine the step gives it" if ctas > 0 else "this kernel on every SM"))
    if ctas > 0 and rl.get("achieved"):
        # the same kernel given the whole machine (how the step ran it before the overlap): its own ceiling
        try:
            ag2 = make_agent(k_total, flags=args.flags)
            L.check(ag2._engine.lib.idqn_set_dense_update_ctas(ag2._engine.h, 0))
            # idqn_profile_step runs the step on whatever the handle's staging buffers hold: give the fresh handle a valid batch
            # first (a never-fed handle's action buffer is uninitialised device memory, and the loss kernel indexes Q with it)
            ag2._engine.learn_host(pool[0], want_losses=True)
            acc2 = profile_kernels(ag2._engine, L)
            rl["whole_machine"] = {"ctas": "all", "us": round(acc2[top] * 1e3, 2), "achieved": rl["achieved"] * acc[top] / acc2[top],
                                   "frac": rl["frac"] * acc[top] / acc2[top]}
            del ag2
        except Exception as e:
            rl["whole_machine"] = {"error": str(e)}
    # ... and what the same kernel does INSIDE the graph-replayed step, where it is given a capped grid and runs next to
    # the conv backward chain (global-timer stamps of its first CTA start / last CTA end, IDQN_F_TIMELINE)
    try:
        rl["in_step"] = in_step_leg(make_agent, k_total, rb, L, top, rl, acc[top])
    except Exception as e:  # the timeline build is diagnostic only
        rl["in_step"] = {"error": str(e)}

    # (4) configs[3]: ONE K=8 chain over the N GPUs (strong scaling), next to K=8 on a single GPU in the same run
    del agent
    strong = strong_k8_leg(make_agent, iDQN, rb, timed, args, world, rank, local, net, L, _map_stack)
    parity = sharded_parity_leg(make_agent, iDQN, net, L, _map_stack, head_partition, world, rank, local, dist) if world > 1 else None

    # (5) the other BASELINE configs on one GPU: us per step
    other = other_configs_leg(iDQN, rb, timed, args, local) if world == 1 and not args.no_other_configs else None

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cpu_rate, cpu_n, cpu_threads = cpu_reference_rate(k_total, min_seconds=10.0, max_steps=60)
            cpu4_rate, cpu4_n, _ = cpu_reference_rate(k_total, min_seconds=6.0, max_steps=30, threads=4)
            cpu = {"value": cpu_rate, "unit": "steps/s", "cores": cpu_threads, "kind": "port",
                   "sample": f"{cpu_n} full learn_on_batch steps (K={k_total}, B=32) of the torch-CPU fp32 oracle, median",
                   "four_threads": {"value": cpu4_rate, "steps": cpu4_n,
                                    "note": "the authors' own Atari i-DQN allocation (launch_job/atari/cluster_idqn.sh:8)"}}
        value = steps_per_s * world  # head-normalised: each rank processes one K=5 agent's worth of heads per step
        out = {
            "metric": METRIC, "value": value, "unit": "steps/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config(world),
            "precision": "fp32 parameters/activations/accumulation; GEMM products as bf16x3 split on tcgen05 "
                         "(losses within 1e-6 of fp64; gradients within 1e-4 given equal relu gates, DESIGN.md §4)",
            "unit_note": "value = chain steps/s x (heads_total / 5); replay store resident in HBM",
            "frames_per_s": value * B * 8, "transitions_per_s": value * B,
            "step_hbm_frac": (BYTES_PER_HEAD_STEP * eng.K + BATCH_BYTES) / (ms / args.steps * 1e-3) / 1e9 / pk["hbm"],
            "step_tflops": FLOP_PER_HEAD_STEP * eng.K / (ms / args.steps * 1e-3) / 1e12,
            "wall_s": wall, "clocks": clocks,
            "e2e": {"value": e2e_rate * world, "unit": "steps/s", "h2d_bytes_per_step": BATCH_BYTES,
                    "d2h_bytes_per_step": 4 * eng.K,
                    "how": "idqn_submit_batch_host / idqn_wait_losses: pinned H2D of step t+1 on a copy stream while "
                           "step t computes, losses of every step read back one step behind (two steps in flight)",
                    "blocking_call_value": dropin_rate * world,
                    "blocking_call_how": "the reference-signature call agent.update_online_params(step, host_replay_buffer) + "
                                         "update_target_params(step): H2D of every batch, losses summed on the device and "
                                         "read at T-updates (idqn.py:72,82-87)",
                    "serial_call_value": e2e_sync_rate * world,
                    "serial_call_how": "idqn_learn_on_batch_host returning the losses: H2D, step, D2H strictly in sequence"},
            "gpu_launches": kernels_per_step * args.steps,
            "roofline": rl, "kernel_ms": {k: round(v, 5) for k, v in acc.items()},
            "strong_k8": strong,
        }
        if parity is not None:
            out["sharded_parity"] = parity
        if other is not None:
            out["other_configs_us_per_step"] = other
        if prio is not None:
            out["prioritized_replay"] = prio
        if cpu is not None:
            out["cpu_baseline"] = cpu
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def in_step_leg(make_agent, k_total, rb, L, top, rl, alone_ms):
    import ctypes as C
    ag = make_agent(k_total, flags=L.F_TIMELINE)
    eng = ag._engine
    kt, names, n = np.zeros(128, np.uint64), np.zeros(64 * 32, np.uint8), C.c_int(0)
    durs, spans = [], []
    for it in range(12):
        ag.update_online_params(1 + it, rb)
        L.check(eng.lib.idqn_kernel_timeline(eng.h, L.ptr(kt), L.ptr(names), 64, C.byref(n)))
        if it < 2:
            continue
        t = kt[:2 * n.value].astype(np.float64).reshape(-1, 2)
        for i in range(n.value):
            nm = bytes(names[32 * i:32 * i + 32]).split(b"\0")[0].decode()
            if nm == top and t[i, 1] > t[i, 0]:
                durs.append((t[i, 1] - t[i, 0]) / 1e3)
        ok = t[:, 1] > 0
        spans.append((t[ok, 1].max() - t[ok, 0].min()) / 1e3)
    ctas = int(eng.lib.idqn_dense_update_ctas(eng.h))
    us = float(np.median(durs))
    out = {"ctas": ctas if ctas > 0 else "all", "us": round(us, 2), "step_span_us": round(float(np.median(spans)), 2)}
    if rl.get("achieved"):
        ach = rl["achieved"] * alone_ms * 1e3 / us
        out.update({"achieved": ach, "frac": ach / rl["peak"],
                    "note": "first CTA start to last CTA end inside the graph, where the conv backward kernels run on the other SMs "
                            "(DESIGN.md section 3): the step is faster with this kernel on part of the machine than alone on all of it"})
    del ag
    return out


def profile_kernels(eng, L, reps=5):
    import ctypes as C
    names_buf, ms_buf, acc = np.zeros(64 * 32, np.uint8), np.zeros(64, np.float32), {}
    for rep in range(reps + 1):
        n = C.c_int(0)
        L.check(eng.lib.idqn_profile_step(eng.h, 1, 64, L.ptr(ms_buf), L.ptr(names_buf), C.byref(n)))
        if rep == 0:
            continue
        for i in range(n.value):
            nm = bytes(names_buf[32 * i:32 * i + 32]).split(b"\0")[0].decode()
            acc[nm] = acc.get(nm, 0.0) + float(ms_buf[i]) / reps
    return acc


def strong_k8_leg(make_agent, iDQN, rb, timed, args, world, rank, local, net, L, _map_stack):
    """BASELINE configs[3]: a K=8 chain sharded ceil(8/N) heads per GPU; chain steps/s (max over ranks) and, measured in
    the same run on rank 0's GPU, the K=8 rate of one GPU."""
    K8 = 8
    if world > K8:
        return {"skipped": f"{world} GPUs > 8 heads"}
    steps = max(args.steps, 100)
    ag = make_agent(K8)

    def step_fn(step):
        ag.update_online_params(step, rb)
        ag.update_target_params(step)

    ms, _, _, _ = timed(ag._engine, step_fn, steps, max(args.warmup, 10), 1)
    chain_rate = steps / (ms / 1e3)
    heads_here = ag._engine.K
    out = {"heads_total": K8, "heads_per_gpu": -(-K8 // world), "chain_steps_per_s": chain_rate, "ms_per_step": ms / steps,
           "timed_steps": steps, "events": "T=200, D=10 (D-sync every 10 steps in the timed window)"}
    del ag
    if world == 1:
        out["single_gpu_k8_steps_per_s"] = chain_rate
        out["speedup"], out["efficiency"] = 1.0, 1.0
        return out
    # the denominator, in the same run: the unsharded K=8 agent on this rank's GPU (rank 0's figure is reported).  Every
    # rank runs it so that the GPUs stay in lockstep for the legs that follow.
    single = iDQN(0, OBS, A, K8, FEATS, "cnn", LR, GAMMA, 1, 1, T_FREQ, D_FREQ, EPS, device=local)
    single._engine.upload_tree(L.TARGET, _map_stack([net.init(1000 + k, np.zeros(OBS, np.float32)) for k in range(K8)]))

    def single_fn(step):
        single.update_online_params(step, rb)
        single.update_target_params(step)

    import torch
    stream = torch.cuda.ExternalStream(int(single._engine.lib.idqn_stream(single._engine.h)), device=f"cuda:{local}")
    for s in range(1, 21):
        single_fn(s)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for s in range(21, 21 + steps):
        single_fn(s)
    e1.record(stream)
    torch.cuda.synchronize()
    single_rate = steps / (e0.elapsed_time(e1) / 1e3)
    del single
    out["single_gpu_k8_steps_per_s"] = single_rate
    out["speedup"] = chain_rate / single_rate
    out["efficiency"] = chain_rate / single_rate / world
    out["heads_on_rank0"] = heads_here
    return out


def sharded_parity_leg(make_agent, iDQN, net, L, _map_stack, head_partition, world, rank, local, dist):
    """The product's sharded K=8 chain (NVLink peer exchange at the D / T events) against the UNSHARDED K=8 agent run on
    this rank's own GPU, same seeds, same batches, 18 steps with T=8 / D=4: losses and all four arenas of this rank's
    heads must be bit-identical (every reduction of the step is grouped independently of the head count)."""
    import torch
    from idqn_b200 import _prng
    K8, T, D, steps = 8, 8, 4, 18
    if world > K8:
        return "skipped"
    sh = make_agent(K8, T=T, D=D)
    start, cnt = head_partition(K8, world)[rank]
    full = iDQN(0, OBS, A, K8, FEATS, "cnn", LR, GAMMA, 1, 1, T, D, EPS, device=local)
    keys = _prng.split(0, K8)
    full._engine.upload_tree(L.ONLINE, _map_stack([full.network.init(k, np.zeros(OBS, np.float32)) for k in keys]))
    full._engine.upload_tree(L.TARGET, _map_stack([net.init(1000 + k, np.zeros(OBS, np.float32)) for k in range(K8)]))
    rng = np.random.default_rng(5)
    bad = 0
    for step in range(1, steps + 1):
        batch = synthetic_batch(rng)
        ls = sh._engine.learn_host(batch, want_losses=True)
        lf = full._engine.learn_host(batch, want_losses=True)
        sh.update_target_params(step)
        full.update_target_params(step)
        bad += int(not np.array_equal(ls, lf[start:start + cnt]))
    for which in (L.ONLINE, L.TARGET, L.MU, L.NU):
        a, b = sh._engine.download_arena(which), full._engine.download_arena(which)[start:start + cnt]
        bad += int(not np.array_equal(a, b))
    t = torch.tensor([bad], device=f"cuda:{local}")
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    total = int(t.item())
    del sh, full
    return "bit-identical" if total == 0 else f"DIFFERENT ({total} mismatching comparisons over all ranks)"


def other_configs_leg(iDQN, rb, timed, args, local):
    """us per gradient step of BASELINE configs[0] (Lunar Lander MLP K=3), [1] (NatureCNN DQN K=1), [2] (NatureCNN K=3)."""
    out = {}
    steps = max(args.steps, 200)
    for name, k in (("configs[1] NatureCNN K=1", 1), ("configs[2] NatureCNN K=3", 3)):
        ag = iDQN(0, OBS, A, k, FEATS, "cnn", LR, GAMMA, 1, 1, T_FREQ, D_FREQ, EPS, device=local)

        def fn(step, ag=ag):
            ag.update_online_params(step, rb)
            ag.update_target_params(step)

        ms, _, _, _ = timed(ag._engine, fn, steps, 10, 1)
        out[name] = round(ms / steps * 1e3, 2)
        del ag
    # Lunar Lander: MLP [100, 100] on 8-dim states, T=200, D=10, host batches (the README example; float32 states)
    ag = iDQN(0, 8, 4, 3, [100, 100], "fc", 3e-4, GAMMA, 1, 1, 200, 10, 1e-8, device=local)
    r = np.random.default_rng(3)
    batches = [dict(state=r.standard_normal((B, 8, 1)).astype(np.float32), next_state=r.standard_normal((B, 8, 1)).astype(np.float32),
                    action=r.integers(0, 4, B).astype(np.int32), reward=r.uniform(-1, 1, B).astype(np.float32),
                    is_terminal=(r.random(B) < 0.05)) for _ in range(4)]

    class Buf:
        i = 0

        def sample(self):
            Buf.i += 1
            return batches[Buf.i % 4]

    buf = Buf()

    def fn_mlp(step):
        ag.update_online_params(step, buf)
        ag.update_target_params(step)

    ms, _, _, _ = timed(ag._engine, fn_mlp, steps, 10, 1)
    out["configs[0] Lunar Lander MLP K=3 (host batches)"] = round(ms / steps * 1e3, 2)
    del ag
    # the reference's third architecture (architectures/dqn.py:7-29,54-60; only its unit tests use it): IMPALA at the Atari
    # sizes, K = 1, on the fp32 CUDA-core kernels -- 52 GFLOP per head-step (13x NatureCNN), not a tuned path
    ag = iDQN(0, OBS, A, 1, FEATS, "impala", LR, GAMMA, 1, 1, T_FREQ, D_FREQ, EPS, device=local)
    ib = [synthetic_batch(np.random.default_rng(40 + i)) for i in range(2)]

    class IBuf:
        i = 0

        def sample(self):
            IBuf.i += 1
            return ib[IBuf.i % 2]

    ibuf = IBuf()

    def fn_impala(step):
        ag.update_online_params(step, ibuf)
        ag.update_target_params(step)

    ms, _, _, _ = timed(ag._engine, fn_impala, 20, 3, 1)
    out["IMPALA K=1 (generic tcgen05 + pool kernels, host batches)"] = round(ms / 20 * 1e3, 2)
    return out


def prioritized_leg(agent, frames, timed, eng, args, nxt, local):
    from idqn_b200.sample_collection.replay_buffer import ReplayBuffer, TransitionElement
    from idqn_b200.sample_collection.samplers import PrioritizedSamplingDistribution
    rb_p = ReplayBuffer(PrioritizedSamplingDistribution(seed=0, max_capacity=1 << 20, priority_exponent=1.0, device=local),
                        batch_size=B, max_capacity=4096, stack_size=4, clipping=lambda r: np.clip(r, -1, 1), device=local)
    rng_p = np.random.default_rng(1)
    wired = hasattr(rb_p, "update_from_learner")
    for t in range(4200):
        kw = {} if wired else {"priority": float(rng_p.random() + 0.1)}
        rb_p.add(TransitionElement(frames[t], int(rng_p.integers(0, A)), float(rng_p.integers(-1, 2)),
                                   bool(rng_p.random() < 0.01), False), **kw)

    def prio_step(step):
        agent.update_online_params(step, rb_p)
        if wired:
            rb_p.update_from_learner(eng)  # rb.update(keys, |TD|) with the priorities the step just produced, on the device
        agent.update_target_params(step)

    p_steps = max(args.steps // 2, 5)
    ms_p, _, _, _ = timed(eng, prio_step, p_steps, 3, nxt)
    return {"value": p_steps / (ms_p / 1e3), "unit": "steps/s", "sum_tree_capacity": 1 << 20,
            "priority_update_in_loop": bool(wired),
            "how": "resident step with PrioritizedSamplingDistribution: host PCG64 uniforms -> device SumTree descent "
                   "(float64, depth 21) -> keys -> replay slots" + ("; per-sample |TD| of the step written back into the tree "
                   "(rb.update) inside the timed loop, new elements inserted at max_recorded_priority" if wired else "")}


def kernel_roofline(name: str, ms: float, k_heads: int, pk):
    """Algorithmic work of one launch of kernel `name` (DESIGN.md "Kernels") over its live-measured duration."""
    mac = {"fwd_L0": 2 * 3_612_672, "fwd_L1": 2 * 3_964_928, "fwd_L2": 2 * 4_460_544, "fwd_L3": 2 * 3_964_928,
           "wgrad_L0": 3_612_672, "wgrad_L1": 3_964_928, "wgrad_L2": 4_460_544, "wgrad_L3": 3_964_928,
           "dgrad_L1": 3_964_928, "dgrad_L2": 4_460_544, "dgrad_L3": 3_964_928}
    base = name
    for prefix in ("tc_", "img_", "dense_"):
        if base.startswith(prefix):
            base = base[len(prefix):]
    tensor_path = base != name
    dense0 = 7744 * 512 + 512
    if base.startswith("wgrad_adam"):
        # reads W, mu, nu and writes W, mu, nu of Dense_0 (+ the 1 MB of activations feeding the outer product)
        gb = (6 * dense0 * 4 + (32 * 7744 + 32 * 512) * 4) * k_heads / 1e9
        ach = gb / (ms * 1e-3)
        return {"bound": "hbm", "achieved": ach, "peak": pk["hbm"], "unit": "GB/s", "frac": ach / pk["hbm"]}
    if base.startswith("adam"):
        n = P_HEAD - (dense0 if base != "adam" else 0)
        gb = 7 * n * 4 * k_heads / 1e9
        ach = gb / (ms * 1e-3)
        return {"bound": "hbm", "achieved": ach, "peak": pk["hbm"], "unit": "GB/s", "frac": ach / pk["hbm"]}
    if base in ("fwd_L3", "dgrad_L3") and tensor_path:
        # weight streaming (M or N = batch 32): bound by reading the 15.9 MB Dense_0 kernel per net
        nets = 2 * k_heads if base == "fwd_L3" else k_heads
        gb = dense0 * 4 * nets / 1e9
        ach = gb / (ms * 1e-3)
        return {"bound": "hbm", "achieved": ach, "peak": pk["hbm"], "unit": "GB/s", "frac": ach / pk["hbm"]}
    if base in mac:
        tf = 2 * mac[base] * B * k_heads / 1e12
        ach = tf / (ms * 1e-3)
        return {"bound": "tensor", "achieved": ach, "peak": pk["tf_sus"], "unit": "TFLOP/s", "frac": ach / pk["tf_sus"]}
    return {"bound": "hbm", "achieved": None, "peak": pk["hbm"], "unit": "GB/s", "frac": None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-prioritized", action="store_true", help="skip the prioritised-replay (configs[4]) leg")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the us/step figures of configs[0..2]")
    ap.add_argument("--flags", type=int, default=0, help="IDQN_F_* engine flags (A/B experiments)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the state the resident path computed as DIR/<name>.npy "
                         "(rank 0's heads), to compare two builds output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the CUDA path computed: it needs --impl ours")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
