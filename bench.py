#!/usr/bin/env python
"""bench.py — UAV env-steps/s of the batched environment step on B200, next to the reference CPU step.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c4s|...] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path (one `uavca_step_*` launch) over one batch of B envs.  Default workload:
BASELINE.json configs[2] at N=1 GPU — multi-UAV, N=8 UAVs per env, B=65,536 envs, random cartesian actions, auto-reset
on dones[0] / 1,500 steps from the on-device Philox stream — and configs[3] when `--gpus` > 1 — N=32, 1,048,576 envs
IN TOTAL, sharded over the GPUs (`c4s`).  Small batches are L2-resident on a B200, so the bench cycles through a ring
of independent batches whose combined footprint exceeds L2 several times over: every timed launch reads its state and
actions from HBM.  Steps are replayed from a CUDA graph and timed with CUDA events: >= 5 repetitions of the K-step
region, each bracketed by events; the line reports the MEDIAN repetition (`value`, `ms_per_step`) and the best one.
Multi-GPU runs are one process per GPU (torchrun), envs sharded with no per-step collective, time = max over ranks.

The JSON line carries
  value        device-resident throughput of the workload (inputs resident in HBM) through the fastest product path for
               open-loop actions: `uavca_rollout`, K env steps per launch from an action block, ONE stream (bit-identical
               to K single steps); `per_step_launch` holds the one-launch-per-step numbers (`--headline per_step` swaps them);
  e2e          the same metric through `uavca_step_host` with pinned HOST buffers: H2D actions + step + D2H
               obs/reward/done inside the timed region, next to the PCIe copy ceiling measured on the same rank;
  roofline     algorithmic bytes per launch / measured launch time against MEASURED_PEAKS.json (+ the same for one
               dependent launch at a time, `frac_single_stream`);
  rollout      both rollout variants (action block / on-device Philox actions: the run_multi.py loop), one stream;
  cpu_baseline the oracle port of the reference step on one host thread, `cpu_baseline_literal` the LITERAL Python
               reference (oracle/_ref, when it travelled) on one core.
`--impl reference` times the reference's CPU algorithm (oracle port, all host threads) on the same workload.
`--workload c1` is BASELINE configs[0] (single-UAV gym loop, 1,000 steps): the literal reference against the B=1
drop-in class.  `--workload c5r` is configs[4]: policy inference + env step + replay append per acting step.
"""
from __future__ import annotations

import argparse
import json
import os
import copy
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: kind, N, B per GPU, default steps
    "c1": dict(kind="single", N=1, B=1, desc="single-UAV gym loop, random actions, 1,000 steps (BASELINE configs[0])", steps=1000, loop=True),
    "c3": dict(kind="multi", N=8, B=65536, desc="multi-UAV N=8, B=65,536 envs/GPU (BASELINE configs[2])", steps=20000),
    "c2": dict(kind="single", N=1, B=65536, desc="single-UAV, B=65,536 envs/GPU (BASELINE configs[1])", steps=20000, streams=4),
    "c4": dict(kind="multi", N=32, B=1048576, desc="multi-UAV N=32, B=1,048,576 envs/GPU (BASELINE configs[3] shape)", steps=300),
    "c4s": dict(kind="multi", N=32, B=1048576, desc="multi-UAV N=32, B=1,048,576 envs IN TOTAL, sharded over the GPUs (BASELINE configs[3])",
                steps=600, shard_total=True),
    "c5": dict(kind="multi", N=10, B=16384, desc="multi-UAV N=10, B=16,384 envs/GPU (BASELINE configs[4] env part)", steps=20000, streams=4),
    "c5r": dict(kind="multi", N=10, B=16384, desc="SAC-style acting step: policy 10-256-256-2 + env step (polar map fused) + replay append, "
                                                   "N=10, B=16,384 envs/GPU (BASELINE configs[4])", steps=2000, acting=True),
}
L2_BYTES = 126e6
GRAPH_STEPS = 200
MIN_REPS, MAX_REPS, LOADED_MS = 5, 400, 60.0  # repetitions of the K-step region; enough of them to sample clocks under load
DUMP_BYTES = 60_000_000  # --dump-outputs writes at most this much (plus .npy headers), under 64 MB


def algorithmic_bytes_per_unit(kind: str, N: int) -> float:
    """SURVEY.md §8d: multi 107 B per UAV-step + 24/N for the per-env counters; single 89 B per env-step."""
    return 89.0 if kind == "single" else 107.0 + 24.0 / N


def rollout_bytes_per_unit(kind: str, N: int, block: bool) -> float:
    """What a K-step rollout has to move per UAV-step (state stays in registers): obs + reward + done (+ the action)."""
    return (16 if kind == "single" else 40) + 4 + 1 + (8 if block else 0)


def footprint_bytes_per_unit(kind: str) -> float:
    # resident bytes per UAV of one batch: state (pos 8, vel 16, tgt 8, init 4, prev 4, flags 1) + io (action 8, obs, reward 4, done 1)
    return 41.0 + 8 + (16 if kind == "single" else 40) + 4 + 1


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---- clocks sampled DURING the timed region ---------------------------------------------------------------------


class ClockSampler:
    REASONS = {
        0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
        0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown",
        0x100: "display_clock_setting",
    }

    def __init__(self, index: int, period_s: float = 0.004):
        self.index, self.period = index, period_s
        self.sm, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.sm.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                bits = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for b, name in self.REASONS.items():
                    if bits & b and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def __enter__(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thread:
            self._thread.join()

    def summary(self):
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unsampled"]}
        s = sorted(self.sm)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s),
                "sampled": "during the timed repetitions"}


# ---- CPU side ---------------------------------------------------------------------------------------------------


def time_oracle(kind: str, N: int, envs: int, steps: int, nthreads: int, seed: int = 0):
    """UAV-steps/s of oracle/uav_oracle.c (the restated reference step) on `nthreads` host threads."""
    import numpy as np

    from oracle import oracle as O

    if kind == "single":
        cfg = O.single_config(envs, reset_mode=O.RESET_ON_ANY_DONE, max_episode_steps=1500, seed=seed)
        amax = 12.0
    else:
        cfg = O.multi_config(envs, N, reset_mode=O.RESET_ON_DONE0, max_episode_steps=1500, seed=seed)
        amax = 10.0
    orc = O.Oracle(cfg, nthreads=nthreads)
    orc.reset()
    rng = np.random.default_rng(seed)
    acts = [rng.uniform(-amax, amax, size=(envs, N, 2)).astype(np.float32) for _ in range(4)]
    orc.step(acts[0])
    t0 = time.perf_counter()
    for k in range(steps):
        orc.step(acts[k % 4])
    dt = time.perf_counter() - t0
    return envs * N * steps / dt, dt


def time_literal(kind: str, N: int, steps: int, repeats: int = 3):
    """The LITERAL Python reference on one core (BASELINE.md §5 item 1): the run.py / run_multi.py loop — random
    actions, reset on done (dones[0] for the multi world), np.random.seed(0), best of `repeats`.  Returns
    (UAV-steps/s, seconds of the best repeat) or None where neither /root/reference nor oracle/_ref exists."""
    import numpy as np

    from oracle import ref_loader as R

    if not R.reference_available():
        return None
    UAVWorld2D, MultiUAVWorld2D = R.load_reference()
    best = None
    for _ in range(repeats):
        np.random.seed(0)
        env = UAVWorld2D() if kind == "single" else MultiUAVWorld2D(num_agents=N)
        env.reset()
        if kind == "single":
            acts = [env.action_space.sample() for _ in range(steps)]
        else:
            acts = [[np.random.uniform(-10, 10, 2).astype(np.float32) for _ in range(N)] for _ in range(steps)]
        t0 = time.perf_counter()
        for a in acts:
            _, _, done, _ = env.step(a)
            if done if kind == "single" else done[0]:
                env.reset()
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return N * steps / best, best


def cpu_model() -> str:
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def workload_config(args, wl, world, B_per_gpu):
    """The part of `config` both arms share (the driver compares it)."""
    return {"workload": wl["desc"], "uavs_per_env": wl["N"], "envs_per_gpu": B_per_gpu, "envs_total": B_per_gpu * world if not wl.get("shard_total") else wl["B"],
            "actions": "uniform random cartesian", "auto_reset": "dones[0] or 1500 steps"}


def shard_envs(wl, rank, world):
    if wl.get("shard_total"):
        from gym_uav_collision_avoidance_b200 import sharding as _sh

        return _sh.shard_range(wl["B"], rank, world)[1]
    return wl["B"]


def literal_baseline(kind, N):
    """cpu_baseline_literal: a bounded sample (~3-10 s) of the literal reference, or why it is absent."""
    steps = 1000 if kind == "single" else max(20, int(4000 // (N * N // 8 + 1)))
    try:
        res = time_literal(kind, N, steps, repeats=2)
    except Exception as exc:  # noqa: BLE001
        return {"unavailable": f"literal reference failed to run: {exc!r}"[:200]}
    if res is None:
        return {"unavailable": "oracle/_ref was not built (python -m oracle.build_ref needs /root/reference)"}
    ups, dt = res
    return {"value": ups, "unit": "UAV env-steps/s", "cores": 1, "kind": "reference",
            "sample": f"1 env x {N} UAVs x {steps} steps, the run.py / run_multi.py loop on the unmodified reference env "
                      f"(oracle/_ref), best of 2 ({dt:.2f} s)"}


def run_reference(args, wl, rank, world):
    """--impl reference: the reference's CPU algorithm for the path on all host threads (oracle port: the Python
    reference is single-threaded and ~300x slower; it is reported beside it as `cpu_baseline_literal`)."""
    if rank != 0:
        return
    from oracle import oracle as O

    steps, warm = max(1, args.steps), max(0, args.warmup)
    unit = "UAV env-steps/s"
    if wl.get("loop"):  # c1: the literal reference itself, one core (it is single-threaded)
        lit = time_literal("single", 1, steps if args.steps else 1000, repeats=3)
        if lit is None:
            emit({"impl": "reference", "unavailable": "oracle/_ref missing: the literal reference did not travel"})
            return
        ups, dt = lit
        emit({"impl": "reference", "metric": "UAV env-steps/sec", "value": ups, "unit": unit, "n_gpus": args.gpus, "steps": steps,
              "warmup": args.warmup, "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
              "dtype": "f64/f32 mixed (as the reference)", "data": "synthetic",
              "config": dict(workload_config(args, wl, 1, 1), host_cpu=cpu_model()),
              "cpu_baseline": {"value": ups, "unit": unit, "cores": 1, "kind": "reference",
                               "sample": f"UAVWorld2D, {steps} steps of the run.py loop, np.random.seed(0), best of 3"},
              "e2e": {"value": ups, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0})
        return
    nthreads = O.max_threads()
    B = shard_envs(wl, 0, max(1, args.gpus))
    envs = min(B, 131072 if wl["N"] >= 16 else B)  # the full per-GPU batch; N=32 is bounded to the 8-GPU shard size
    steps = min(steps, 200)
    time_oracle(wl["kind"], wl["N"], envs, max(1, min(warm, 3)), nthreads)
    ups, dt = time_oracle(wl["kind"], wl["N"], envs, steps, nthreads)
    sample = (f"{envs} envs x {wl['N']} UAVs x {steps} steps of the {args.workload} workload "
              f"(oracle/uav_oracle.c, persistent pool of {nthreads} pthreads)")
    line = {
        "impl": "reference", "metric": "UAV env-steps/sec", "value": ups, "unit": unit, "n_gpus": args.gpus,
        "steps": steps, "warmup": args.warmup, "ms_per_step": dt / steps * 1e3, "higher_is_better": True,
        "scaling": "strong" if wl.get("shard_total") else "weak", "vs_baseline": None, "dtype": "f64/f32 mixed (as the reference)", "data": "synthetic",
        "config": dict(workload_config(args, wl, max(1, args.gpus), B), envs_per_step=envs, host_cpu=cpu_model(), host_threads=nthreads),
        "cpu_baseline": {"value": ups, "unit": unit, "cores": nthreads, "kind": "port", "sample": sample},
        "cpu_baseline_literal": literal_baseline(wl["kind"], wl["N"]),
        "e2e": {"value": ups, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ---- host topology (e2e) ------------------------------------------------------------------------------------------


def gpu_numa_node(index: int):
    try:
        import pynvml

        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(index)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        for cand in (bus.lower(), bus.lower()[4:] if len(bus) > 12 else bus.lower()):
            p = f"/sys/bus/pci/devices/{cand}/numa_node"
            if os.path.exists(p):
                return int(open(p).read().strip())
    except Exception:
        pass
    return None


def bind_to_gpu_numa_node(index: int) -> dict:
    """Pin this rank to the CPUs of its GPU's NUMA node (pinned host buffers are then allocated next to the GPU's PCIe
    root instead of all ranks sharing one socket's memory).  Best effort; reports what happened."""
    info = {"gpu_numa_node": gpu_numa_node(index), "cpu_affinity_before": len(os.sched_getaffinity(0))}
    node = info["gpu_numa_node"]
    if node is None or node < 0:
        info["bound"] = False
        return info
    try:
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        os.sched_setaffinity(0, cpus)
        info["bound"] = True
        info["cpus"] = len(cpus)
    except Exception as exc:  # noqa: BLE001  (cpuset of the container may not include that node)
        info["bound"] = False
        info["why"] = repr(exc)[:120]
    return info


# ---- GPU side ---------------------------------------------------------------------------------------------------


def timed_reps(torch, stream, replay_fn, est_ms, dev, barrier):
    """>= MIN_REPS repetitions of `replay_fn` (one K-step region), each bracketed by CUDA events on `stream`; enough of
    them to keep the GPU loaded for LOADED_MS so that the clock sampler sees the timed region.  Returns per-rep ms."""
    reps = int(min(MAX_REPS, max(MIN_REPS, LOADED_MS / max(est_ms, 1e-3))))
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
    barrier()
    with torch.cuda.stream(stream):
        evs[0].record(stream)
        for i in range(reps):
            replay_fn()
            evs[i + 1].record(stream)
    stream.synchronize()
    barrier()
    return [evs[i].elapsed_time(evs[i + 1]) for i in range(reps)]


def run_ours(args, wl, rank, world, local_rank):
    import torch

    import gym_uav_collision_avoidance_b200 as G
    from gym_uav_collision_avoidance_b200 import sharding

    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    topo = bind_to_gpu_numa_node(local_rank) if not args.no_numa_bind else {"bound": False, "why": "--no-numa-bind"}
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    if wl.get("loop"):
        return run_c1(args, wl, G, torch, dev)
    if wl.get("acting"):
        return run_acting(args, wl, G, torch, dev, rank, world, dist, barrier)

    kind, N = wl["kind"], wl["N"]
    B = shard_envs(wl, rank, world)
    K, W = args.steps, max(args.warmup, 3)
    units_per_step = B * N
    # ring of independent batches: combined footprint > 3x L2 so that every launch streams from HBM
    per_batch = units_per_step * footprint_bytes_per_unit(kind)
    ring = max(1, int(-(-3.2 * L2_BYTES // per_batch)))
    S = max(1, min(args.streams, ring))
    if ring > 1 and ring % S:
        ring += S - ring % S  # every stream serves the same number of batches (no idle stream at the end of a ring cycle)
    amax = 12.0 if kind == "single" else 10.0
    envs = []
    for r in range(ring):
        kw = dict(device=dev, seed=0x5EED, max_episode_steps=1500, env_index_base=(rank * ring + r) * B)
        if kind == "single":
            e = G.BatchedUAVWorld2D(B, reset_mode=G.RESET_ON_ANY_DONE, **kw)
        else:
            e = G.BatchedMultiUAVWorld2D(B, num_agents=N, reset_mode=G.RESET_ON_DONE0, **kw)
        e.reset()
        envs.append(e)
    n_act = max(ring, min(32, int(2e9 // (units_per_step * 8))))
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    actions = [(torch.rand((B, N, 2), generator=gen, device=dev) * 2 - 1) * amax for _ in range(n_act)]

    def one_step(k):
        envs[k % ring].step(actions[(k + k // ring) % n_act])

    def launches():
        return sum(e.launch_count for e in envs)

    # The batches of the ring are independent environments: like a double-buffered env pool they are pipelined over
    # `S` streams, so that one batch's ramp-up overlaps the previous batch's tail.  A batch always runs on the same
    # stream (its own steps stay ordered).  S=1 (--streams 1) serialises every launch behind the previous one.
    for k in range(W):
        one_step(k)
    torch.cuda.synchronize(dev)
    stream = torch.cuda.Stream(device=dev)

    def capture(n, k0, n_streams):
        side = [torch.cuda.Stream(device=dev) for _ in range(n_streams - 1)]
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=stream):
            fork = torch.cuda.Event()
            fork.record(stream)
            for s_ in side:
                s_.wait_event(fork)
            for k in range(n):
                lane = ((k0 + k) % ring) % n_streams
                with torch.cuda.stream(stream if lane == 0 else side[lane - 1]):
                    one_step(k0 + k)
            for s_ in side:
                join = torch.cuda.Event()
                join.record(s_)
                stream.wait_event(join)
        return g

    def graphs_for(n_streams):
        """Graphs replaying exactly K steps: q replays of a GRAPH_STEPS-step graph + one graph of the remainder."""
        q, rem = divmod(K, GRAPH_STEPS)
        g_main = capture(GRAPH_STEPS, W, n_streams) if q > 0 else None
        g_rem = capture(rem, W + GRAPH_STEPS, n_streams) if rem > 0 else None
        for g in (g_main, g_rem):
            if g is not None:
                g.replay()  # graph warm-up (upload)
        torch.cuda.synchronize(dev)

        def replay():
            for _ in range(q):
                g_main.replay()
            if g_rem is not None:
                g_rem.replay()
        return replay, (g_main, g_rem)

    # launches of ours per K-step region: one kernel per step (a batch whose ragged rest needs its own launch has two)
    l0 = launches()
    one_step(0)
    torch.cuda.synchronize(dev)
    per_region_launches = (launches() - l0) * K
    est_ms = units_per_step * algorithmic_bytes_per_unit(kind, N) / 3.5e12 * 1e3 * K  # rough, only sizes the repetition count

    # one stream: every launch waits for the previous one (what a single env pool with a policy between steps sees)
    replay1, keep1 = graphs_for(1)
    with ClockSampler(local_rank) as clocks1:
        t1 = timed_reps(torch, stream, replay1, est_ms, dev, barrier)
    del keep1
    # S streams: independent batches in flight
    if S > 1:
        replayS, keepS = graphs_for(S)
        with ClockSampler(local_rank) as clocks:
            tS = timed_reps(torch, stream, replayS, est_ms, dev, barrier)
        del keepS
    else:
        tS, clocks = t1, clocks1
    dump = args.dump_outputs if rank == 0 else None
    per_step_out = None
    if dump:  # the batch that took the last step of the timed graphs (graphs_for: steps W .. W+199, then the remainder)
        e = envs[(W + GRAPH_STEPS - 1 + K % GRAPH_STEPS) % ring]
        last = dict(obs=e.obs, reward=e.reward, done=e.done)
        if kind == "single":
            last["distance"] = e.distance
        per_step_out = output_sample(last)

    def reduce_reps(ts):
        ts = [sharding.max_over_ranks(t, device=dev) for t in ts] if dist is not None else ts
        return statistics.median(ts), min(ts), len(ts)

    ms_med, ms_best, n_reps = reduce_reps(tS)
    ms1_med, ms1_best, n_reps1 = reduce_reps(t1)
    gpu_launches = per_region_launches * (n_reps + (n_reps1 if S > 1 else 0))
    per_step_value = world * units_per_step * K / (ms_med * 1e-3)

    # ---- K steps per launch (uavca_rollout), ONE stream: an action block resident in HBM, and on-device Philox actions
    rollout = rollout_out = None
    if not args.no_rollout:
        rollout = measure_rollout(torch, G, envs, ring, kind, N, B, amax, dev, stream, barrier, reduce_reps, world, args.rollout_k, K,
                                  local_rank, keep_last=dump is not None)
        if rollout is not None:
            gpu_launches += rollout.pop("_launches")
            rollout_out = rollout.pop("_last", None)
    headline_rollout = rollout is not None and args.headline == "rollout"
    if dump:
        write_outputs(dump, rollout_out if headline_rollout else per_step_out)

    # ---- BASELINE configs[4] beside it (one GPU, default workload only): policy + env step + replay append per acting step
    acting = None
    if world == 1 and args.workload == "c3" and not args.no_acting:
        a_wl = WORKLOADS["c5r"]
        rows, a_launches, _ = measure_acting(args, G, torch, dev, rank, world, dist, barrier, a_wl["B"], a_wl["N"],
                                             max(2, min(K, 400) // 2 * 2))
        acting = {"workload": a_wl["desc"], "rows": rows,
                  "what": "us per acting step and UAV env-steps/s; fp32 = eager PyTorch policy in the reference's arithmetic, "
                          "fused = uavca_policy_act (one tcgen05 kernel, fp16 operands / fp32 accumulate)"}
        gpu_launches += a_launches

    # ---- end to end through the host-buffer C-ABI call (uavca_step_host): pinned host buffers, H2D + step + D2H
    D = 4 if kind == "single" else 10
    h_act = [torch.empty((B, N, 2), dtype=torch.float32).pin_memory() for _ in range(2)]
    for h, a in zip(h_act, actions):
        h.copy_(a.cpu())
    h_obs = torch.empty((B, N, D), dtype=torch.float32).pin_memory()
    h_rew = torch.empty((B, N), dtype=torch.float32).pin_memory()
    h_done = torch.empty((B, N), dtype=torch.uint8).pin_memory()
    e2e_steps = max(1, min(K, 200 if units_per_step < 4e6 else 20))
    e2e_ring = min(ring, 4)  # PCIe-bound: L2 residency is irrelevant here; keep the lazily created staging small
    for k in range(2 * e2e_ring):
        envs[k % e2e_ring].step_host(h_act[k % 2], h_obs, h_rew, h_done)
    l0 = launches()
    e2e_times = []
    for _ in range(3):
        barrier()
        t0 = time.perf_counter()
        for k in range(e2e_steps):
            envs[k % e2e_ring].step_host(h_act[k % 2], h_obs, h_rew, h_done)
        torch.cuda.synchronize(dev)
        e2e_times.append(sharding.max_over_ranks(time.perf_counter() - t0, device=dev))
    e2e_s = statistics.median(e2e_times)
    e2e_value = world * units_per_step * e2e_steps / e2e_s
    gpu_launches += launches() - l0
    # the PCIe ceiling of this rank, measured the same way: one pinned D2H copy of a step's outputs + the H2D of its actions
    d2h_bytes, h2d_bytes = units_per_step * (D * 4 + 4 + 1), units_per_step * 8
    pcie = measure_pcie(torch, dev, envs[0], h_obs, h_act[0], actions[0], barrier, sharding)

    # episode statistics: the only collective of the path (NCCL all-reduce of 4 counters, outside the timed region)
    local = dict.fromkeys(sharding.STAT_KEYS, 0)
    for e in envs:
        s = e.stats()
        for k in sharding.STAT_KEYS:
            local[k] += s[k]
    stats = sharding.reduce_stats(local, device=dev)
    topos = gather_objects(dist, topo, world)

    # strong-scaling workloads (configs[3]): the SAME total workload on ONE GPU, measured by rank 0 alone while the other
    # ranks wait — the N=1 bench line is a different workload (configs[2]), so this is the number to scale against
    one_gpu = None
    if wl.get("shard_total") and world > 1 and not args.no_rollout:
        for e in envs:
            e.close()
        envs.clear()
        torch.cuda.empty_cache()
        if rank == 0:
            try:
                one_gpu = measure_one_gpu_total(torch, G, wl, dev, amax, args.headline)
            except Exception as exc:  # noqa: BLE001
                one_gpu = {"unavailable": repr(exc)[:200]}
        barrier()

    if rank == 0:
        peak, peak_src = measured_peaks()
        alg = algorithmic_bytes_per_unit(kind, N)
        serial_us = ms1_med / K * 1e3
        step_us = ms_med / K * 1e3
        per_step = {
            "what": "one uavca_step_* launch per env step (closed-loop capable: the caller sees every observation before it acts)",
            "value": per_step_value, "us_per_step": step_us, "streams": S,
            "pipelining": (f"independent batches of the ring pipelined over {S} streams (a batch's own steps stay ordered)"
                           if S > 1 else "none: every launch waits for the previous one"),
            "frac": units_per_step * alg / (step_us * 1e-6) / 1e9 / peak,
            "frac_best_rep": units_per_step * alg / (ms_best * 1e-3 / K) / 1e9 / peak, "repetitions": n_reps,
            "single_stream_us_per_step": serial_us, "single_stream_value": world * units_per_step * K / (ms1_med * 1e-3),
            "frac_single_stream": units_per_step * alg / (serial_us * 1e-6) / 1e9 / peak,
            "clocks": clocks.summary(),
        }
        if headline_rollout:
            hb = rollout["block"]
            value, ms_step, head_clocks = hb["value"], hb["us_per_step"] / 1e3, hb["clocks"]
            units_per_launch = units_per_step * rollout["steps_per_launch"]
            path = (f"uavca_rollout: {rollout['steps_per_launch']} env steps per launch, actions from a [K,B,N,2] block resident in HBM, "
                    "per-step obs/reward/done written to [K,...] blocks; ONE stream (every launch waits for the previous one); "
                    "bit-identical to one uavca_step_* launch per step (tests/test_rollout_gpu.py), whose numbers are in `per_step_launch`")
            n_head_reps, frac_best = hb["repetitions"], hb["frac_best_rep"]
            l2 = (f"ring of {ring} independent batches; per launch the state is read once and {rollout['steps_per_launch']} steps of actions / "
                  f"outputs ({units_per_launch * 53 / 1e6:.0f} MB > L2) stream through HBM")
        else:
            value, ms_step, head_clocks = per_step_value, ms_med / K, clocks.summary()
            units_per_launch, path, n_head_reps, frac_best = units_per_step, per_step["what"] + "; " + per_step["pipelining"], n_reps, per_step["frac_best_rep"]
            l2 = f"ring of {ring} independent batches ({ring * per_batch / 1e6:.0f} MB > L2) so every launch streams from HBM"
        launch_s = ms_step * 1e-3 * (units_per_launch / units_per_step)
        achieved = units_per_launch * alg / launch_s / 1e9
        cpu = lit = None
        if not args.no_cpu_baseline and world == 1:  # reported baselines, timed on rank 0 at N=1 only
            c_envs = min(B, 4096 if N <= 8 else 512)
            c_steps = max(20, int(12e6 // (c_envs * N)))
            ups, dt = time_oracle(kind, N, c_envs, c_steps, 1)
            cpu = {"value": ups, "unit": "UAV env-steps/s", "cores": 1, "kind": "port",
                   "sample": f"{c_envs} envs x {N} UAVs x {c_steps} steps of the same workload, oracle/uav_oracle.c on 1 thread "
                             f"({dt:.1f} s; host: {cpu_model()}, {os.cpu_count()} logical cores)"}
            lit = literal_baseline(kind, N)
        traffic = None  # DRAM bytes per launch of the headline kernel, from the ncu captures under profiles/
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as f:
                tj = json.load(f)
            if headline_rollout:  # recorded per UAV-step (a launch's byte count scales with its K)
                per_unit = tj.get(f"rollout_{kind}_n{N}_bytes_per_unit")
                traffic = per_unit * units_per_launch if per_unit else None
            else:
                traffic = tj.get(args.workload)
        e2e_bytes_s = e2e_value / world * (D * 4 + 4 + 1 + 8)
        line = {
            "metric": "UAV env-steps/sec", "value": value, "unit": "UAV env-steps/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong" if wl.get("shard_total") else "weak",
            "vs_baseline": None, "dtype": "f64 velocity / f32 position+obs (as the reference)", "data": "synthetic",
            "config": dict(workload_config(args, wl, world, B), env_steps_per_s=value / N, path=path,
                           actions_resident="in HBM", auto_reset_source="on-device Philox", l2=l2,
                           timing=f"CUDA events around each of {n_head_reps} repetitions of the {K}-step region; value = median repetition",
                           parallelism=f"env-sharded x{world}, no per-step collective", repetitions=n_head_reps,
                           one_gpu_same_workload=one_gpu),
            "e2e": {"value": e2e_value, "unit": "UAV env-steps/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                    "steps": e2e_steps, "host_gbs_per_gpu": e2e_bytes_s / 1e9, "pcie_ceiling": pcie,
                    "frac_of_pcie_ceiling": (e2e_bytes_s / 1e9) / pcie["duplex_gbs"] if pcie and pcie.get("duplex_gbs") else None,
                    "host_topology": topos,
                    "path": "one uavca_step_host call per env step on the caller's stream, pinned host buffers: outputs >= 256 MB leave by DMA "
                            "(chunked H2D/step/D2H pipeline over two streams), smaller batches are zero-copy (the kernel reads/writes mapped "
                            "host memory through PCIe)" + (f" [forced: {os.environ['UAVCA_HOST_PATH']}]" if os.environ.get("UAVCA_HOST_PATH") else "")},
            "gpu_launches": int(gpu_launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_unit": alg,
                         "units_per_launch": units_per_launch, "launch_us": launch_s * 1e6,
                         "kernel": ("rollout_multi_kernel" if kind == "multi" else "rollout_single_kernel") if headline_rollout
                                   else ("step_multi_kernel" if kind == "multi" else "step_single_kernel"),
                         "frac_best_rep": frac_best,
                         "frac_of_bytes_moved": rollout["block"]["frac_of_bytes_moved"] if headline_rollout else None,
                         "bytes_moved_per_unit": rollout["block"]["bytes_moved_per_unit"] if headline_rollout else None,
                         "note": (rollout["frac_is"] if headline_rollout else None),
                         "frac_per_step_launch": per_step["frac"], "frac_single_stream": per_step["frac_single_stream"]},
            "per_step_launch": per_step,
            "rollout": rollout,
            "acting_c5r": acting,
            "cpu_baseline": cpu,
            "cpu_baseline_literal": lit,
            "clocks": head_clocks,
            "episode_stats": stats,
        }
        emit(line)
    if dist is not None:
        dist.destroy_process_group()


def measure_one_gpu_total(torch, G, wl, dev, amax, headline):
    """The whole strong-scaling workload (all wl["B"] envs) on one GPU through the headline path: UAV env-steps/s."""
    B, N = wl["B"], wl["N"]
    env = G.BatchedMultiUAVWorld2D(B, num_agents=N, reset_mode=G.RESET_ON_DONE0, max_episode_steps=1500, seed=0x5EED, device=dev)
    env.reset()
    M = B * N
    reps = 5
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if headline == "rollout":
        Kr = int(max(1, min(4, 12e9 // (2 * M * 45))))
        acts = (torch.rand((Kr, B, N, 2), device=dev) * 2 - 1) * amax
        out = env.rollout(Kr, acts, sync_last=False)
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(reps):
            env.rollout(Kr, acts, out=out, sync_last=False)
        e1.record()
        steps = reps * Kr
        path = f"uavca_rollout, {Kr} steps per launch, action block"
    else:
        acts = (torch.rand((B, N, 2), device=dev) * 2 - 1) * amax
        for _ in range(3):
            env.step(acts)
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(4 * reps):
            env.step(acts)
        e1.record()
        steps = 4 * reps
        path = "one launch per step"
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1)
    env.close()
    return {"n_gpus": 1, "envs": B, "value": M * steps / (ms * 1e-3), "us_per_step": ms * 1e3 / steps, "path": path,
            "what": "the same total workload on ONE GPU (rank 0 alone, the other ranks idle), for the strong-scaling ratio"}


def gather_objects(dist, obj, world):
    if dist is None:
        return [obj]
    out = [None] * world
    dist.all_gather_object(out, obj)
    return out


def measure_pcie(torch, dev, env, h_obs, h_act, d_act, barrier, sharding):
    """Pinned D2H of one step's observation block and pinned H2D of its actions, alone and together (GB/s, this rank,
    max time over ranks: all ranks copy at once, as in the e2e leg)."""
    try:
        d_obs = env.obs
        s1, s2 = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
        reps = max(3, int(2e9 // max(1, h_obs.numel() * 4)))
        reps = min(reps, 200)

        def run(d2h, h2d):
            barrier()
            t0 = time.perf_counter()
            for _ in range(reps):
                if d2h:
                    with torch.cuda.stream(s1):
                        h_obs.copy_(d_obs, non_blocking=True)
                if h2d:
                    with torch.cuda.stream(s2):
                        d_act.copy_(h_act, non_blocking=True)
            torch.cuda.synchronize(dev)
            return sharding.max_over_ranks(time.perf_counter() - t0, device=dev) / reps

        run(True, True)
        t_d2h, t_h2d, t_both = run(True, False), run(False, True), run(True, True)
        b_d2h, b_h2d = h_obs.numel() * 4, h_act.numel() * 4
        return {"d2h_gbs": b_d2h / t_d2h / 1e9, "h2d_gbs": b_h2d / t_h2d / 1e9, "duplex_gbs": (b_d2h + b_h2d) / t_both / 1e9,
                "how": f"cudaMemcpyAsync of one step's observations ({b_d2h / 1e6:.0f} MB, D2H) and actions ({b_h2d / 1e6:.0f} MB, H2D) "
                       f"between pinned host memory and HBM, {reps} repetitions, every rank at once"}
    except Exception as exc:  # noqa: BLE001
        return {"unavailable": repr(exc)[:160]}


def measure_rollout(torch, G, envs, ring, kind, N, B, amax, dev, stream, barrier, reduce_reps, world, Kr, K, local_rank,
                    keep_last=False):
    """`uavca_rollout` on ONE stream: a repetition is exactly K env steps, done as launches of Kr steps (+ one launch of
    the remainder), each launch on the next batch of the ring (every launch finds its state in HBM, not in L2); the
    [Kr, ...] output blocks (>> L2) are shared by the batches.  Two variants: actions from an action block resident in
    HBM, and on-device Philox actions (the run_multi.py loop).  `keep_last`: `_last` holds the `output_sample` of the
    last step of the action-block variant."""
    M = B * N
    if kind != "single" and (M * 10 * 4) % 16:
        return None
    out_bytes = M * ((4 if kind == "single" else 10) * 4 + 4 + 1)
    Kr = int(max(1, min(Kr, K, 12e9 // (2 * out_bytes))))
    q, rem = divmod(K, Kr)
    res = {"steps_per_launch": Kr, "launches_per_rep": q + (1 if rem else 0), "_launches": 0, "streams": 1}
    outs = [envs[0].rollout(Kr, None, action_seed=1, step0=0, sync_last=False) for _ in range(2)]
    outs_rem = [{k: v[:rem] for k, v in o.items()} for o in outs] if rem else None
    n_blocks = int(max(1, min(4, 3e9 // (Kr * M * 8))))
    gen = torch.Generator(device=dev).manual_seed(99)
    blocks = [(torch.rand((Kr, B, N, 2), generator=gen, device=dev) * 2 - 1) * amax for _ in range(n_blocks)]
    peak, _ = measured_peaks()
    alg = algorithmic_bytes_per_unit(kind, N)
    for name in ("philox", "block"):
        state = {"t": 0, "j": 0}

        def rep(name=name):
            for i in range(q + (1 if rem else 0)):
                k = Kr if i < q else rem
                j = state["j"]
                acts = None if name == "philox" else blocks[j % n_blocks][:k]
                o = (outs if i < q else outs_rem)[j % 2]
                envs[j % ring].rollout(k, acts, action_seed=1, step0=state["t"], out=o, sync_last=False)
                state["t"] += k
                state["j"] = j + 1
                state["last"] = (o, k)

        with torch.cuda.stream(stream):
            rep()
        torch.cuda.synchronize(dev)
        est_ms = K * M * 45 / 3.0e12 * 1e3
        with ClockSampler(local_rank) as clocks:
            ts = timed_reps(torch, stream, rep, est_ms, dev, barrier)
        if keep_last and name == "block":
            o, k = state["last"]
            res["_last"] = output_sample({key: v[k - 1] for key, v in o.items()})
        med, best, n = reduce_reps(ts)
        us_per_step = med * 1e3 / K
        moved = rollout_bytes_per_unit(kind, N, name == "block")
        res[name] = {"us_per_step": us_per_step, "ms_per_rep": med, "value": world * M / us_per_step * 1e6,
                     "best_us_per_step": best * 1e3 / K, "frac": M * alg / (us_per_step * 1e-6) / 1e9 / peak,
                     "frac_best_rep": M * alg / (best * 1e3 / K * 1e-6) / 1e9 / peak,
                     "bytes_moved_per_unit": moved, "frac_of_bytes_moved": M * moved / (us_per_step * 1e-6) / 1e9 / peak,
                     "repetitions": n, "clocks": clocks.summary()}
        res["_launches"] += (q + (1 if rem else 0)) * (n + 1)
    res["frac_is"] = (f"SURVEY 8d algorithmic bytes of a step ({alg:g} B per UAV-step) x UAV-steps of the launch / launch time / peak — the "
                      "contract's definition; the env state stays in registers for the K steps of a launch, so only obs/reward/done (+ the "
                      "action block) really cross HBM (`bytes_moved_per_unit`, `frac_of_bytes_moved`): the kernel is instruction-issue bound")
    del outs, blocks
    return res


def run_c1(args, wl, G, torch, dev):
    """BASELINE configs[0]: the run.py loop through the B=1 drop-in class (`compat.UAVWorld2D`): one env, one step per
    call, python floats back on the host every step — latency, not throughput."""
    import numpy as np

    from gym_uav_collision_avoidance_b200 import compat

    K = args.steps
    best = None
    launches = 0
    for _ in range(3):
        np.random.seed(0)
        env = compat.UAVWorld2D()
        env.reset()
        acts = [env.action_space.sample() for _ in range(K)]
        l0 = env._b.launch_count
        t0 = time.perf_counter()
        for a in acts:
            obs, reward, done, info = env.step(a)
            if done:
                env.reset()
        dt = time.perf_counter() - t0
        launches = env._b.launch_count - l0
        best = dt if best is None else min(best, dt)
    if args.dump_outputs:
        write_outputs(args.dump_outputs, output_sample(dict(obs=obs[None], reward=np.array([reward]), done=np.array([done], np.float32),
                                                            distance=np.array([info["distance"]]))))
    lit = literal_baseline("single", 1) if not args.no_cpu_baseline else None
    emit({"metric": "UAV env-steps/sec", "value": K / best, "unit": "UAV env-steps/s", "n_gpus": 1, "steps": K, "warmup": args.warmup,
          "ms_per_step": best / K * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
          "dtype": "f64 velocity / f32 position+obs (as the reference)", "data": "synthetic",
          "config": dict(workload_config(args, wl, 1, 1), note="one env, one launch + one host read-back per step: launch/sync latency bound; "
                         "the batched classes are the product, this row only shows the drop-in runs the reference's own loop"),
          "e2e": {"value": K / best, "unit": "UAV env-steps/s", "h2d_bytes_per_step": 8, "d2h_bytes_per_step": 4 * 4 + 4 + 1},
          "gpu_launches": int(launches), "roofline": None, "cpu_baseline": lit, "cpu_baseline_literal": lit})


def measure_acting(args, G, torch, dev, rank, world, dist, barrier, B, N, K, keep_row=None):
    """BASELINE configs[4]: one acting step = policy forward over all B*N observations + env step (polar action map
    fused) + append of the B*N transitions to the device replay ring.  Rows: eager fp32 (the reference's arithmetic),
    TF32, and the fused tcgen05 acting kernel.  A repetition is K acting steps (K even: the rollout ping-pongs two
    observation buffers, so every CUDA graph holds an even number of steps).  Returns (rows, launches of ours, the
    `output_sample` of the last step of row `keep_row` or None)."""
    from gym_uav_collision_avoidance_b200 import sharding

    torch.manual_seed(0)
    tf32_before = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    rows = {}
    stream = torch.cuda.Stream(device=dev)
    total_launches = 0
    kept = None
    for row in ("fp32", "tf32", "fused", "fused_separate_append"):
        precision = "fused" if row.startswith("fused") else row
        env = G.BatchedMultiUAVWorld2D(B, num_agents=N, reset_mode=G.RESET_ON_DONE0, max_episode_steps=1500, seed=0x5EED,
                                       env_index_base=rank * B, device=dev)
        policy = G.GaussianPolicy(10, 2).to(dev)
        replay = G.DeviceReplay(min(B * N * 16, 4_000_000), 10, 2, device=dev)
        # default: the step kernel appends the transitions itself (uavca_step_multi_replay: 2 launches per acting step with
        # the fused policy); "fused_separate_append" keeps round 2's three launches (policy, step, append) beside it
        ro = G.BatchedRollout(env, policy, replay, action_mode="polar", precision=precision,
                              fused_append=row != "fused_separate_append")
        ro.reset()
        head_err = policy_head_error(G, torch, policy, ro, env) if row in ("tf32", "fused") else None
        with torch.cuda.stream(stream):
            for _ in range(3):
                ro.step()
        torch.cuda.synchronize(dev)
        n_graph = min(K, 50)
        q, rem = divmod(K, n_graph)

        def capture(n):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=stream):
                for _ in range(n):
                    ro.step()
            g.replay()
            return g

        g, g_rem = capture(n_graph), capture(rem) if rem else None
        torch.cuda.synchronize(dev)

        def rep(g=g, q=q, g_rem=g_rem):
            for _ in range(q):
                g.replay()
            if g_rem is not None:
                g_rem.replay()

        ts = timed_reps(torch, stream, rep, (0.07 if precision == "fused" else 1.0) * K, dev, barrier)
        ts = [sharding.max_over_ranks(t, device=dev) for t in ts] if dist is not None else ts
        if row == keep_row:
            kept = output_sample(dict(obs=env.obs, reward=env.reward, done=env.done, action=ro.action))
        med = statistics.median(ts)
        us = med * 1e3 / K
        rows[row] = {"us_per_acting_step": us, "value": world * B * N / us * 1e6, "best_us": min(ts) * 1e3 / K,
                     "repetitions": len(ts), "steps_per_repetition": K, "replay_size": len(replay),
                     "launches_per_acting_step": (2 if ro.fused_append else 3) if precision == "fused" else None}
        if head_err is not None:
            rows[row]["head_max_abs_err_vs_fp64"] = head_err
        total_launches += env.launch_count
        del g, g_rem, ro, replay, env
    torch.backends.cuda.matmul.allow_tf32 = tf32_before
    return rows, total_launches, kept


def policy_head_error(G, torch, policy, ro, env):
    """max |(mean, log_std) - float64 policy| over this env's reset observations: the acting precision of a row.  TF32 and
    fp16 operands both carry 10 explicit mantissa bits into an fp32 accumulator; this shows the two side by side."""
    x = env.obs.view(-1, env.obs_dim)[:65536].contiguous()
    p64 = copy.deepcopy(policy).double()
    with torch.no_grad():
        m64, s64 = p64(x.double())
        if ro.precision == "fused":
            head = torch.empty((x.shape[0], 4), dtype=torch.float32, device=x.device)
            ro.fused.act(x, noise=torch.zeros((x.shape[0], 2), dtype=torch.float32, device=x.device), head=head)
            m, sd = head[:, 0:2], head[:, 2:4]
        else:
            prev = torch.backends.cuda.matmul.allow_tf32
            torch.backends.cuda.matmul.allow_tf32 = ro.precision == "tf32"
            try:
                m, sd = policy(x)
            finally:
                torch.backends.cuda.matmul.allow_tf32 = prev
        return float(torch.maximum((m.double() - m64).abs().max(), (sd.double() - s64).abs().max()))


def run_acting(args, wl, G, torch, dev, rank, world, dist, barrier):
    """`--workload c5r`: the acting step as the headline; value = the fp32 row unless --acting-precision says otherwise."""
    B, N, K = wl["B"], wl["N"], args.steps
    head = args.acting_precision
    rows, total_launches, last = measure_acting(args, G, torch, dev, rank, world, dist, barrier, B, N, K,
                                                keep_row=head if args.dump_outputs and rank == 0 else None)
    if last is not None:
        write_outputs(args.dump_outputs, last)
    if rank == 0:
        us = rows[head]["us_per_acting_step"]
        emit({"metric": "UAV env-steps/sec", "value": rows[head]["value"], "unit": "UAV env-steps/s", "n_gpus": world, "steps": K,
              "warmup": max(args.warmup, 3), "ms_per_step": us / 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
              "dtype": f"env: f64 velocity / f32; policy: {head}", "data": "synthetic (random-init policy: the reference ships no weights)",
              "config": dict(workload_config(args, wl, world, B), actions="policy samples mapped by the fused polar action map",
                             headline_precision=head, rows=rows,
                             timing="CUDA events around repetitions of CUDA-graph replays of the whole acting step (policy + step + replay append)"),
              "e2e": None, "gpu_launches": int(total_launches), "roofline": None, "cpu_baseline": None})
    if dist is not None:
        dist.destroy_process_group()


_REAL_STDOUT = None


def protect_stdout():
    """The driver reads ONE JSON line from stdout.  Libraries print there too (NCCL announces its version on stdout at
    init): point fd 1 at stderr for the whole run and keep the real stdout for the result line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def output_sample(arrays: dict, seed: int = 0) -> dict:
    """Host copies of the outputs a caller of the timed path received in its last step (`arrays`: name -> tensor or array
    whose axis 0 is the env axis), as float32 (float64 and int64 as float64).  Where all of them together exceed
    DUMP_BYTES, the same envs of every array are kept: a sorted sample drawn with `seed`, so that runs with the same
    arguments keep the same envs.  `env_index` lists the envs kept (indices into the batch)."""
    import numpy as np
    import torch

    ts = {k: torch.as_tensor(v) for k, v in arrays.items()}
    wide = (torch.float64, torch.int64)
    n = next(iter(ts.values())).shape[0]
    per_env = 8 + sum(t[:1].numel() * (8 if t.dtype in wide else 4) for t in ts.values())
    keep = min(n, DUMP_BYTES // per_env)
    idx = np.arange(n) if keep == n else np.sort(np.random.default_rng(seed).choice(n, keep, replace=False))
    out = {}
    for k, t in ts.items():
        sel = t[torch.as_tensor(idx, device=t.device)] if keep < n else t
        out[k] = sel.to(torch.float64 if t.dtype in wide else torch.float32).cpu().numpy()
    out["env_index"] = idx.astype(np.float64)
    return out


def write_outputs(path: str, sample: dict):
    """--dump-outputs: one DIR/<name>.npy per array of `output_sample`."""
    import numpy as np

    os.makedirs(path, exist_ok=True)
    for k, a in sample.items():
        np.save(os.path.join(path, k + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS),
                    help="default: c3 (BASELINE configs[2]) on one GPU, c4s (configs[3]: N=32, 1,048,576 envs sharded) with --gpus > 1")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-rollout", action="store_true")
    ap.add_argument("--no-acting", action="store_true", help="skip the configs[4] acting-step rows of the default line")
    ap.add_argument("--no-numa-bind", action="store_true")
    ap.add_argument("--rollout-k", type=int, default=32, help="steps per launch of the rollout measurement")
    ap.add_argument("--headline", default="rollout", choices=["rollout", "per_step"],
                    help="which product path `value` / `roofline` describe: K steps per launch from an action block (default: the "
                         "bench's actions are open-loop random) or one launch per step; the other one is reported beside it")
    ap.add_argument("--acting-precision", default="fp32", choices=["fp32", "tf32", "fused"])
    ap.add_argument("--streams", type=int, default=None,
                    help="streams the independent batches of the ring are pipelined over (default: 2; 4 for the small c2/c5 batches)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the headline path returned in its last step as DIR/<name>.npy "
                         "(float32 / float64, at most 64 MB: a fixed sample of envs where the batch is larger; rank 0's "
                         "shard); inputs are seeded, so runs with the same arguments can be compared file by file")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the outputs of --impl ours")
    protect_stdout()
    if args.workload is None:
        args.workload = "c3" if args.gpus <= 1 else "c4s"
    wl = WORKLOADS[args.workload]
    if args.workload == "c5r" and args.steps is not None and args.steps % 2:
        ap.error("--workload c5r times an even number of steps (the acting step alternates two observation buffers)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.steps is None:
        args.steps = wl["steps"] if args.impl == "ours" else 100
    if args.streams is None:
        args.streams = wl.get("streams", 2)
    if args.impl == "reference":
        run_reference(args, wl, rank, world)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under torch.distributed.run
        import subprocess

        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29513", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd, stdout=_REAL_STDOUT))  # the ranks inherit the REAL stdout
    run_ours(args, wl, rank, world, local_rank)


if __name__ == "__main__":
    main()
