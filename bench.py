#!/usr/bin/env python
"""bench.py — headline benchmark of the b2048 hot path (see BASELINE.json / DESIGN.md).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

Workload at every N (weak scaling): BASELINE.json configs[1] per GPU — random-action batched env
stepping on 1,048,576 packed boards (uniform over the legal moves from the Philox action word,
reset-on-done).  One "step" = one fused `b2048_step_many` launch over all boards of the rank.

  value      env-steps/s, whole job, boards resident in HBM: ONE CUDA-event pair around K back-to-back launches that
             rotate over 12 resident 1 M-board batches (276 MB of state > the 126 MB L2, so no launch finds its inputs
             in L2 and no flush kernel sits between the launches); max over ranks.  Consecutive step launches overlap
             through programmatic dependent launch.  `env_flushed` repeats the round-1 protocol (one batch, a 256 MiB
             memset and an event pair around every launch) for continuity.
  e2e        the same metric through the host-facing API with HOST (pinned) buffers: per step the actions
             are copied host->device and board/reward/flags device->host inside the timed region
  roofline   HBM: 22 algorithmic bytes per env-step (SURVEY.md section 8d) over the measured kernel time
  cpu_baseline  the reference's algorithm on this box's host cores (Python port, all cores), rank 0, N=1 only
  env_multi_step  secondary: env-steps/s with 64 steps per launch (state kept in registers across the steps)
  env_trained_boards  secondary: the same env-step measurement on boards harvested from a trained policy (north_star)
  rollout    secondary: policy-rollout steps/s (MLP 16-256-256-4 forward + masked sampling + env step), 65,536 boards
  rollout_onehot  secondary: the same for the reference's documented one-hot 272-256-128-64-4 policy (shape-generic tcgen05
             policy kernel + step kernel), 262,144 boards
  train_iter / train_iter_actor_critic   secondary: BASELINE.json configs[2] / configs[3] (rollout to termination +
             one update; 65,536 / 262,144 boards per GPU)
  train_iter_actor_critic_shared   secondary: configs[3] as BASELINE.json words it (shared MLP trunk + value head, advantage
             scan with lambda = 0.95) on the same kernels (b2048/shared_trunk.py)
  train_iter_actor_critic_onehot   secondary: the reference's documented configuration (one-hot observations, hidden
             [256, 128, 64], Adam; SURVEY.md section 8d config 4) at configs[3]'s 262,144 boards per GPU, on the shape-generic
             tcgen05 kernels (csrc/b2048_mlp_gen.cu)
  sharded_sweep  secondary, N >= 2 only: BASELINE.json configs[4] — 64 M boards in total, 16-step episodes, one update
  summary    the key numbers of every leg once more, LAST in the line (a truncated tail still shows them)

`--impl reference` times the CPU side alone (the reference is pure Python and cannot travel to the GPU
box; oracle/pyport.py restates it at the same per-environment granularity).

`--dump-outputs DIR` writes the outputs of the last timed env step as .npy files (see dump_outputs).  The boards, seeds
and step counters depend on the arguments alone, so two builds run with the same arguments can be compared output for
output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "2048 env-steps/sec (random-legal batched env stepping, 1M packed boards per GPU)"
UNIT = "env-steps/s"
BOARDS_PER_GPU = 1 << 20
ALGO_BYTES_PER_STEP = 22  # board r 8 + board w 8 + action/mask r 1 + reward w 4 + flags w 1
RUNNER_ENV = dict(obs_mode="log2", obs_log2_scale=0.0625, reward_mode="log2", base_reward_scale=0.5,
                  bonus_mode="off", max_steps=1024)


def measured_tensor_peaks():
    """(burst, sustained) dense bf16 TFLOP/s from MEASURED_PEAKS.json, else the profiling guide's fallback."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["bf16_tflops"]), float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 1590.0, 1400.0, "fallback (B200_PROFILING.md)"


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


_UNIT = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}


def profile_traffic(candidates, launch_filter=None):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from a committed ncu summary (profiles/*.csv written by
    profiles/summarize_ncu.py): the first candidate file that exists; the mean over its launch columns whose header
    contains `launch_filter`.  Returns (bytes or None, file name or None)."""
    import csv
    for name in candidates:
        path = os.path.join(ROOT, "profiles", name)
        if not os.path.exists(path):
            continue
        try:
            with open(path) as f:
                rows = list(csv.reader(f))
            hdr = rows[0]
            cols = [i for i in range(2, len(hdr)) if launch_filter is None or launch_filter in hdr[i]]
            tot = None
            for r in rows[1:]:
                if r and r[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum") and cols:
                    v = sum(float(r[i]) for i in cols) / len(cols) * _UNIT.get(r[1], 1.0)
                    tot = v if tot is None else tot + v
            if tot is not None:
                return tot, "profiles/" + name
        except Exception:
            continue
    return None, None


class ClockSampler:
    """Samples SM clocks / throttle reasons WHILE the timed region runs (NVML every ~2 ms; nvidia-smi fallback)."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.sm, self.reasons, self.max_mhz, self.source = [], set(), None, "nvml"
        self._stop = threading.Event()
        self._th = threading.Thread(target=self._run, daemon=True)
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nvml = None
            self.source = "nvidia-smi"

    def _sample_nvml(self):
        n = self._nvml
        self.sm.append(int(n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM)))
        r = int(n.nvmlDeviceGetCurrentClocksEventReasons(self._h)) if hasattr(n, "nvmlDeviceGetCurrentClocksEventReasons") \
            else int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self._h))
        for name, bit in (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20),
                          ("hw_thermal_slowdown", 0x40)):
            if r & bit:
                self.reasons.add(name)

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                              str(self.index)], capture_output=True, text=True, timeout=5).stdout
        parts = [x.strip() for x in out.strip().split(",")]
        if len(parts) >= 6 and parts[0].isdigit():
            self.sm.append(int(parts[0]))
            self.max_mhz = int(parts[1]) if parts[1].isdigit() else self.max_mhz
            for i, nm in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
                if parts[2 + i].lower().startswith("active"):
                    self.reasons.add(nm)

    def _run(self):
        while not self._stop.is_set():
            try:
                if self._nvml is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            self._stop.wait(0.002 if self._nvml is not None else 0.05)

    def __enter__(self):
        self._th.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._th.join(timeout=6)

    def summary(self):
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(sm), "source": self.source}


def cpu_baseline(seconds: float = 10.0):
    """The reference's algorithm on the host cores: per-env Python/NumPy port, one process per core."""
    from oracle import pyport
    cores = len(os.sched_getaffinity(0))
    rate, nsteps = pyport.time_multiprocess(seconds, cores)
    return {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{nsteps} random-legal env steps (runner-default env, reset-on-done) in ~{seconds:.0f} s, "
                      f"{cores} processes of oracle/pyport.py (per-env Python+NumPy restatement of the reference)"}


def cpu_rollout_baseline(seconds: float = 5.0):
    """north_star: "the reference's CPU env + rollout timed on the box's own host cores" — the rollout half: the
    reference's run_episode loop (NumPy MLP forward + sampling + env step) per environment, one process per core."""
    from oracle import pyport
    cores = len(os.sched_getaffinity(0))
    rate, nsteps = pyport.time_rollout_multiprocess(seconds, cores)
    return {"value": rate, "unit": "rollout-steps/s", "cores": cores, "kind": "port",
            "sample": f"{nsteps} policy-rollout steps (16-256-256-4 NumPy MLP + masked sampling + env step, runner-default env) in "
                      f"~{seconds:.0f} s, {cores} processes of oracle/pyport.py"}


def cpu_native_baseline(n=1 << 18, steps=20):
    """Extra context: the C oracle (same rules, compiled, multi-threaded) — a much stronger CPU baseline."""
    import oracle
    cores = len(os.sched_getaffinity(0))
    cfg = oracle.make_cfg(action_mode="random_legal", auto_reset=True, **RUNNER_ENV)
    secs = oracle.bench_steps(n, steps, cores, cfg)
    return {"value": n * steps / secs, "unit": UNIT, "cores": cores, "kind": "port-native-C",
            "sample": f"{n} boards x {steps} steps, oracle/b2048_oracle.c on {cores} threads"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warm = max(1, args.steps), args.warmup
    from oracle import pyport
    cores = len(os.sched_getaffinity(0))
    # each "step" is a bounded sample of all-core stepping on one persistent worker pool; the whole run is capped
    # at about a minute and a half of CPU work whatever K is
    per = min(1.0, 90.0 / (steps + warm))
    t0 = time.perf_counter()
    samples = pyport.time_multiprocess_series(per, cores, steps + warm)[warm:]
    wall = (time.perf_counter() - t0) * steps / (steps + warm)
    total = sum(n for _, n in samples)
    rate_acc = sum(r for r, _ in samples)
    value = rate_acc / steps
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warm, "ms_per_step": 1e3 * wall / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": {"workload": "random-legal env stepping, runner-default Game2048Env, reset-on-done; "
                                   "bounded sample per step on all host cores"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{total} env steps in {steps} samples of {per:.2f} s x {cores} processes"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def run_b200(args):
    import torch
    import torch.distributed as dist
    import b2048

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # before any pinned allocation: staging buffers of the host-buffer (e2e) leg on the GPU's own NUMA node
    numa = {"bound": False, "why": "--no-numa-bind"} if args.no_numa_bind else b2048.dist.bind_to_gpu_numa_node(local_rank)
    info = b2048.dist.init_distributed("nccl")
    if world > 1:                       # every rank's node / outcome, for the line rank 0 prints
        nn = torch.full((world, 2), 0, dtype=torch.int32, device=dev)
        nn[rank, 0] = -1 if numa.get("numa_node") is None else int(numa["numa_node"])
        nn[rank, 1] = int(bool(numa.get("bound")))
        dist.all_reduce(nn)
        numa["all_ranks_node"], numa["all_ranks_bound"] = nn[:, 0].tolist(), nn[:, 1].tolist()
    n = args.boards
    K, W = args.steps, max(3, args.warmup)

    R = args.batches                    # resident batches the launches rotate over: R x 23 MB of state > the 126 MB L2
    envs = [b2048.Batched2048Env(n, b2048.Game2048EnvConfig(**RUNNER_ENV), device=dev, seed=0xB200 + r, gid0=rank * n,
                                 track_state=not args.lean) for r in range(R)]
    for e in envs:
        e.reset_many()
        # spread the boards over the episode distribution before timing (64 untimed steps, SURVEY 8d)
        e.step_many_n(64, action_mode="random_legal", auto_reset=True)
    env = envs[0]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for k in range(max(W, R)):
        envs[k % R].step_many(action_mode="random_legal", auto_reset=True)
    t0e, t1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    with ClockSampler(local_rank) as clk:
        # a short spin kernel in front lets the host enqueue ahead of the device, so the K launches run back to back
        torch.cuda._sleep(2_000_000)
        t0e.record()
        for k in range(K):
            envs[k % R].step_many(action_mode="random_legal", auto_reset=True)
        t1e.record()
        barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(envs[(K - 1) % R], args.dump_outputs)
    kernel_ms = t0e.elapsed_time(t1e)
    t = torch.tensor([kernel_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    kernel_ms = float(t.item())
    value = world * n * K / (kernel_ms * 1e-3)
    clocks = clk.summary()

    # ---- the round-1 protocol for continuity: one batch, L2 flushed by a 256 MiB memset and an event pair around every launch
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
    Kf = min(K, 50)
    for _ in range(3):
        flush.zero_()
        env.step_many(action_mode="random_legal", auto_reset=True)
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(Kf)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(Kf)]
    barrier()
    for k in range(Kf):
        flush.zero_()                      # evict boards from L2 between timed launches
        starts[k].record()
        env.step_many(action_mode="random_legal", auto_reset=True)
        ends[k].record()
    barrier()
    tf = torch.tensor([sum(a.elapsed_time(b) for a, b in zip(starts, ends))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tf, op=dist.ReduceOp.MAX)
    flushed_ms = float(tf.item()) / Kf

    # ---- e2e: host (pinned) buffers through the public API, copies inside the timed region.  Per step the actions go
    #      host -> device and board / reward / flags come back device -> host (13 B per board: PCIe-bound).  The step
    #      writes into one of two output slots (step_many's board_out / reward_out / flags_out), so the copy-back of
    #      step k runs on a second stream under the H2D + kernel of step k + 1.
    Ke = min(K, 100)
    h_act = torch.randint(0, 4, (n,), dtype=torch.uint8).pin_memory()
    d_act = torch.empty(n, dtype=torch.uint8, device=dev)
    h_board = [torch.empty(n, dtype=torch.int64).pin_memory() for _ in range(2)]
    h_rew = [torch.empty(n, dtype=torch.float32).pin_memory() for _ in range(2)]
    h_flags = [torch.empty(n, dtype=torch.uint8).pin_memory() for _ in range(2)]
    d_board = [torch.empty(n, dtype=torch.int64, device=dev) for _ in range(2)]
    d_rew = [torch.empty(n, dtype=torch.float32, device=dev) for _ in range(2)]
    d_flags = [torch.empty(n, dtype=torch.uint8, device=dev) for _ in range(2)]
    copy_stream = torch.cuda.Stream(device=dev)
    step_done = [torch.cuda.Event() for _ in range(2)]
    d2h_done = [torch.cuda.Event() for _ in range(2)]
    main = torch.cuda.current_stream(dev)
    for ev in d2h_done:
        ev.record(main)
    e2e_k = [0]

    def e2e_step():
        slot = e2e_k[0] & 1
        e2e_k[0] += 1
        d_act.copy_(h_act, non_blocking=True)
        main.wait_event(d2h_done[slot])              # the slot's previous copy-back has read its device buffers
        env.step_many(d_act, auto_reset=True, board_out=d_board[slot], reward_out=d_rew[slot], flags_out=d_flags[slot])
        step_done[slot].record(main)
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(step_done[slot])
            h_board[slot].copy_(d_board[slot], non_blocking=True)
            h_rew[slot].copy_(d_rew[slot], non_blocking=True)
            h_flags[slot].copy_(d_flags[slot], non_blocking=True)
            d2h_done[slot].record(copy_stream)

    def e2e_drain():
        main.wait_event(d2h_done[0])
        main.wait_event(d2h_done[1])

    for _ in range(3):
        e2e_step()
    e2e_drain()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(Ke):
        e2e_step()
    e2e_drain()                                      # the last results are on the host before the clock stops
    e1.record()
    barrier()
    te = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * n * Ke / (float(te.item()) * 1e-3)
    last = (e2e_k[0] - 1) & 1
    checksum = int(h_board[last].sum().item()) ^ int(h_flags[last].sum().item())

    e2e_ms = float(te.item()) / Ke
    if rank == 0:
        peak, peak_src = measured_peaks()
        per_launch_s = kernel_ms * 1e-3 / K
        achieved = n * ALGO_BYTES_PER_STEP / per_launch_s / 1e9
        kname = "b2::step_fast_kernel<RANDOM_LEGAL, %s, plain>" % ("false" if args.lean else "true")
        traffic, traffic_src = (None, None)
        if n == BOARDS_PER_GPU and not args.lean:
            traffic, traffic_src = profile_traffic(["r02_ncu_step_fast_kernel.csv", "r01_ncu_step_fast_kernel.csv"], "step_fast")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": max(W, R),
            "ms_per_step": kernel_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64", "data": "synthetic",
            "config": {"workload": f"random-legal batched env stepping, {n} packed boards per GPU "
                                   f"(BASELINE.json configs[1]), runner-default env, reset-on-done",
                       "boards_per_gpu": n, "numa": numa,
                       "l2": f"inputs larger than L2: the launches rotate over {R} resident {n}-board batches "
                             f"({R * n * (22 if args.lean else 23) / 1e6:.0f} MB of state vs 126 MB L2), no flush kernel between them; "
                             "one CUDA-event pair around the K back-to-back launches",
                       "state": "board only (22 B/step variant)" if args.lean else
                                "board + score/step/max_tile counters kept per step (+18 B/step, not counted)"},
            "clocks": clocks,
            # pcie_gbs: bytes that cross PCIe per GPU per step (both directions) over the e2e step time — the e2e figure
            # is bound by the host link / host memory system, not by the kernel (14 B per board per step)
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": n * 1, "d2h_bytes_per_step": n * 13,
                    "steps": Ke, "checksum": checksum, "ms_per_step": e2e_ms,
                    "pcie_gbs_per_gpu": n * 14 / (e2e_ms * 1e-3) / 1e9, "pcie_gbs_all_gpus": world * n * 14 / (e2e_ms * 1e-3) / 1e9,
                    "bound": "host link (PCIe) per GPU; the host memory system when several GPUs copy at once"},
            "gpu_launches": K,
            # traffic: dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of this kernel on 1,048,576 boards, read
            # from the committed `ncu --set full` summary named in traffic_source (the outputs of a profiled single launch
            # are still dirty in the 126 MB L2 when it ends, so they do not all show up as DRAM writes)
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "algorithmic_bytes_per_env_step": ALGO_BYTES_PER_STEP, "kernel": kname,
                         "avg_launch_us": per_launch_s * 1e6,
                         "limiter": "integer (ALU) issue, not HBM: see profiles/ and DESIGN.md section 3"},
            "env_flushed": {"value": world * n / (flushed_ms * 1e-3), "unit": UNIT, "ms_per_step": flushed_ms, "steps": Kf,
                            "frac": n * ALGO_BYTES_PER_STEP / (flushed_ms * 1e-3) / 1e9 / peak,
                            "protocol": "round-1 protocol: one batch, 256 MiB memset + an event pair around every launch"},
        }
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_baseline(args.cpu_seconds)
            line["cpu_baseline_rollout"] = cpu_rollout_baseline(min(5.0, args.cpu_seconds))
            try:
                line["cpu_baseline_native"] = cpu_native_baseline()
            except Exception as e:  # the native leg is context only
                line["cpu_baseline_native"] = {"error": str(e)}
    del envs[1:]
    # ---- secondary: the same stepping with 64 steps per launch (b2048_step_many_n: state in registers across steps)
    multi = None
    if not args.lean:
        Kn, Tn = 20, 64
        for _ in range(3):
            env.step_many_n(Tn, action_mode="random_legal", auto_reset=True)
        s2 = [torch.cuda.Event(enable_timing=True) for _ in range(Kn)]
        e2 = [torch.cuda.Event(enable_timing=True) for _ in range(Kn)]
        barrier()
        for k in range(Kn):
            flush.zero_()
            s2[k].record()
            env.step_many_n(Tn, action_mode="random_legal", auto_reset=True)
            e2[k].record()
        barrier()
        tn = torch.tensor([sum(a.elapsed_time(b) for a, b in zip(s2, e2))], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tn, op=dist.ReduceOp.MAX)
        multi = {"metric": "env-steps/s, 64 steps per launch (b2048_step_many_n)", "value": world * n * Kn * Tn / (float(tn.item()) * 1e-3),
                 "unit": UNIT, "steps_per_launch": Tn, "launches": Kn, "ms_per_launch": float(tn.item()) / Kn,
                 "note": "boards, counters and legal masks stay in registers across the 64 steps; only the final state is written"}
    # secondary legs (every rank takes part: the update all-reduces gradients over NCCL)
    extra = {}
    if multi is not None:
        extra["env_multi_step"] = multi
    if not args.no_rollout:
        try:
            for key, prec in (("rollout", 1), ("rollout_fp32", 0)):
                # tensor-core leg: 256 steps = one persistent launch; fp32 leg: 64 steps (two launches per step)
                r = b2048.bench_rollout(dev, gid0=rank * 65536, precision=prec, steps=256 if prec == 1 else 64)
                v = torch.tensor([r["value"]], dtype=torch.float64, device=dev)
                if world > 1:
                    dist.all_reduce(v, op=dist.ReduceOp.SUM)
                r["value_all_gpus"] = float(v.item())
                if prec == 1:   # tensor-core roofline of the fused policy + env kernel (a multi-millisecond launch: sustained peak)
                    burst, sustained, src = measured_tensor_peaks()
                    tr, tr_src = profile_traffic(["r02_ncu_rollout_tc_kernel_65k.csv", "r01_ncu_rollout_tc_kernel_65k.csv"], "policy_tc")
                    r["roofline"] = {"bound": "tensor", "achieved": r["achieved_tflops"], "peak": sustained, "unit": "TFLOP/s",
                                     "frac": r["achieved_tflops"] / sustained, "peak_burst": burst, "peak_source": src,
                                     "algorithmic_flops_per_rollout_step": r["flops_per_step"],
                                     "kernel": "b2::policy_tc_kernel<rollout>", "traffic": tr,
                                     "traffic_source": (tr_src + " (DRAM bytes of the profiled 16-step launch on 65,536 boards)") if tr_src else None}
                extra[key] = r
            # the reference's documented one-hot 272-256-128-64-4 policy on the shape-generic tcgen05 policy kernel (262,144 boards)
            r = b2048.bench_rollout(dev, boards=262144, gid0=rank * 262144, precision=1, steps=32, network="onehot")
            v = torch.tensor([r["value"]], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(v, op=dist.ReduceOp.SUM)
            r["value_all_gpus"] = float(v.item())
            burst, sustained, src = measured_tensor_peaks()
            r["roofline"] = {"bound": "tensor", "achieved": r["achieved_tflops"], "peak": sustained, "unit": "TFLOP/s",
                             "frac": r["achieved_tflops"] / sustained, "peak_burst": burst, "peak_source": src,
                             "algorithmic_flops_per_rollout_step": r["flops_per_step"], "kernel": "b2::gen_mlp_kernel<ReLU> (+ step_kernel)",
                             "traffic": None,
                             "note": "MMA phases are shared-memory bound: the weights stream through a 3-slot ring (DESIGN.md section 3)"}
            extra["rollout_onehot"] = r
            r = b2048.bench_env_trained_boards(dev, boards=n, gid0=rank * n)
            v = torch.tensor([r["value"]], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(v, op=dist.ReduceOp.SUM)
            r["value_all_gpus"] = float(v.item())
            extra["env_trained_boards"] = r
            extra["train_iter"] = b2048.bench_train_iter(dev, boards=args.train_boards, info=info, precision="auto")
            extra["train_iter_actor_critic"] = b2048.bench_train_iter(dev, boards=args.ac_boards, info=info, precision="auto",
                                                                      use_critic=True, iters=3)
            # configs[3]'s literal wording: one shared trunk with a policy head and a value head, lambda advantage scan
            extra["train_iter_actor_critic_shared"] = b2048.bench_train_iter(dev, boards=args.ac_boards, info=info, precision="auto",
                                                                             use_critic=True, iters=2, shared_trunk=True)
            # SURVEY.md section 8d config 4 as the reference documents it (one-hot 272-256-128-64 networks): the shape-generic
            # tensor-core kernels (gen_mlp_kernel / gen_dw_kernel)
            extra["train_iter_actor_critic_onehot"] = b2048.bench_train_iter(dev, boards=args.onehot_boards, info=info, precision="auto",
                                                                             use_critic=True, iters=2, network="onehot")
            if world > 1 and not args.no_sweep:
                extra["sharded_sweep"] = b2048.bench_sharded_sweep(dev, total_boards=args.sweep_boards, info=info)
        except Exception as e:
            extra["rollout_error"] = repr(e)
    if rank == 0:
        line.update(extra)
        # the key numbers once more, LAST in the line
        g = lambda d, *ks: (g(d.get(ks[0], {}), *ks[1:]) if len(ks) > 1 else d.get(ks[0])) if isinstance(d, dict) else None
        line["summary"] = {
            "env_steps_per_s": value, "env_ms_per_step": kernel_ms / K, "env_hbm_frac": line["roofline"]["frac"],
            "env_flushed_ms_per_step": flushed_ms, "e2e_env_steps_per_s": e2e_value,
            "e2e_pcie_gbs_per_gpu": line["e2e"]["pcie_gbs_per_gpu"],
            "env_multi_step_per_s": g(extra, "env_multi_step", "value"),
            "rollout_steps_per_s": g(extra, "rollout", "value_all_gpus"), "rollout_tensor_frac": g(extra, "rollout", "roofline", "frac"),
            "rollout_onehot_steps_per_s": g(extra, "rollout_onehot", "value_all_gpus"),
            "rollout_onehot_tensor_frac": g(extra, "rollout_onehot", "roofline", "frac"),
            "train_iter_rollout_ms": g(extra, "train_iter", "rollout_ms"), "train_iter_update_ms": g(extra, "train_iter", "update_ms"),
            "train_iter_update_mode": g(extra, "train_iter", "update_precision"),
            "train_iter_update_ms_bf16": g(extra, "train_iter", "update_ms_bf16"),
            "ac_rollout_ms": g(extra, "train_iter_actor_critic", "rollout_ms"), "ac_update_ms": g(extra, "train_iter_actor_critic", "update_ms"),
            "ac_shared_rollout_ms": g(extra, "train_iter_actor_critic_shared", "rollout_ms"),
            "ac_shared_update_ms": g(extra, "train_iter_actor_critic_shared", "update_ms"),
            "ac_onehot_rollout_ms": g(extra, "train_iter_actor_critic_onehot", "rollout_ms"),
            "ac_onehot_update_ms": g(extra, "train_iter_actor_critic_onehot", "update_ms"),
            "ac_onehot_mode": g(extra, "train_iter_actor_critic_onehot", "update_precision"),
            "sweep_rollout_steps_per_s": g(extra, "sharded_sweep", "rollout_steps_per_s"),
            "sweep_update_samples_per_s": g(extra, "sharded_sweep", "update_samples_per_s"),
            "error": extra.get("rollout_error")}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(env, out_dir: str) -> None:
    """Writes what the last timed step_many returned to its caller, as out_dir/<name>.npy: reward and flags, and the
    state it updated in place (packed board as [low, high] 32-bit words, score, step, max tile exponent).  Integers are
    stored exactly as float32 (8-bit) or float64 (32-bit and wider).  Above 64 MB in all, a fixed seeded sample of the
    boards is written instead, with its board indices in index.npy."""
    import numpy as np
    board = env.board.cpu().numpy().view(np.uint64)
    out = {"board": np.stack([board & np.uint64(0xFFFFFFFF), board >> np.uint64(32)], axis=1).astype(np.float64),
           "reward": env.reward.cpu().numpy().astype(np.float32),
           "flags": env.flags.cpu().numpy().astype(np.float32)}
    if env.track_state:
        out["score"] = env.score.cpu().numpy().astype(np.float64)
        out["step"] = env.step_count.cpu().numpy().astype(np.float64)
        out["max_exp"] = env.max_exp.cpu().numpy().astype(np.float32)
    n = len(board)
    per_board = sum(a.nbytes for a in out.values()) // n
    if per_board * n > DUMP_LIMIT_BYTES:
        m = DUMP_LIMIT_BYTES // (per_board + 8)
        idx = np.sort(np.random.default_rng(0).choice(n, m, replace=False))
        out = {k: a[idx] for k, a in out.items()}
        out["index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The ONE JSON line of the contract, written to the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


def main():
    # Libraries (NCCL prints its version banner) must not pollute stdout: keep the real stdout for the JSON
    # line only and send everything else to stderr.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--boards", type=int, default=BOARDS_PER_GPU)
    ap.add_argument("--lean", action="store_true", help="board-only state (no score/step/max_tile arrays)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true", help="leave the process on whatever CPUs the launcher gave it")
    ap.add_argument("--no-rollout", action="store_true")
    ap.add_argument("--onehot-boards", type=int, default=262144, help="actor-critic leg on the reference's documented one-hot network")
    ap.add_argument("--no-sweep", action="store_true", help="skip the BASELINE.json configs[4] leg (runs at N >= 2)")
    ap.add_argument("--sweep-boards", type=int, default=64 << 20, help="total boards of the configs[4] leg")
    ap.add_argument("--batches", type=int, default=12, help="resident 1 M-board batches the timed launches rotate over")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--train-boards", type=int, default=65536)
    ap.add_argument("--ac-boards", type=int, default=262144, help="actor-critic leg (BASELINE.json configs[3])")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write rank 0's outputs of the last timed env step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl b200: the reference arm only times the CPU")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
