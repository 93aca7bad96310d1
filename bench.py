#!/usr/bin/env python
"""Headline benchmark: agent-steps/sec of the fused navigation_graph step (+obs +reward +auto-reset
with lexifair assignment), BASELINE.json config 2: 3 agents / 3 goals / 3 obstacles, FA+FR reward,
goal_rew = collision_rew = 30, episode_length 25, 65 536 envs per B200, random actions.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One process per GPU (torchrun for N > 1; envs sharded by global env index, weak scaling: 65 536
envs per GPU).  Prints ONE JSON line on rank 0.  A "step" is one env step of the whole batch.

* ``value``  device-resident throughput: actions and outputs stay in HBM, K steps launched through
  ``fm_step_many``; outputs cycle through a 25-slot slab ring (3.1 GB > L2) so stores go to HBM.
* ``e2e``    the same metric through the reference-facing API ``B200GraphVecEnv.step(actions_env)``
  (numpy one-hot in, numpy out): one ``fm_step_host`` C-ABI call per step that copies the actions
  H2D and obs / node_obs / adj / reward / done D2H inside the timed region.
* ``roofline``  algorithmic HBM bytes per launch (SURVEY.md section 8d: W = 30N + 2O + 5 + 11NE + E^2 words per
  env-step) / average step-kernel duration from CUDA events, against MEASURED_PEAKS.json hbm_gbs.
* ``cpu_baseline``  the numpy oracle port (oracle/navgraph.py) on all host cores, bounded sample.
* ``--impl reference``  times that CPU port as the reference arm (the reference itself is pure Python that
  needs a checkout of the original project, which this repository does not contain; the port is pinned to it by tests/golden).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_AGENTS, N_OBST, EPISODE = 3, 3, 25
N_WALLS = 0            # --walls W: diagnostic run of the wall instantiations (SURVEY N4); 0 in every BASELINE config
ENVS_PER_GPU = 65536
METRIC = "agent-steps/sec, navigation_graph step+obs+reward"
WORKLOAD = ("navigation_graph 3 agents / 3 goals / 3 obstacles, FA+FR reward, goal_rew=collision_rew=30, "
            "episode_length 25 with auto-reset + lexifair assignment, random actions")
GOAL_REW = COLL_REW = 30.0
FAIRNESS = True

# BASELINE.json configs (the headline line is c2; the others are diagnostic runs: --config c1|c3|c4)
CONFIGS = {
    "c1": dict(agents=3, obstacles=3, envs=128, rew=5.0, fairness=False,
               workload="navigation_graph 3 agents / 3 goals / 3 obstacles, FA (no fairness reward), 128 envs, random actions"),
    "c2": dict(agents=3, obstacles=3, envs=65536, rew=30.0, fairness=True, workload=WORKLOAD),
    "c3": dict(agents=7, obstacles=3, envs=262144, rew=5.0, fairness=True,
               workload="navigation_graph 7 agents / 7 goals / 3 obstacles, FA+FR, 262144 envs, random actions"),
    "c4": dict(agents=16, obstacles=3, envs=131072, rew=5.0, fairness=True,
               workload="navigation_graph 16 agents / 16 goals / 3 obstacles, FA+FR, 131072 envs per GPU (1M over 8), random actions"),
    # config 5: the rollout loop (policy forward in torch + simulator step + buffer insert), all on the device
    # widened row N3 (diagnostic): the formation-family scenario of BASELINE config 2's wording, on its own kernels
    "form": dict(agents=3, obstacles=3, envs=65536, rew=30.0, fairness=True,
                 workload="nav_fairassign_fairrew_formation_graph 3 agents / 3 goals / 3 obstacles, FA+FR, 65536 envs, random actions"),
    "c5": dict(agents=3, obstacles=3, envs=65536, rew=30.0, fairness=True,
               workload="rmappo rollout loop at 3 agents: dense GNN actor + critic forward (torch) -> fused simulator step writing "
                        "the device-resident rollout buffer -> insert; sampled actions"),
}


def select_config(name: str, envs: int | None):
    global N_AGENTS, N_OBST, ENVS_PER_GPU, WORKLOAD, GOAL_REW, COLL_REW, FAIRNESS
    c = CONFIGS[name]
    N_AGENTS, N_OBST, WORKLOAD = c["agents"], c["obstacles"], c["workload"]
    GOAL_REW = COLL_REW = c["rew"]
    FAIRNESS = c["fairness"]
    ENVS_PER_GPU = envs if envs else c["envs"]


def lookup_traffic_entry(table: dict, kernel_name: str, envs_per_gpu: int, walls: int):
    """Entry of profiles/step_kernel_traffic.json (one ncu --set full capture) that matches this run, else None."""
    for key, ent in table.get("by_kernel", {}).items():
        if kernel_name.startswith(key + " ") and ent.get("envs_per_gpu") == envs_per_gpu and ent.get("walls", 0) == walls:
            return ent
    return None


def lookup_traffic(table: dict, kernel_name: str, envs_per_gpu: int, walls: int):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the ncu capture that matches this run, else None."""
    ent = lookup_traffic_entry(table, kernel_name, envs_per_gpu, walls)
    return ent.get("dram_bytes_per_launch") if ent else None


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path: str, per_env: dict, whole: dict) -> None:
    """``--dump-outputs``: write every array as ``path/<name>.npy`` (float64 stays float64, the rest becomes float32).
    ``per_env`` arrays have the env index first; if all arrays together exceed DUMP_LIMIT_BYTES, every per-env array
    keeps the same env rows: a sample drawn with a fixed seed from the batch size alone, in ascending env order."""
    import numpy as np
    as_float = lambda a: np.asarray(a, dtype=np.float64 if a.dtype == np.float64 else np.float32)
    per_env = {k: as_float(v) for k, v in per_env.items()}
    whole = {k: as_float(v) for k, v in whole.items()}
    B = next(iter(per_env.values())).shape[0]
    row_bytes = sum(v.nbytes // B for v in per_env.values())
    room = DUMP_LIMIT_BYTES - sum(v.nbytes for v in whole.values()) - 4096        # 4096: the .npy headers
    if row_bytes * B > room:
        rows = np.sort(np.random.default_rng(0).choice(B, room // row_bytes, replace=False))
        per_env = {k: v[rows] for k, v in per_env.items()}
    os.makedirs(path, exist_ok=True)
    for name, a in {**per_env, **whole}.items():
        np.save(os.path.join(path, name + ".npy"), a)


def sim_kwargs():
    kw = dict(num_agents=N_AGENTS, num_obstacles=N_OBST, goal_rew=GOAL_REW, collision_rew=COLL_REW,
              episode_length=EPISODE, fairness_reward=FAIRNESS)
    if N_WALLS:
        kw["num_walls"] = N_WALLS
    return kw


# ----------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the run (NVML, the library behind nvidia-smi;
    falls back to the nvidia-smi query of B200_PROFILING.md)."""

    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index: int, period: float = 0.02):
        self.index, self.period = index, period
        self.samples = []          # (t, sm_mhz, reasons_mask)
        self.sm_max = None
        self._stop = threading.Event()
        self._thread = None
        self._nvml = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._dev = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.sm_max = int(pynvml.nvmlDeviceGetMaxClockInfo(self._dev, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nvml = None
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()

    def sample_now(self):
        """One sample taken by the calling thread (NVML only)."""
        try:
            if self._nvml is not None:
                n = self._nvml
                mhz = int(n.nvmlDeviceGetClockInfo(self._dev, n.NVML_CLOCK_SM))
                mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(self._dev)) if hasattr(
                    n, "nvmlDeviceGetCurrentClocksEventReasons") else int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self._dev))
                self.samples.append((time.perf_counter(), mhz, mask))
        except Exception:
            pass

    def _run(self):
        import subprocess
        while not self._stop.is_set():
            try:
                if self._nvml is not None:
                    n = self._nvml
                    mhz = int(n.nvmlDeviceGetClockInfo(self._dev, n.NVML_CLOCK_SM))
                    mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(self._dev)) if hasattr(
                        n, "nvmlDeviceGetCurrentClocksEventReasons") else int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self._dev))
                    self.samples.append((time.perf_counter(), mhz, mask))
                else:
                    q = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=clocks.sm,clocks.max.sm,"
                                        "clocks_event_reasons.active", "--format=csv,noheader,nounits"],
                                       capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                    self.sm_max = int(q[1])
                    self.samples.append((time.perf_counter(), int(q[0]), int(q[2].strip(), 16)))
            except Exception:
                pass
            self._stop.wait(self.period)

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=2)

    def summary(self, t0: float, t1: float) -> dict:
        inside = [s for s in self.samples if t0 <= s[0] <= t1]
        scope = "timed_region"
        if not inside:                       # region shorter than the sampling period
            inside, scope = self.samples, "whole_run"
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": [], "samples": 0, "scope": "none"}
        mask = 0
        for s in inside:
            mask |= s[2]
        reasons = [name for bit, name in self.REASONS.items() if mask & bit and name != "gpu_idle"]
        return {"sm_mhz": statistics.median(s[1] for s in inside), "sm_max_mhz": self.sm_max, "reasons": reasons,
                "samples": len(inside), "scope": scope}


# ----------------------------------------------------------------------------------------------
def _cpu_worker(args):
    """One host process: B envs of the numpy oracle, `steps` steps with auto-reset."""
    seed, B, steps, warm, config = args
    select_config(config, None)
    import numpy as np
    from oracle.navgraph import NavConfig, NavGraphOracle
    cfg = NavConfig(**sim_kwargs())
    orc = NavGraphOracle(cfg, B, seed=seed, env_offset=seed * B)
    orc.reset()
    rng = np.random.default_rng(seed)
    acts = rng.integers(0, 5, (steps + warm, B, N_AGENTS))
    for k in range(warm):
        orc.step(actions=acts[k])
    t0 = time.perf_counter()
    for k in range(warm, warm + steps):
        orc.step(actions=acts[k])
    return time.perf_counter() - t0


def cpu_port_throughput(steps: int, warm: int, envs_per_proc: int = 2048, config: str = "c2"):
    """agent-steps/s of the oracle port on all host cores (one process per core, env-sharded)."""
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    ctx = mp.get_context("spawn")
    t0 = time.perf_counter()
    with ctx.Pool(cores) as pool:
        times = pool.map(_cpu_worker, [(r, envs_per_proc, steps, warm, config) for r in range(cores)])
    wall = time.perf_counter() - t0
    worst = max(times)
    value = cores * envs_per_proc * N_AGENTS * steps / worst
    sample = (f"{cores} procs x {envs_per_proc} envs x {steps} steps of the same workload "
              f"(slowest proc {worst:.2f}s, pool wall {wall:.1f}s incl. spawn)")
    return value, cores, sample, worst / steps * 1e3


def run_reference(args, rank: int, world: int):
    if rank != 0:
        return
    steps, warm = args.steps, max(0, args.warmup)
    value, cores, sample, ms = cpu_port_throughput(steps, warm, config=args.config)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "agent-steps/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "envs_per_step": cores * 2048, "note": "CPU port of the reference path; "
                   "a step here is one oracle step over the bounded sample batch"},
        "cpu_baseline": {"value": value, "unit": "agent-steps/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
def run_rollout(args, rank: int, local_rank: int, world: int):
    """BASELINE config 5 (diagnostic line, not the headline): GMPERunner's collect -> step -> insert loop with the
    dense torch policy and the device-resident rollout buffer.  A step = one env step of the whole batch including
    the actor + critic forward that produced its actions.  Envs are sharded over ranks (weak scaling), policy
    parameters are replicated; there is no collective on this path."""
    import torch
    import torch.distributed as dist
    import fair_marl_b200 as fm

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.envs
    cfg = fm.SimConfig(**sim_kwargs(), mapping=args.mapping)
    env = fm.B200GraphVecEnv(cfg, num_envs=B, device=local_rank, seed=0, env_offset=rank * B)
    pc = fm.PolicyConfig(num_agents=N_AGENTS)
    torch.manual_seed(0)
    actor, critic = fm.DenseGraphActor(pc).to(dev).eval(), fm.DenseGraphCritic(pc).to(dev).eval()
    col = fm.RolloutCollector(env, actor, critic, max_graphs=args.max_graphs,
                              generator=torch.Generator(device=dev).manual_seed(1234 + rank))
    col.warmup()
    episodes = args.steps // EPISODE               # main() admits whole episodes only
    K = episodes * EPISODE
    col.run()                                       # warm-up episode (allocator, library handles)
    col.buffer.after_update()
    graph = "eager"
    if not args.no_graph:
        try:
            col.capture()
            col.run()                                   # one replay before timing
            col.buffer.after_update()
            graph = "one CUDA graph per episode"
        except Exception as exc:                        # noqa: BLE001 -- report and time the eager loop
            graph = f"eager (capture failed: {type(exc).__name__}: {exc})"[:200]
    torch.cuda.synchronize(dev)
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.05)
    if world > 1:
        dist.barrier()
    launches0 = env.kernel_launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    ev0.record()
    for _ in range(episodes):
        col.run()
        col.buffer.after_update()
    ev1.record()
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    t1 = time.perf_counter()
    elapsed_ms = ev0.elapsed_time(ev1)
    # the simulator's share: the same number of steps without the policy (same buffer slabs, recorded actions)
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    for _ in range(episodes):
        for t in range(EPISODE):
            env.step_tensor(col.buffer.actions_env[t], out=col.buffer.env_views(t + 1))
    s1.record()
    torch.cuda.synchronize(dev)
    sim_ms = s0.elapsed_time(s1)
    launches = env.kernel_launches - launches0
    clocks = sampler.summary(t0, t1)
    sampler.stop()
    if world > 1:
        tt = torch.tensor([elapsed_ms, sim_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        elapsed_ms, sim_ms = float(tt[0].item()), float(tt[1].item())
    if rank == 0:
        value = B * world * N_AGENTS * K / (elapsed_ms * 1e-3)
        line = {
            "metric": "agent-steps/sec, rollout loop (policy forward + navigation_graph step + buffer insert)", "value": value,
            "unit": "agent-steps/s", "n_gpus": world, "steps": K, "warmup": EPISODE, "ms_per_step": elapsed_ms / K,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "envs_per_gpu": B, "envs_total": B * world, "agents": N_AGENTS,
                       "policy": "DenseGraphActor + DenseGraphCritic (EmbedConv 16 -> 3 x TransformerConv 3 heads x 16 -> MLP 64 -> GRU 64), "
                                 "random init, sampled actions", "policy_chunk_graphs": args.max_graphs,
                       "buffer": f"DeviceRolloutBuffer, {EPISODE + 1} slabs written in place by the step kernel",
                       "launch": graph},
            "simulator_share": {"ms_per_step": sim_ms / K, "frac_of_step": sim_ms / elapsed_ms,
                                "api": "step_tensor(out=buffer slab): one launch per step"},
            "gpu_launches": launches, "clocks": clocks,
            "mem_gb": torch.cuda.max_memory_allocated(dev) / 1e9,
        }
        print(json.dumps(line), flush=True)
    env.close()
    if world > 1:
        dist.destroy_process_group()


def run_formation(args, rank: int, local_rank: int, world: int):
    """Widened row N3 (diagnostic line, not the headline): the formation-family scenario the shipped weights were trained on
    (nav_fairassign_fairrew_formation_graph, 3 agents / 3 goals / 3 obstacles, FA+FR, reward 30, per-step lexifair
    re-assignment) -- fm_formation_step_many rollouts over pre-generated random actions (per step a logic kernel and an image
    kernel), auto-reset inside the timed region; `closed_loop`: one fm_formation_step call
    per step."""
    import torch
    import torch.distributed as dist
    import fair_marl_b200 as fm

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, K, W = args.envs, args.steps, max(args.warmup, 3)
    N, O = N_AGENTS, N_OBST
    E = 2 * N + O
    cfg = fm.FormationSimConfig(num_agents=N, num_obstacles=O, goal_rew=GOAL_REW, collision_rew=COLL_REW, episode_length=EPISODE,
                                fairness_reward=FAIRNESS, info_every_step=False)
    env = fm.B200FormationVecEnv(cfg, num_envs=B, device=local_rank, seed=0, env_offset=rank * B, num_slots=args.form_slots)
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    actions = torch.randint(0, 5, (EPISODE, B, N), generator=g, device=dev, dtype=torch.int32)
    def run_steps(n, phase):
        """n steps from action-table phase `phase` as fm_formation_step_many rollouts (chunks end at the table's end)."""
        while n > 0:
            t = min(n, EPISODE - phase)
            env.rollout_tensor(actions[phase:phase + t])
            n -= t
            phase = (phase + t) % EPISODE
        return phase

    # dry run of the exact call sequence (lane stream, kernel attributes), then the measured one from the same state
    env.reset_tensor()
    ph = run_steps(W, 0)
    run_steps(K, ph)
    torch.cuda.synchronize(dev)
    env.reset_tensor()
    ph = run_steps(W, 0)
    torch.cuda.synchronize(dev)
    sampler = ClockSampler(local_rank, period=0.0005)
    sampler.start()
    time.sleep(0.02)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    ev0.record()
    run_steps(K, ph)
    ev1.record()
    sampler.sample_now()
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    t1 = time.perf_counter()
    elapsed_ms = ev0.elapsed_time(ev1)
    clocks = sampler.summary(t0, t1)
    sampler.stop()
    if world > 1:
        tt = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        elapsed_ms = float(tt.item())
    # closed loop: one fm_formation_step call per step (what a policy in the loop uses)
    Kc = max(K, 100)
    for k in range(10):
        env.step_tensor(actions[k % EPISODE])
    torch.cuda.synchronize(dev)
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for k in range(Kc):
        env.step_tensor(actions[k % EPISODE])
    c1.record()
    torch.cuda.synchronize(dev)
    closed_ms = c0.elapsed_time(c1) / Kc
    # algorithmic bytes per env-step, counted like SURVEY 8(d): state read once + dynamic state written once + every output once
    words = (17 * N + 2 * O + 4 + N / 4) + (14 * N + 3 + N / 4) + (11 * N + 13 * N * E + E * E + N + N / 4)
    alg_bytes = int(words * 4 * B)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak = float(json.load(open(peaks_path))["hbm_gbs"]) if os.path.isfile(peaks_path) else 6650.0
    achieved = alg_bytes / (elapsed_ms / K * 1e-3) / 1e9
    if rank == 0:
        line = {
            "metric": "agent-steps/sec, formation-family step+obs+reward+per-step assignment", "value": B * world * N * K / (elapsed_ms * 1e-3),
            "unit": "agent-steps/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": elapsed_ms / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64 logic / f32 state", "data": "synthetic",
            "config": {"workload": "nav_fairassign_fairrew_formation_graph 3 agents / 3 goals / 3 obstacles, FA+FR, goal_rew=collision_rew=30, "
                                   "episode_length 25 with auto-reset, lexifair re-assignment every step, random actions",
                       "envs_per_gpu": B, "envs_total": B * world, "agents": N, "entities": E,
                       "launch": "fm_formation_step_many, one call per chunk of steps", "l2": f"outputs cycle through {args.form_slots} buffer sets ({args.form_slots * B * (11 * N + 13 * N * E + E * E + N) * 4 / 1e9:.2f} GB > 126 MB L2)"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                         "kernel": f"fm::formation_logic_kernel<{N}, {O}> + fm::formation_image_kernel<{N}, {O}> (+ fm::formation_prefetch_kernel<{N}> on a side stream)",
                         "algorithmic_bytes_per_step": alg_bytes,
                         "note": "a step is three launches: logic (thread per env) -> image (node_obs / adj from the recipes; programmatic "
                                 "dependent launch), and the pending-reset prefetch on a side stream; the "
                                 "bytes are those of the whole step, the time is the whole step's"},
            "cpu_baseline": None, "e2e": None,
            "closed_loop": {"value": B * world * N / (closed_ms * 1e-3), "unit": "agent-steps/s", "ms_per_step": closed_ms, "steps": Kc,
                            "frac": alg_bytes / (closed_ms * 1e-3) / 1e9 / peak,
                            "api": "B200FormationVecEnv.step_tensor -> fm_formation_step, one call per step"},
            "gpu_launches": 3 * K, "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    env.close()
    if world > 1:
        dist.destroy_process_group()


def run_ours(args, rank: int, local_rank: int, world: int):
    import numpy as np
    import torch
    import torch.distributed as dist
    import fair_marl_b200 as fm

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback; use --impl reference for the CPU port)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.envs
    K, W = args.steps, args.warmup
    cfg = fm.SimConfig(**sim_kwargs(), mapping=args.mapping)
    E = cfg.num_entities
    out_bytes = B * (N_AGENTS * 7 + N_AGENTS * E * 11 + E * E + N_AGENTS) * 4 + B * N_AGENTS
    slots = max(2, min(EPISODE, int(12e9 // out_bytes)))        # ring > L2, bounded to ~12 GB of HBM
    slab_gb = slots * out_bytes / 1e9
    env = fm.B200GraphVecEnv(cfg, num_envs=B, device=local_rank, seed=0, env_offset=rank * B, num_slots=slots)
    args.graph = args.step_graph == "on" or (args.step_graph == "auto" and K <= 250 and env.mapping == "aw")
    stats = fm.EpisodeStats(N_AGENTS, device=dev)

    # synthetic random actions for one episode, resident in HBM before the timed region
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    actions = torch.randint(0, 5, (EPISODE, B, N_AGENTS), generator=g, device=dev, dtype=torch.int32)
    stats_vec = torch.empty(env.lib.fm_stats_len(N_AGENTS), dtype=torch.float64, device=dev)
    Wn = max(W, 3)
    # Episode phase at which the warm-up starts, chosen so that a terminal step (auto-reset + lexifair + statistics
    # reduction + all-reduce) lies in the MIDDLE of the timed region, as in a long rollout: its all-reduce then overlaps
    # the following steps instead of being the last thing the timer waits for.
    phase0 = (-(Wn + (K + 1) // 2)) % EPISODE

    graphs = {}                                   # (phase, steps, slot) -> captured fm_step_many launch sequence
    replayed = [0]                                # kernels launched through graph replays (the handle counts eager launches only)

    def rollout_chunk(phase, t):
        if not args.graph:
            env.rollout_tensor(actions[phase:phase + t])
            return
        key = (phase, t, env._slot)
        g = graphs.get(key)
        if g is None:                             # captured during the dry run, replayed in the timed region
            torch.cuda.synchronize(dev)
            slot0, n0 = env._slot, env.kernel_launches
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                env.rollout_tensor(actions[phase:phase + t])
            graphs[key] = (g, env._slot, env.kernel_launches - n0)
            env._slot = slot0
            g = graphs[key]
        g[0].replay()
        env._slot = g[1]
        replayed[0] += g[2]

    def run_steps(n, phase):
        """n env steps from episode phase `phase`, in chunks that end at episode boundaries; every terminal step is
        followed by the statistics reduction and its all-reduce (side stream).  Returns the new phase."""
        while n > 0:
            t = min(n, EPISODE - phase)
            rollout_chunk(phase, t)
            n -= t
            phase = (phase + t) % EPISODE
            if phase == 0:
                stats.all_reduce_async(env.read_stats(out=stats_vec))
        return phase

    def prepare():
        env.reset_tensor()
        env._slot = 0                             # same walk through the slab ring in the dry run and in the measured run
        return run_steps(phase0, 0)

    # One GPU: the whole timed sequence (rollout chunks, statistics reductions) is ONE captured graph.  Several GPUs: one
    # graph per rollout chunk; the NCCL all-reduce between them stays an eager launch on the side stream.
    region = {}

    def timed_sequence(phase):
        if not (args.graph and world == 1):
            run_steps(K, phase)
            stats.join()
            return
        if "g" not in region:                     # captured in the dry run below, replayed in the timed region
            torch.cuda.synchronize(dev)
            slot0, n0 = env._slot, env.kernel_launches
            saved, args.graph = args.graph, False          # the region graph holds the eager launches themselves
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                run_steps(K, phase)
                stats.join()
            args.graph = saved
            region["g"], region["slot"], region["kernels"] = g, env._slot, env.kernel_launches - n0
            env._slot = slot0
        region["g"].replay()
        env._slot = region["slot"]
        replayed[0] += region["kernels"]

    # dry run of the exact call sequence (plans, lazily created streams / buffers, NCCL channels, graphs), then the real one
    ph = prepare()
    ph = run_steps(Wn, ph)
    timed_sequence(ph)
    torch.cuda.synchronize(dev)
    env.read_stats(clear=True, out=stats_vec)
    ph = prepare()
    ph = run_steps(Wn, ph)
    stats.join()
    torch.cuda.synchronize(dev)
    sampler = ClockSampler(local_rank, period=0.0005)
    sampler.start()
    time.sleep(0.02)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    launches0 = env.kernel_launches
    replayed[0] = 0
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    ev0.record()
    timed_sequence(ph)                            # incl. stats.join(): the all-reduce of the region's terminal steps is inside
    ev1.record()
    sampler.sample_now()                          # one NVML read by this thread while the GPU is still working on the region
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    t1 = time.perf_counter()
    sampler.period = 0.02
    launches = (env.kernel_launches - launches0) + replayed[0]           # eager launches + kernels inside the replayed graphs
    elapsed_ms = ev0.elapsed_time(ev1)
    clocks = sampler.summary(t0, t1)
    if world > 1:
        tt = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        elapsed_ms = float(tt.item())
    value = B * world * N_AGENTS * K / (elapsed_ms * 1e-3)
    total_stats = stats.summary()
    if args.dump_outputs and rank == 0:          # before the closed-loop and e2e steps below overwrite the slab ring
        last = env.slot_outputs(env._slot)       # the slab the last timed step wrote
        dump_outputs(args.dump_outputs,
                     {k: last[k].cpu().numpy() for k in ("obs", "node_obs", "adj_env", "reward", "done", "info")},
                     {"episode_stats": stats.result().cpu().numpy()})

    # roofline of the step kernel: algorithmic bytes per launch / average launch duration
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    alg_bytes = env.algorithmic_bytes_per_step
    kernel_name = {"aw": (f"fm::aw_roll_kernel<{N_AGENTS},{N_OBST},11> (agent-warp, persistent rollout)"
                          if os.environ.get("FM_ROLL", "0") not in ("", "0") else (f"fm::aw_kernel<{N_AGENTS},{N_OBST},0,11,{N_WALLS}> (agent-warp, {N_WALLS} wall(s))" if N_WALLS
                                else f"fm::aw_kernel<{N_AGENTS},{N_OBST},0> (agent-warp)")),
                   "group": f"fm::step_kernel<{4 if N_AGENTS <= 4 else 8 if N_AGENTS <= 8 else 16 if N_AGENTS <= 16 else 32}{', true' if N_WALLS else ''}> (group-per-env)"}[env.mapping]
    # One step = the step kernel's work over the whole batch (agent-warp mapping: (step, tile) items of one persistent
    # launch per chunk of steps; group mapping: concurrent env-range launches on side streams); that kernel is > 99 %
    # of the timed region (profiles/: launch list), so bytes per step / time per step is its achieved algorithmic bandwidth.
    step_kernel_ms = elapsed_ms / K              # rank-max
    achieved = alg_bytes / (step_kernel_ms * 1e-3) / 1e9
    traffic = traffic_alg = None
    tpath = os.path.join(ROOT, "profiles", "step_kernel_traffic.json")
    if os.path.isfile(tpath):                    # ncu --set full captures, per launch; only the entry of THIS kernel / size
        ent = lookup_traffic_entry(json.load(open(tpath)), kernel_name, B, N_WALLS)
        if ent:                                  # one captured launch = one env-range lane of fm_step_many (half a step)
            traffic, traffic_alg = ent.get("dram_bytes_per_launch"), ent.get("algorithmic_bytes_per_launch")
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_launch_algorithmic_bytes": traffic_alg, "kernel": kernel_name,
                "algorithmic_bytes_per_step": alg_bytes,
                "launches_per_step": launches / K, "peak_source": peak_src,
                "note": "the SoA state (14 % of the algorithmic bytes) is L2-resident between steps; the outputs "
                        "(86 %) stream to HBM through a slab ring larger than L2"}

    # closed loop: one fm_step per call (what a policy-in-the-loop rollout does), no host sync in between
    cl_steps = max(200, min(K, 1000))
    for k in range(3):
        env.step_tensor(actions[k])
    torch.cuda.synchronize(dev)
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for k in range(cl_steps):
        env.step_tensor(actions[k % EPISODE])
    c1.record()
    torch.cuda.synchronize(dev)
    cl_ms = c0.elapsed_time(c1)
    if world > 1:
        tt = torch.tensor([cl_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        cl_ms = float(tt.item())
    closed_loop = {"value": B * world * N_AGENTS * cl_steps / (cl_ms * 1e-3), "unit": "agent-steps/s",
                   "ms_per_step": cl_ms / cl_steps, "steps": cl_steps,
                   "api": "B200GraphVecEnv.step_tensor -> fm_step, one launch per step (programmatic dependent launch behind the previous step), device tensors"}

    # policy-side edge list (a-7, process_adj) emitted after every step: SURVEY 8(d) asks for it at config 3
    edge_list = None
    if args.edge_list or args.config == "c3":
        import ctypes as C
        from fair_marl_b200 import _lib
        lib = _lib.load()
        cap = B * E * E                                  # what always suffices (include/fairmarl.h): no capacity tests in the emission
        offsets = torch.empty(B + 1, dtype=torch.int64, device=dev)
        eidx = torch.empty((2, cap), dtype=torch.int64, device=dev)
        eattr = torch.empty(cap, dtype=torch.float32, device=dev)
        nnz = torch.zeros(1, dtype=torch.int64, device=dev)
        stream = torch.cuda.current_stream(dev).cuda_stream

        def step_and_edges(k):
            o = env.step_tensor(actions[k % EPISODE])
            _lib.check(lib.fm_edge_list(local_rank, o["adj_env"].data_ptr(), B, E, float(cfg.max_edge_dist), 0, 1, cap,
                                        offsets.data_ptr(), eidx.data_ptr(), eattr.data_ptr(), nnz.data_ptr(), stream), "fm_edge_list")
        el_steps = min(K, 100)
        for k in range(3):
            step_and_edges(k)
        torch.cuda.synchronize(dev)
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for k in range(el_steps):
            step_and_edges(k)
        g1.record()
        torch.cuda.synchronize(dev)
        el_ms = g0.elapsed_time(g1) / el_steps
        n_edges = int(nnz.item())
        edge_list = {"ms_per_step_with_edge_list": el_ms, "ms_per_step_closed_loop": closed_loop["ms_per_step"],
                     "edges_per_step": n_edges, "edge_bytes_per_step": n_edges * 20,
                     "value": B * N_AGENTS / (el_ms * 1e-3), "unit": "agent-steps/s",
                     "api": "step_tensor + fm_edge_list (form %s: one graph per env, int64 edge_index + fp32 attr)" % os.environ.get("FM_EDGE_FORM", "stream")}

    # e2e through the reference-facing API with host buffers
    e2e_steps = max(3, min(args.e2e_steps, K))
    rng = np.random.default_rng(rank)
    eye = np.eye(5, dtype=np.float32)
    host_actions = [eye[rng.integers(0, 5, (B, N_AGENTS))] for _ in range(4)]
    for k in range(3):
        env.step(host_actions[k % 4])
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    te0 = time.perf_counter()
    for k in range(e2e_steps):
        obs, ag_id, node, adj, rew, done, infos = env.step(host_actions[k % 4])
    torch.cuda.synchronize(dev)
    te = time.perf_counter() - te0
    if world > 1:
        tt = torch.tensor([te], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        te = float(tt.item())
    sampler.stop()
    h2d = B * N_AGENTS * 5 * 4
    d2h = B * (N_AGENTS * 7 + N_AGENTS * E * 11 + E * E + N_AGENTS) * 4 + B * N_AGENTS
    e2e = {"value": B * world * N_AGENTS * e2e_steps / te, "unit": "agent-steps/s", "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": d2h, "steps": e2e_steps, "ms_per_step": te / e2e_steps * 1e3,
           "api": "B200GraphVecEnv.step(actions_env) -> fm_step_host (pinned host buffers)"}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        per_proc = 2048 if N_AGENTS <= 4 else (512 if N_AGENTS <= 8 else 128)
        v, cores, sample, _ = cpu_port_throughput(100, 5, envs_per_proc=per_proc, config=args.config)
        cpu = {"value": v, "unit": "agent-steps/s", "cores": cores, "kind": "port", "sample": sample}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "agent-steps/s", "n_gpus": world, "steps": K, "warmup": max(W, 3),
            "ms_per_step": elapsed_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "envs_per_gpu": B, "envs_total": B * world, "agents": N_AGENTS,
                       "entities": E, "sharding": f"env-index x{world}" if world > 1 else "single GPU",
                       "l2": f"outputs cycle through a {slots}-slot slab ring ({slab_gb:.1f} GB per GPU > 126 MB L2); the SoA "
                             "state is read+written every step",
                       "stats_allreduce": ("after every terminal step, side stream, joined before the timer stops" if world > 1
                                           else "local reduce after every terminal step"),
                       "episode_phase_at_start": (phase0 + Wn) % EPISODE,
                       "launch": ("fm_step_many: one persistent kernel per chunk of steps (chunks end at episode boundaries)"
                                  if env.mapping == "aw" and os.environ.get("FM_ROLL", "0") not in ("", "0") else
                                  "fm_step_many: one-shot step kernels on env-range lanes (side streams)") +
                                 ((", the region's call sequence replayed as ONE captured CUDA graph" if world == 1 else
                                   ", every chunk replayed as a captured CUDA graph") if args.graph else ", eager launches")},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "closed_loop": closed_loop, "edge_list": edge_list,
            "gpu_launches": launches, "clocks": clocks,
            "episode_stats": {"episodes": total_stats["episodes"], "env_steps": total_stats["env_steps"]},
        }
        print(json.dumps(line), flush=True)
    env.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    global N_WALLS, WORKLOAD
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5000)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=None, help="envs per GPU (default: the config's)")
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS), help="BASELINE.json config (headline: c2)")
    ap.add_argument("--e2e-steps", type=int, default=50)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--mapping", default="auto", choices=["auto", "group", "aw"], help="kernel mapping (diagnostic)")
    ap.add_argument("--max-graphs", type=int, default=1 << 17, help="c5: graphs per policy forward chunk")
    ap.add_argument("--edge-list", action="store_true", help="also time step + policy-side edge list (default on for c3)")
    ap.add_argument("--walls", type=int, default=0, choices=[0, 1, 2], help="diagnostic: num_walls (wall kernels, SURVEY N4)")
    ap.add_argument("--no-graph", action="store_true", help="c5: time the eager loop instead of the captured CUDA graph")
    ap.add_argument("--form-slots", type=int, default=8, help="form: output buffer sets the steps cycle through")
    ap.add_argument("--step-graph", default="auto", choices=["auto", "on", "off"],
                    help="replay the timed region's fm_step_many call sequence from a captured CUDA graph.  auto: for short "
                         "regions (<= 250 steps) on the agent-warp mapping, where launch latency is what a graph removes; long "
                         "regions keep a deep eager launch queue anyway (measured: 0.93 eager vs 0.87 replayed at 5000 steps), "
                         "and the group mapping's next-episode prefetch is a host-side decision that a replay cannot make")
    ap.add_argument("--no-step-graph", dest="step_graph", action="store_const", const="off")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (obs, node_obs, adj_env, reward, done, "
                         "info; a fixed env sample if above 64 MB) and the episode statistics as DIR/<name>.npy (rank 0); "
                         "configs c1-c4")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.config == "c5" and args.impl == "ours" and args.steps % EPISODE:
        ap.error(f"--config c5 times whole episodes: --steps must be a multiple of {EPISODE}")
    if args.dump_outputs and (args.impl == "reference" or args.config in ("c5", "form")):
        ap.error("--dump-outputs covers the step configs c1-c4 of --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    select_config(args.config, args.envs)
    args.envs = ENVS_PER_GPU
    if args.walls:
        N_WALLS = args.walls
        WORKLOAD += f" + {args.walls} wall(s) [diagnostic, not a BASELINE config]"
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit(f"bench.py --gpus {args.gpus} must be launched with torchrun --nproc-per-node {args.gpus}")
    if args.config == "c5":
        run_rollout(args, rank, local_rank, world)
        return
    if args.config == "form":
        run_formation(args, rank, local_rank, world)
        return
    run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
