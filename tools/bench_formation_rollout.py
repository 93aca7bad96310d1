"""Cost of the formation-family episode statistics and throughput of the device rollout loop on this family, in one process
on one GPU (the card's name and power limit are recorded beside the numbers).

  (a) fm_formation_step_many at 65 536 envs x 3 agents, FA+FR (bench.py --config form's workload), statistics off and on
      on the same handle (fm_formation_stats_enable toggled), alternated and repeated: us per step and the spread.
  (b) RolloutCollector with one captured CUDA graph per episode (policy PolicyConfig(obs_dim=11, node_feat_dim=13), fused
      graph network, sampled actions, statistics on as make_train_env builds the env) at 4 096 and 65 536 envs: agent-steps/s,
      and the simulator's share (a captured graph of the episode's env steps alone, writing the same buffer slabs).
  (c) with --main-tree: `bench.py --config form` of that tree and of this one, alternated in this call.

    python tools/bench_formation_rollout.py --out DIR [--main-tree PATH] [--repeats R]
    python tools/bench_formation_rollout.py --out DIR --profile      # per-kernel breakdown of (a), a run of its own

Writes DIR/bench_formation_rollout.json (--profile: DIR/bench_formation_rollout_profile.json) and prints it.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N, O, EPISODE = 3, 3, 25


def gpu_info():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def spread(xs):
    med = statistics.median(xs)
    return {"runs": xs, "median": med, "min": min(xs), "max": max(xs), "spread_rel": (max(xs) - min(xs)) / med}


def sim_config(**kw):
    import fair_marl_b200 as fm
    return fm.FormationSimConfig(num_agents=N, num_obstacles=O, goal_rew=30.0, collision_rew=30.0, episode_length=EPISODE,
                                 fairness_reward=True, **kw)


def part_a(repeats: int, steps: int):
    """step_many, statistics off / on alternated on one handle (same state sequence for both)."""
    import torch
    import fair_marl_b200 as fm
    B = 65536
    env = fm.B200FormationVecEnv(sim_config(info_every_step=False), num_envs=B, seed=0, num_slots=8, episode_stats=True)
    g = torch.Generator(device="cuda").manual_seed(1234)
    actions = torch.randint(0, 5, (EPISODE, B, N), generator=g, device="cuda", dtype=torch.int32)
    stream = env._stream()

    def run(n):
        ph = 0
        while n > 0:
            t = min(n, EPISODE - ph)
            env.rollout_tensor(actions[ph:ph + t])
            n -= t
            ph = (ph + t) % EPISODE

    env.reset_tensor()
    res = {"off": [], "on": []}
    for mode in ("off", "on"):                                  # warm both variants
        fm._lib.check(env.lib.fm_formation_stats_enable(env._h, int(mode == "on"), stream))
        run(2 * EPISODE)
    torch.cuda.synchronize()
    for r in range(repeats):
        for mode in (("off", "on") if r % 2 == 0 else ("on", "off")):
            fm._lib.check(env.lib.fm_formation_stats_enable(env._h, int(mode == "on"), stream))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run(steps)
            e1.record()
            torch.cuda.synchronize()
            res[mode].append(e0.elapsed_time(e1) * 1e3 / steps)
    fm._lib.check(env.lib.fm_formation_stats_enable(env._h, 1, stream))
    vec = env.read_stats().cpu()
    env.close()
    out = {k: spread(v) for k, v in res.items()}
    out["on_minus_off_us"] = out["on"]["median"] - out["off"]["median"]
    out["config"] = {"envs": B, "agents": N, "obstacles": O, "scenario": "FA+FR", "episode_length": EPISODE, "steps_per_run": steps,
                     "actions": "random", "outputs": "8 slots round robin (> L2)", "info_every_step": False,
                     "episodes_counted_while_on": float(vec[15 * N])}
    return out


def part_a_profile(out_dir: str, episodes: int = 4):
    """Where the statistics cost goes: torch.profiler kernel times of `episodes` episodes of single steps with statistics
    off, then on (same handle), per kernel name; the logic kernel's time split into the terminal steps (every env times
    out together under random actions: info sums) and the others.  A run of its own (tracing slows the host)."""
    import torch
    import fair_marl_b200 as fm
    from torch.profiler import ProfilerActivity, profile
    B = 65536
    env = fm.B200FormationVecEnv(sim_config(info_every_step=False), num_envs=B, seed=0, num_slots=8, episode_stats=True)
    g = torch.Generator(device="cuda").manual_seed(1234)
    actions = torch.randint(0, 5, (EPISODE, B, N), generator=g, device="cuda", dtype=torch.int32)
    stream = env._stream()
    env.reset_tensor()
    for t in range(2 * EPISODE):
        env.step_tensor(actions[t % EPISODE])
    torch.cuda.synchronize()
    res = {}
    for mode in ("off", "on"):
        fm._lib.check(env.lib.fm_formation_stats_enable(env._h, int(mode == "on"), stream))
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for t in range(episodes * EPISODE):
                env.step_tensor(actions[t % EPISODE])
            torch.cuda.synchronize()
        evs = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA), key=lambda e: e.time_range.start)
        per = {}
        for e in evs:
            d = per.setdefault(e.name, [])
            d.append(e.time_range.elapsed_us())
        logic = next((v for k, v in per.items() if "formation_logic_kernel" in k), [])
        res[mode] = {"kernels_us_mean": {k: sum(v) / len(v) for k, v in per.items()}, "launches": {k: len(v) for k, v in per.items()},
                     "logic_terminal_steps_us": [x for i, x in enumerate(logic) if i % EPISODE == EPISODE - 1],
                     "logic_other_steps_us_mean": statistics.mean([x for i, x in enumerate(logic) if i % EPISODE != EPISODE - 1])}
    env.close()
    with open(os.path.join(out_dir, "bench_formation_rollout_profile.json"), "w") as f:
        f.write(json.dumps(res, indent=1))
    return res


def part_b(B: int, episodes: int):
    import torch
    import fair_marl_b200 as fm
    env = fm.B200FormationVecEnv(sim_config(info_every_step=False), num_envs=B, seed=0, episode_stats=True)
    pc = fm.PolicyConfig(num_agents=N, obs_dim=11, node_feat_dim=13)
    torch.manual_seed(0)
    actor, critic = fm.DenseGraphActor(pc).cuda().eval(), fm.DenseGraphCritic(pc).cuda().eval()
    col = fm.RolloutCollector(env, actor, critic, generator=torch.Generator(device="cuda").manual_seed(1))
    buf = col.buffer
    col.warmup(); col.run(); buf.after_update()
    col.capture()
    col.run(); buf.after_update()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(episodes):
        col.run(); buf.after_update()
    e1.record()
    torch.cuda.synchronize()
    loop_ms = e0.elapsed_time(e1) / episodes
    # the simulator alone: the episode's T env steps into the same slabs, captured as one graph
    g = torch.cuda.CUDAGraph()
    torch.cuda.synchronize()
    with torch.cuda.graph(g):
        for t in range(EPISODE):
            env.step_tensor(buf.actions_env[t], out=buf.env_views(t + 1))
    g.replay()
    torch.cuda.synchronize()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    for _ in range(episodes):
        g.replay()
    s1.record()
    torch.cuda.synchronize()
    sim_ms = s0.elapsed_time(s1) / episodes
    stats = env.read_stats().cpu()
    env.close()
    return {"envs": B, "agents": N, "episode_length": EPISODE, "episodes_timed": episodes, "fused_policy": col.fused,
            "ms_per_episode": loop_ms, "agent_steps_per_s": B * N * EPISODE / (loop_ms * 1e-3),
            "sim_ms_per_episode": sim_ms, "sim_share": sim_ms / loop_ms, "episodes_in_stats": float(stats[15 * N])}


def part_c(main_tree: str, repeats: int, steps: int, warmup: int):
    trees = {"main": os.path.abspath(main_tree), "branch": ROOT}
    res = {"main": [], "branch": []}
    raw = []
    for r in range(repeats):
        for name in (("main", "branch") if r % 2 == 0 else ("branch", "main")):
            cmd = [sys.executable, os.path.join(trees[name], "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup),
                   "--config", "form"]
            p = subprocess.run(cmd, capture_output=True, text=True, cwd=trees[name])
            line = [l for l in p.stdout.splitlines() if l.startswith("{")]
            if p.returncode != 0 or not line:
                raise RuntimeError(f"{name}: {p.stdout[-2000:]}{p.stderr[-2000:]}")
            d = json.loads(line[-1])
            res[name].append(d["ms_per_step"] * 1e3)
            raw.append({"tree": name, "value": d["value"], "ms_per_step": d["ms_per_step"], "closed_loop_ms": d["closed_loop"]["ms_per_step"]})
    out = {k: spread(v) for k, v in res.items()}
    out["unit"] = "us per step (bench.py ms_per_step x 1000)"
    out["branch_minus_main_us"] = out["branch"]["median"] - out["main"]["median"]
    out["runs"] = raw
    out["command"] = f"bench.py --gpus 1 --steps {steps} --warmup {warmup} --config form"
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True)
    ap.add_argument("--main-tree", default=None, help="(c): another checkout to compare bench.py --config form against")
    ap.add_argument("--repeats", type=int, default=6)
    ap.add_argument("--steps", type=int, default=500, help="(a): steps per timed run")
    ap.add_argument("--episodes", type=int, default=20, help="(b): episodes timed per size")
    ap.add_argument("--bench-repeats", type=int, default=3)
    ap.add_argument("--profile", action="store_true", help="only the per-kernel breakdown of (a), torch.profiler, separate JSON")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_formation_rollout.py: no CUDA device")
    os.makedirs(args.out, exist_ok=True)
    if args.profile:
        print(json.dumps({"gpu": gpu_info(), **part_a_profile(args.out)}, indent=1))
        return
    t0 = time.time()
    result = {"gpu": gpu_info()}

    def save():                                                  # after every part: a later failure keeps what was measured
        with open(os.path.join(args.out, "bench_formation_rollout.json"), "w") as f:
            f.write(json.dumps(result, indent=1))

    result["a_step_many_stats"] = part_a(args.repeats, args.steps)
    save()
    result["b_collector"] = [part_b(B, args.episodes) for B in (4096, 65536)]
    save()
    if args.main_tree:
        result["c_bench_form"] = part_c(args.main_tree, args.bench_repeats, 200, 20)
    result["gpu_after"] = gpu_info()
    result["wall_s"] = time.time() - t0
    save()
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
