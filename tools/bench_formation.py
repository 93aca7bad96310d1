"""Formation kernel timing (diagnostic; the formation family is not a BASELINE config): agent-steps/s of
fm_formation_step over B envs with CUDA events, and its algorithmic-bytes fraction of the HBM roofline.
usage: python tools/bench_formation.py [--envs 65536] [--agents 3] [--obstacles 3] [--steps 300] [--assignment fair]
--assignment optimal | random: the base scenarios OA / RA (no fairness term); the default is FA+FR."""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import fair_marl_b200 as fm  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--agents", type=int, default=3)
    ap.add_argument("--obstacles", type=int, default=3)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=30)
    ap.add_argument("--assignment", choices=("fair", "optimal", "random"), default="fair")
    a = ap.parse_args()
    B, N, O = a.envs, a.agents, a.obstacles
    E = 2 * N + O
    kw = {} if a.assignment == "fair" else dict(assignment=a.assignment, fairness_reward=False)
    cfg = fm.FormationSimConfig(num_agents=N, num_obstacles=O, goal_rew=30.0, collision_rew=30.0, **kw)
    env = fm.B200FormationVecEnv(cfg, num_envs=B, seed=0)
    env.reset_tensor()
    g = torch.Generator(device="cuda").manual_seed(1234)
    acts = torch.randint(0, 5, (25, B, N), generator=g, device="cuda", dtype=torch.int32)
    for t in range(a.warmup):
        env.step_tensor(acts[t % 25])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for t in range(a.steps):
        env.step_tensor(acts[t % 25])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / a.steps
    # algorithmic bytes per env-step: actions + state read, dynamic state written, every output written once
    state_rd = 4 * (N + 16 * N + 2 * O + 4) + N              # fp32 / int32 words, + status bytes
    state_wr = 4 * (16 * N - 2 * N + 4) + N                   # landmarks stay (except on resets)
    outs = 4 * (11 * N + 13 * N * E + E * E + N + 14 * N) + N
    alg = (state_rd + state_wr + outs) * B
    peak = 6551.7
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(pk):
        peak = float(json.load(open(pk))["hbm_gbs"])
    ach = alg / (ms * 1e-3) / 1e9
    scenario = {"fair": "fairrew", "optimal": "optimal assignment", "random": "random assignment"}[a.assignment]
    print(json.dumps({"metric": "agent-steps/sec, formation step+obs+reward+per-step assignment", "value": B * N / (ms * 1e-3),
                      "unit": "agent-steps/s", "ms_per_step": ms, "steps": a.steps, "warmup": a.warmup,
                      "config": {"workload": f"formation ({scenario}) {N} agents / {N} goals / {O} obstacles, {B} envs, random actions, "
                                             "episode_length 25 with auto-reset", "l2": f"outputs {outs * B / 1e6:.0f} MB per step"},
                      "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                                   "kernel": f"fm::formation_step_kernel<{N}> (thread per env, float64)",
                                   "algorithmic_bytes_per_step": alg}, "dtype": "f64", "data": "synthetic"}))


if __name__ == "__main__":
    main()
