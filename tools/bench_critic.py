#!/usr/bin/env python
"""The centralised-observation and per-agent critics in the device rollout loop: the collector's step with each critic
configuration, fused (graph network + head kernels) and fused=False (the dense torch modules), and the wide critic head
kernel (critic_head_kernel behind fm_critic_head) alone.
usage: python tools/bench_critic.py [--quick]   (needs a CUDA device) -> one JSON line per measurement, the card first.

Step times are CUDA events around `steps` collector steps after a warm-up episode (no CUDA graph).  Head kernel times are
CUDA events around back-to-back launches whose inputs (cent_obs, nbd, rnn states) are larger than the 126 MB L2."""
import argparse, json, os, subprocess, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import fair_marl_b200 as fm  # noqa: E402

L2_BYTES = 126 << 20
CONFIGS = {"default": {}, "cent_global": dict(use_cent_obs=True), "node": dict(critic_graph_aggr="node"),
           "cent_node": dict(use_cent_obs=True, critic_graph_aggr="node")}


def emit(**kw):
    print(json.dumps(kw), flush=True)


def events_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def collector_bench(N, O, B, steps):
    from oracle.navgraph import NavConfig
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from parity_util import sim_config_from
    for name, kw in CONFIGS.items():
        for fused in (None, False):
            env = fm.B200GraphVecEnv(sim_config_from(NavConfig(num_agents=N, num_obstacles=O, episode_length=steps)),
                                     num_envs=B, seed=1)
            torch.manual_seed(0)
            actor = fm.DenseGraphActor(fm.PolicyConfig(num_agents=N)).cuda().eval()
            critic = fm.DenseGraphCritic(fm.PolicyConfig(num_agents=N, **kw)).cuda().eval()
            col = fm.RolloutCollector(env, actor, critic, fused=fused, generator=torch.Generator(device="cuda").manual_seed(2))
            col.warmup(); col.run(); col.buffer.after_update(); torch.cuda.synchronize()
            ms = events_ms(lambda: col.run(steps), 1) / steps
            emit(kind="collector_step", N=N, O=O, E=env.num_entities, num_envs=B, critic=name, fused=col.fused,
                 head_in=critic._head_in, ms_per_step=round(ms, 4), agent_steps_per_s=round(B * N / ms * 1e3))
            env.close()
            del col, env, actor, critic
            torch.cuda.empty_cache()


def head_bench(quick):
    for family, N, name in [("navigation", 3, "cent_global"), ("navigation", 16, "cent_node"), ("navigation", 32, "cent_node"),
                            ("navigation", 32, "node"), ("formation", 7, "cent_node")]:
        obs_dim = 7 if family == "navigation" else 11
        cfg = fm.PolicyConfig(num_agents=N, obs_dim=obs_dim, **CONFIGS[name])
        torch.manual_seed(0)
        net = fm.DenseGraphCritic(cfg).cuda().eval()
        nbd_dim = 16 * (N if cfg.critic_graph_aggr == "node" else 1)
        per_row = 4 * (nbd_dim + 64 + 64 + 1 + 1 + (obs_dim if cfg.use_cent_obs else 0))
        M = (int(3 * L2_BYTES / per_row) // N) * N if not quick else 4096 // N * N
        g = torch.Generator(device="cuda").manual_seed(1)
        cent = torch.randn(M // N, N * obs_dim, generator=g, device="cuda") if cfg.use_cent_obs else None
        nbd = torch.randn(M, nbd_dim, generator=g, device="cuda")
        rnn = torch.randn(M, 1, 64, generator=g, device="cuda")
        masks = torch.ones(M, 1, device="cuda")
        c = None if cent is None else (cent, N)
        with torch.no_grad():
            net._run_critic_head(c, nbd, rnn, masks)
            ms = events_ms(lambda: net._run_critic_head(c, nbd, rnn, masks), 20)
            x = nbd if cent is None else torch.cat([cent.repeat_interleave(N, 0), nbd], dim=1)

            def dense():
                h, _ = net.rnn(net.base(x), rnn, masks)
                return net.v_out(h)
            dense()
            ms_dense = events_ms(dense, 20)
        D = net._head_in
        flop = 2 * M * (D * 64 + cfg.layer_N * 64 * 64 + 2 * 64 * 192 + 64)
        emit(kind="critic_head_kernel", family=family, N=N, critic=name, head_in=D, rows=M, ms=round(ms, 4),
             gflops=round(flop / ms / 1e6, 1), dense_torch_ms_same_inputs=round(ms_dense, 4))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true")
    a = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    emit(kind="card", nvidia_smi=q, torch_device=torch.cuda.get_device_name(0))
    head_bench(a.quick)
    collector_bench(3, 3, 1024 if a.quick else 65536, 4 if a.quick else 16)
    collector_bench(16, 3, 256 if a.quick else 4096, 4 if a.quick else 16)


if __name__ == "__main__":
    main()
