#!/usr/bin/env python
"""The fused graph-network forward at the shapes of both kernel mappings (csrc/fm_policy.cu): gnn_kernel (mapping 1, warp
per graph) and gnn_wide_kernel (mapping 2, CTA per graph), against the dense torch modules, and the device rollout loop
(RolloutCollector) at shapes only the CTA-per-graph kernel serves.
usage: python tools/bench_gnn_wide.py [--quick]   (on the GPU box) -> one JSON line per measurement, the card first.

Kernel times are CUDA events around back-to-back fm_gnn_forward launches whose inputs (node rows + adjacency) are larger
than the 126 MB L2.  FMA counts per graph are computed from the shapes and the graph's edges (`fma_per_graph`)."""
import argparse, json, os, subprocess, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import fair_marl_b200 as fm  # noqa: E402
from fair_marl_b200.policy import DenseGNNBase, edge_mask  # noqa: E402

L2_BYTES = 126 << 20


def emit(**kw):
    print(json.dumps(kw), flush=True)


def fma_per_graph(E, KF, edges, embed_layers, conv_layers):
    """Multiply-adds of the forward as the kernels compute it: lin1's node part per node, the edge MLP per edge, the 16 -> 160
    projection per node and conv, and per edge, head and conv the q.k dot product, the edge term and the weighted value."""
    H, heads = 16, 3
    a0 = E * KF * H
    a = edges * (H + embed_layers * H * H)
    b1 = conv_layers * E * H * 160
    b2 = conv_layers * (E * heads * H + edges * heads * (H + 1 + H + 1) + E * heads * H)
    return a0 + a + b1 + b2


def events_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def kernel_bench(quick):
    dev = torch.device("cuda", 0)
    shapes = [(9, (1, 2)), (17, (1, 2))] + [(E, (2,)) for E in (16, 22, 24, 35, 45, 64)]
    for E, mappings in shapes:
        torch.manual_seed(E)
        gnn = DenseGNNBase(fm.PolicyConfig(), "node").eval().to(dev)      # default: 1 hidden embed layer, 3 convs, ReLU, LN
        NF, rep = 11, max(1, (E - 3) // 2)                                 # navigation: N ego graphs share an adjacency
        per_graph = E * NF * 4 + E * E * 4 / rep
        M = max(1 << 16, int(3 * L2_BYTES / per_graph) // rep * rep)
        if quick:
            M = 4096 // rep * rep
        g = torch.Generator(device=dev).manual_seed(E)
        pos = torch.rand(M // rep, E, 2, generator=g, device=dev) * 2 - 1
        adj = torch.cdist(pos, pos).float().contiguous()
        node = torch.randn(M, E, NF, generator=g, device=dev)
        node[..., -1] = torch.randint(0, 4, (M, E), generator=g, device=dev).float()
        aid = torch.randint(0, E, (M, 1), generator=g, device=dev)
        edges = float(edge_mask(adj, 1.0).sum()) / (M // rep)
        fma = fma_per_graph(E, NF - 1, edges, 1, 3)
        res = {m: [] for m in mappings}
        with torch.no_grad():
            outs = {m: gnn.forward_fused(node, adj, rep, aid, mapping=m) for m in mappings}   # warm-up
            torch.cuda.synchronize()
            for _ in range(1 if quick else 5):                             # alternated
                for m in mappings:
                    res[m].append(events_ms(lambda: gnn.forward_fused(node, adj, rep, aid, mapping=m), 3 if quick else 10))
            # the dense torch forward on the same graphs, in chunks the size RolloutCollector uses (max_graphs = 2^17)
            chunk = min(M, max(rep, (min(1 << 17, int(4e9 / (E * E * 64))) // rep) * rep))
            adj_rep = lambda lo, hi: adj[lo // rep:hi // rep].repeat_interleave(rep, 0)
            dense = lambda: [gnn(node[lo:lo + chunk], adj_rep(lo, lo + chunk), aid[lo:lo + chunk]) for lo in range(0, M, chunk)]
            ref = torch.cat(dense())
            dense_ms = events_ms(dense, 1 if quick else 2)
        for m in mappings:
            ms = sorted(res[m])[len(res[m]) // 2]
            emit(what="kernel", E=E, mapping=m, graphs=M, graphs_per_adj=rep, input_mb=round(M * per_graph / 2**20, 1),
                 edges_per_graph=round(edges, 1), fma_per_graph=int(fma), ms_median=round(ms, 4),
                 ms_all=[round(x, 4) for x in res[m]], graphs_per_s=M / (ms * 1e-3), fma_per_s=M * fma / (ms * 1e-3),
                 max_abs_diff_vs_dense=float((outs[m] - ref).abs().max()))
        emit(what="dense_torch", E=E, graphs=M, chunk=chunk, ms=round(dense_ms, 3), graphs_per_s=M / (dense_ms * 1e-3),
             speedup_of_fused=dense_ms / min(sorted(res[m])[len(res[m]) // 2] for m in mappings))
        del node, adj, aid, outs, ref
        torch.cuda.empty_cache()


def collector_bench(quick):
    from oracle.navgraph import NavConfig
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from parity_util import sim_config_from
    runs = [("C4 navigation N=16 O=3", "nav", 4096, True), ("C4 navigation N=16 O=3", "nav", 4096, False),
            ("C4 navigation N=16 O=3", "nav", 65536, True),
            ("formation N=7 O=8", "form", 65536, True), ("formation N=7 O=8", "form", 65536, False)]
    for name, fam, B, fused in runs:
        if quick:
            B = 64
        if fam == "nav":
            env = fm.B200GraphVecEnv(sim_config_from(NavConfig(num_agents=16, num_obstacles=3)), num_envs=B, seed=1)
            pc = fm.PolicyConfig(num_agents=16)
        else:
            env = fm.B200FormationVecEnv(fm.FormationSimConfig(num_agents=7, num_obstacles=8), num_envs=B, seed=1)
            pc = fm.PolicyConfig(num_agents=7, obs_dim=11, node_feat_dim=13)
        torch.manual_seed(0)
        actor, critic = fm.DenseGraphActor(pc).to(env.device).eval(), fm.DenseGraphCritic(pc).to(env.device).eval()
        row = dict(what="collector", config=name, envs=B, agents=env.num_agents, entities=env.num_entities, fused=fused)
        try:
            col = fm.RolloutCollector(env, actor, critic, deterministic=False, fused=fused,
                                      generator=torch.Generator(device=env.device).manual_seed(3))
            T = col.buffer.episode_length
            col.warmup(); col.run(); col.buffer.after_update()
            col.capture()
            col.run(); col.buffer.after_update()                           # warm replay
            torch.cuda.synchronize()
            ms = events_ms(lambda: (col.run(), col.buffer.after_update()), 1 if quick else 3)
            row.update(episode_length=T, ms_per_episode=round(ms, 3), agent_steps_per_s=B * env.num_agents * T / (ms * 1e-3),
                       captured=True)
        except torch.cuda.OutOfMemoryError as e:
            row.update(not_measured=f"out of memory: {str(e).splitlines()[0][:120]}")
        emit(**row)
        env.close()
        del env, actor, critic
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true", help="tiny sizes: checks that the script runs, measures nothing useful")
    ap.add_argument("--skip-collector", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_gnn_wide.py measures on the GPU; no CUDA device is visible")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    emit(what="card", torch_name=torch.cuda.get_device_name(0), nvidia_smi=q[0] if q else "not available")
    kernel_bench(args.quick)
    if not args.skip_collector:
        collector_bench(args.quick)


if __name__ == "__main__":
    main()
