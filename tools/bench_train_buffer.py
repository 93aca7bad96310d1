#!/usr/bin/env python
"""Times the training side of DeviceRolloutBuffer (csrc/fm_buffer.cu) against its torch equivalent, CUDA events, inputs
larger than L2, on one GPU; prints JSON lines (the card's name and power limit first, read in the same run):

* returns + advantages: fm_buffer_returns + fm_buffer_advantages vs the torch loop compute_returns ran before plus the
  torch nanmean / nan-std normalisation;
* one epoch of recurrent_generator (L = 10) at num_mini_batch 1 and 4: fm_buffer_minibatch vs torch advanced indexing
  of the same buffer (share_obs and adj indexed through the env's rows, as the kernel reads them).

Shapes: navigation 65 536 envs x 3 agents (E = 9) and 4 096 x 16 (E = 35), T = 25.  Bytes are counted from shapes:
what one epoch writes (every field of every mini-batch) and reads (the same rows of the sources plus the permutation).
usage: python tools/bench_train_buffer.py [--reps 10]"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
HBM_PEAK = 7.7e12                       # B/s, NVIDIA HGX B200 data sheet, one GPU


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / reps


def make_buffer(T, B, N, E):
    from fair_marl_b200.rollout import DeviceRolloutBuffer
    b = DeviceRolloutBuffer(T, B, N, E, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(0)
    for name in ("obs", "node_obs", "adj_env", "rnn_states", "rnn_states_critic", "action_log_probs", "value_preds", "rewards"):
        x = getattr(b, name)
        x.copy_(torch.randn(x.shape, device="cuda", generator=g))
    b.masks.copy_((torch.rand(b.masks.shape, device="cuda", generator=g) > 0.05).float())
    b.active_masks.copy_((torch.rand(b.masks.shape, device="cuda", generator=g) > 0.1).float())
    return b


def torch_returns_advantages(b, nv):
    """The loop compute_returns ran on a CUDA buffer before the kernel, then GR_MAPPO.train's normalisation in torch."""
    T = b.episode_length
    b.value_preds[-1] = nv.view_as(b.value_preds[-1])
    gae = torch.zeros_like(b.value_preds[0])
    for t in reversed(range(T)):
        delta = b.rewards[t] + b.gamma * b.value_preds[t + 1] * b.masks[t + 1] - b.value_preds[t]
        gae = delta + b.gamma * b.gae_lambda * b.masks[t + 1] * gae
        b.returns[t] = gae + b.value_preds[t]
    adv = b.returns[:-1] - b.value_preds[:-1]
    x = torch.where(b.active_masks[:-1] == 0, torch.nan, adv)
    mean = torch.nanmean(x)
    std = torch.sqrt(torch.nanmean((x - mean) ** 2))
    return (adv - mean) / (std + 1e-5)


def torch_recurrent_epoch(b, adv, perm, K, L):
    """recurrent_generator by advanced indexing: the same 15 device tensors per mini-batch."""
    T, B, N = b.episode_length, b.n_rollout_threads, b.num_agents
    per = T * B * N // L // K
    out = []
    for k in range(K):
        f = (perm[k * per:(k + 1) * per][None, :] * L + torch.arange(L, device="cuda")[:, None]).reshape(-1)
        t, n, e = f % T, (f // T) % N, f // (T * N)
        f0 = perm[k * per:(k + 1) * per] * L
        t0, n0, e0 = f0 % T, (f0 // T) % N, f0 // (T * N)
        R = f.numel()
        out.append((b.obs[t, e].reshape(R, -1), b.obs[t, e, n], b.node_obs[t, e, n], b.adj_env[t, e], n.int().view(R, 1),
                    torch.arange(N, device="cuda", dtype=torch.int32).expand(R, N).contiguous(),
                    b.rnn_states[t0, e0, n0], b.rnn_states_critic[t0, e0, n0], b.actions[t, e, n], b.value_preds[t, e, n],
                    b.returns[t, e, n], b.masks[t, e, n], b.active_masks[t, e, n], b.action_log_probs[t, e, n], adv[t, e, n]))
    return out


def epoch_bytes(b, K, L):
    T, B, N, E = b.episode_length, b.n_rollout_threads, b.num_agents, b.num_entities
    D, F, H = b.obs.shape[-1], b.node_obs.shape[-1], b.rnn_states.shape[-1] * b.rnn_states.shape[-2]
    per = T * B * N // L // K
    R = per * L
    row = 4 * (N * D + D + E * F + E * E + 1 + N + 7)
    written = K * (R * row + 2 * per * 4 * H)
    read = written - K * R * 4 * (1 + N) + K * per * 8        # ids are synthesised; the permutation is read
    return written, read


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_train_buffer needs a CUDA device"
    print(json.dumps({"card": card()}), flush=True)
    for B, N, O in ((65536, 3, 3), (4096, 16, 3)):
        T, E = 25, 2 * N + O
        b = make_buffer(T, B, N, E)
        nv = torch.randn(B * N, 1, device="cuda")
        v0 = b.value_preds.clone()

        def kern():
            b.compute_returns(nv)
            return b.advantages()

        def ref():
            return torch_returns_advantages(b, nv)
        ms_k, ms_t = timed(kern, args.reps), timed(ref, args.reps)
        b.value_preds.copy_(v0)
        adv_t = ref()
        ret_t = b.returns.clone()
        b.value_preds.copy_(v0)
        adv_k = kern()
        cols = B * N
        ra_bytes = 4 * cols * (T * 5 + 2 * T + T)       # returns scan ~ (v, r, m in; ret out) + advantages (3 in, 1 out, 1 rw)
        print(json.dumps({"what": "returns + advantages", "T": T, "B": B, "N": N, "kernel_ms": round(ms_k, 4), "torch_ms": round(ms_t, 4),
                          "speedup": round(ms_t / ms_k, 2), "approx_bytes": ra_bytes,
                          "kernel_GBps": round(ra_bytes / ms_k / 1e6, 1),
                          "returns_bitwise_equal": bool(torch.equal(b.returns, ret_t)),
                          "advantages_max_abs_diff_vs_torch_stats": float((adv_k - adv_t).abs().max())}), flush=True)
        adv = b.advantages()
        L = 10
        for K in (1, 4):
            units = T * B * N // L
            perm = torch.randperm(units, device="cuda", generator=torch.Generator(device="cuda").manual_seed(K))

            def kern_epoch():
                return list(b.recurrent_generator(adv, K, L, generator=torch.Generator(device="cuda").manual_seed(K)))

            def torch_epoch():
                return torch_recurrent_epoch(b, adv, perm, K, L)
            ms_k, ms_t = timed(kern_epoch, args.reps), timed(torch_epoch, args.reps)
            got, want = kern_epoch(), torch_epoch()
            equal = all(torch.equal(x.reshape(y.shape), y) for g, w in zip(got, want) for x, y in zip(g[:15], w))
            del got, want
            wr, rd = epoch_bytes(b, K, L)
            print(json.dumps({"what": "recurrent_generator epoch", "T": T, "B": B, "N": N, "E": E, "L": L, "num_mini_batch": K,
                              "kernel_ms": round(ms_k, 3), "torch_ms": round(ms_t, 3), "speedup": round(ms_t / ms_k, 2),
                              "bytes_written": wr, "bytes_read": rd, "kernel_GBps": round((wr + rd) / ms_k / 1e6, 1),
                              "frac_of_7.7TBps": round((wr + rd) / (ms_k * 1e-3) / HBM_PEAK, 3),
                              "outputs_bitwise_equal": bool(equal)}), flush=True)
            torch.cuda.empty_cache()
        del b
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
