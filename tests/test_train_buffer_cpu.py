"""CPU-side checks of the trainer's input on the device rollout buffer:

* DeviceRolloutBuffer.compute_returns on a CPU buffer (the torch loop) against oracle/graph_buffer.py, bit for bit, in all
  8 (GAE x proper time limits x value normaliser) combinations, with zeros in masks and bad masks and a normaliser whose
  mean is not 0 and whose std is not 1;
* the ctypes mirrors of FmReturnsConfig, FmMinibatchConfig, FmBufferSlabs and FmMinibatch against the header;
* every refusal of fm_buffer_returns / fm_buffer_advantages / fm_buffer_minibatch comes before any device is touched, and
  the Python generators refuse a CPU buffer and the same arguments.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import graph_buffer as ogb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import fair_marl_b200
    fair_marl_b200.build_library()
    from fair_marl_b200 import _lib
    return _lib.load()


class TorchNorm:
    """The reference's ValueNorm interface (running_mean_var -> float32 tensors on its device) over the oracle's numpy
    state, taken once: a capture may call running_mean_var without a host copy."""

    def __init__(self, vn, device="cpu"):
        self.mean, self.var = (torch.from_numpy(np.array(a, np.float32).reshape(1)).to(device) for a in vn.running_mean_var())

    def running_mean_var(self):
        return self.mean, self.var


def trained_value_norm(seed=0):
    """An oracle ValueNorm after a few updates: mean far from 0, std far from 1."""
    vn = ogb.ValueNorm()
    rng = np.random.default_rng(seed)
    for _ in range(3):
        vn.update((7.5 + 3.0 * rng.standard_normal((64, 1))).astype(np.float32))
    mean, var = vn.running_mean_var()
    assert abs(float(mean[0])) > 1 and abs(float(np.sqrt(var[0])) - 1) > 0.5
    return vn


def random_buffer(T, B, N, rng, device="cpu", **kw):
    """A DeviceRolloutBuffer with random returns-relevant slabs (masks / bad masks / active masks with zeros in them)."""
    from fair_marl_b200.rollout import DeviceRolloutBuffer
    b = DeviceRolloutBuffer(T, B, N, 2 * N + 3, device=device, **kw)
    f = lambda *s: torch.as_tensor(rng.standard_normal(s).astype(np.float32))
    z = lambda *s, p=0.2: torch.as_tensor((rng.random(s) > p).astype(np.float32))
    b.value_preds.copy_(f(T + 1, B, N, 1))
    b.rewards.copy_(f(T, B, N, 1))
    b.masks.copy_(z(T + 1, B, N, 1))
    b.bad_masks.copy_(z(T + 1, B, N, 1, p=0.3))
    b.active_masks.copy_(z(T + 1, B, N, 1, p=0.25))
    return b


def oracle_slabs(b):
    return {k: getattr(b, k).detach().cpu().numpy().copy() for k in ("value_preds", "rewards", "masks", "bad_masks", "returns")}


COMBOS = [(gae, proper, norm) for gae in (True, False) for proper in (False, True) for norm in (False, True)]


@pytest.mark.parametrize("gae,proper,norm", COMBOS)
def test_cpu_compute_returns_matches_the_oracle_bit_for_bit(gae, proper, norm):
    T, B, N = 25, 64, 3
    rng = np.random.default_rng(11)
    b = random_buffer(T, B, N, rng, use_gae=gae, use_proper_time_limits=proper)
    nv = torch.as_tensor(rng.standard_normal((B * N, 1)).astype(np.float32))
    vn = trained_value_norm() if norm else None
    ref = oracle_slabs(b)
    ogb.compute_returns(ref, nv.numpy().reshape(B, N, 1), vn, use_gae=gae, use_proper_time_limits=proper)
    b.compute_returns(nv, TorchNorm(vn) if norm else None)
    assert np.array_equal(b.returns.numpy(), ref["returns"])
    assert np.array_equal(b.value_preds.numpy(), ref["value_preds"])
    if norm and (gae or proper):                      # the normaliser matters in these branches and only these
        plain = oracle_slabs(random_buffer(T, B, N, np.random.default_rng(11)))
        ogb.compute_returns(plain, nv.numpy().reshape(B, N, 1), None, use_gae=gae, use_proper_time_limits=proper)
        assert not np.array_equal(plain["returns"], ref["returns"])


def test_cpu_compute_returns_without_options_is_the_previous_loop():
    """The default configuration computes what the loop computed before the options were added."""
    T, B, N = 9, 7, 2
    rng = np.random.default_rng(2)
    b = random_buffer(T, B, N, rng)
    nv = torch.as_tensor(rng.standard_normal((B * N, 1)).astype(np.float32))
    v, r, m = b.value_preds.clone(), b.rewards.clone(), b.masks.clone()
    v[-1] = nv.view(B, N, 1)
    ret = torch.zeros_like(v)
    gae = torch.zeros_like(v[0])
    for t in reversed(range(T)):
        delta = r[t] + b.gamma * v[t + 1] * m[t + 1] - v[t]
        gae = delta + b.gamma * b.gae_lambda * m[t + 1] * gae
        ret[t] = gae + v[t]
    b.compute_returns(nv)
    assert torch.equal(b.returns[:T], ret[:T])


def test_oracle_value_norm_denormalize_is_x_std_plus_mean():
    vn = trained_value_norm(3)
    mean, var = vn.running_mean_var()
    x = np.linspace(-3, 3, 13, dtype=np.float32)
    assert np.array_equal(vn.denormalize(x), x * np.sqrt(var) + mean)
    assert var[0] >= np.float32(1e-2)


def test_oracle_generators_cover_the_epoch():
    """The restated generators drop exactly the remainder the reference drops."""
    T, B, N, E = 5, 3, 2, 7
    rng = np.random.default_rng(0)
    ids = np.arange(T * B * N, dtype=np.float32).reshape(T, B, N, 1)
    buf = {"share_obs": np.zeros((T + 1, B, N, 2 * N)), "obs": np.zeros((T + 1, B, N, 2)), "node_obs": np.zeros((T + 1, B, N, E, 3)),
           "adj": np.zeros((T + 1, B, N, E, E)), "agent_id": np.zeros((T + 1, B, N, 1)), "share_agent_id": np.zeros((T + 1, B, N, N)),
           "rnn_states": np.zeros((T + 1, B, N, 1, 4)), "rnn_states_critic": np.zeros((T + 1, B, N, 1, 4)),
           "actions": ids, "value_preds": np.zeros((T + 1, B, N, 1)), "returns": np.zeros((T + 1, B, N, 1)),
           "masks": np.zeros((T + 1, B, N, 1)), "active_masks": np.zeros((T + 1, B, N, 1)), "action_log_probs": ids,
           "available_actions": np.ones((T + 1, B, N, 5)), "rewards": np.zeros((T, B, N, 1))}
    adv = ids
    k = ogb.SAMPLE_FIELDS.index("actions")
    perm = rng.permutation(T * B * N)
    got = np.concatenate([mb[k][:, 0] for mb in ogb.feed_forward_batches(buf, adv, perm, 4)])
    assert sorted(got) == sorted(perm[:4 * (T * B * N // 4)])
    L = 4
    chunks = T * B * N // L
    perm = rng.permutation(chunks)
    got = np.concatenate([mb[k][:, 0] for mb in ogb.recurrent_batches(buf, adv, perm, 3, L)])
    flat = ogb._cast(ids)[:, 0]
    want = [flat[c * L + l] for c in perm[:3 * (chunks // 3)] for l in range(L)]
    assert sorted(got) == sorted(want)
    perm = rng.permutation(B * N)
    got = np.concatenate([mb[k][:, 0] for mb in ogb.naive_recurrent_batches(buf, adv, perm, 3)])
    assert sorted(got) == sorted(ids.ravel())
    # B N = 6 not divisible by 4: the reference yields 6 mini-batches of one column, not 4 (with 7 columns and 2 it
    # raises IndexError part-way through the epoch); the device generator refuses both
    assert len(list(ogb.naive_recurrent_batches(buf, adv, perm, 4))) == 6


def test_struct_layouts_match_header(tmp_path):
    from fair_marl_b200 import _lib
    structs = {"FmReturnsConfig": (_lib.FmReturnsConfig, 32), "FmMinibatchConfig": (_lib.FmMinibatchConfig, 48),
               "FmBufferSlabs": (_lib.FmBufferSlabs, 12 * 8), "FmMinibatch": (_lib.FmMinibatch, 15 * 8)}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "fairmarl.h"', 'int main(void) {',
             '  printf("FM_ADV_WORKSPACE_DOUBLES %d\\n", FM_ADV_WORKSPACE_DOUBLES);',
             '  printf("FM_MINIBATCH_FEED_FORWARD %d\\n", FM_MINIBATCH_FEED_FORWARD);',
             '  printf("FM_MINIBATCH_RECURRENT %d\\n", FM_MINIBATCH_RECURRENT);',
             '  printf("FM_MINIBATCH_NAIVE_RECURRENT %d\\n", FM_MINIBATCH_NAIVE_RECURRENT);']
    for name, (cls, _) in structs.items():
        lines.append(f'  printf("{name} %zu\\n", sizeof({name}));')
        lines += [f'  printf("{name}.{f} %zu\\n", offsetof({name}, {f}));' for f, _ in cls._fields_]
    lines += ['  return 0;', '}']
    src, exe = tmp_path / "layout.c", tmp_path / "layout"
    src.write_text("\n".join(lines))
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    for name, (cls, size) in structs.items():
        assert int(got[name]) == ctypes.sizeof(cls) == size, name
        for f, _ in cls._fields_:
            assert int(got[f"{name}.{f}"]) == getattr(cls, f).offset, f"{name}.{f}"
    assert int(got["FM_ADV_WORKSPACE_DOUBLES"]) == _lib.ADV_WORKSPACE_DOUBLES
    for mode, v in _lib.MINIBATCH_MODES.items():
        assert int(got["FM_MINIBATCH_" + mode.upper()]) == v


_REFUSALS = """
import ctypes
from fair_marl_b200 import _lib
lib = _lib.load()
fake = ctypes.c_void_p(256)                  # never dereferenced: every refused call below is refused first
def ret(T=25, B=4, N=3, proper=0, nv=fake, bad=fake, mean=None, std=None, cfg=True):
    c = _lib.FmReturnsConfig(episode_length=T, num_envs=B, num_agents=N, use_gae=1, use_proper_time_limits=proper,
                             gamma=0.99, gamma_lambda=0.99 * 0.95)
    rc = lib.fm_buffer_returns(0, ctypes.byref(c) if cfg else None, nv, fake, fake, fake, bad, mean, std, fake, None)
    return rc, lib.fm_last_error().decode()
rc, msg = ret(cfg=False); assert rc == -1 and "null" in msg, (rc, msg)
rc, msg = ret(nv=None); assert rc == -1 and "null" in msg, (rc, msg)
rc, msg = ret(proper=1, bad=None); assert rc == -1 and "null" in msg, (rc, msg)
rc, msg = ret(mean=fake); assert rc == -1 and "both" in msg, (rc, msg)
rc, msg = ret(T=0); assert rc == -1 and "episode_length 0" in msg, (rc, msg)
rc, msg = ret(B=1 << 20, N=32, T=64); assert rc == -1 and "2^31" in msg, (rc, msg)
rc, msg = ret(B=(1 << 31) // 75 + 1, N=3, T=25); assert rc == -1 and "2^31" in msg, (rc, msg)
rc, msg = ret(proper=0, bad=None); assert rc == -2, (rc, msg)                      # accepted: fails at the device
rc, msg = ret(B=(1 << 31) // 75, N=3, T=25, mean=fake, std=fake); assert rc == -2, (rc, msg)
def adv(T=25, B=4, N=3, ws=fake, mean=None, std=None):
    rc = lib.fm_buffer_advantages(0, T, B, N, fake, fake, fake, mean, std, fake, fake, ws, None)
    return rc, lib.fm_last_error().decode()
rc, msg = adv(ws=None); assert rc == -1 and "null" in msg, (rc, msg)
rc, msg = adv(std=fake); assert rc == -1 and "both" in msg, (rc, msg)
rc, msg = adv(N=0); assert rc == -1, (rc, msg)
rc, msg = adv(T=1 << 16, B=1 << 16); assert rc == -1 and "2^31" in msg, (rc, msg)
rc, msg = adv(); assert rc == -2, (rc, msg)
slabs = _lib.FmBufferSlabs(**{k: 256 for k in _lib.BUFFER_SLAB_FIELDS})
outs = _lib.FmMinibatch(**{k: 256 for k in _lib.MINIBATCH_FIELDS})
def mb(mode=1, K=4, mbs=0, L=10, k=0, T=25, B=8, N=3, perm=fake, slab=None, out=None, E=9):
    c = _lib.FmMinibatchConfig(episode_length=T, num_envs=B, num_agents=N, num_entities=E, obs_dim=7, node_feat_dim=11,
                               rnn_floats=64, mode=mode, num_mini_batch=K, mini_batch_size=mbs, data_chunk_length=L, mini_batch=k)
    rc = lib.fm_buffer_minibatch(0, ctypes.byref(c), ctypes.byref(slab or slabs), perm, ctypes.byref(out or outs), None)
    return rc, lib.fm_last_error().decode()
rc, msg = mb(perm=None); assert rc == -1 and "null" in msg, (rc, msg)
for f in _lib.BUFFER_SLAB_FIELDS:
    s = _lib.FmBufferSlabs(**{k: 256 for k in _lib.BUFFER_SLAB_FIELDS}); setattr(s, f, None)
    rc, msg = mb(slab=s); assert rc == -1 and "null" in msg, (f, rc, msg)
for f in _lib.MINIBATCH_FIELDS:
    o = _lib.FmMinibatch(**{k: 256 for k in _lib.MINIBATCH_FIELDS}); setattr(o, f, None)
    rc, msg = mb(out=o); assert rc == -1 and "null" in msg, (f, rc, msg)
rc, msg = mb(mode=3); assert rc == -1 and "mode 3" in msg, (rc, msg)
rc, msg = mb(L=0); assert rc == -1 and "data_chunk_length 0" in msg, (rc, msg)
rc, msg = mb(K=61); assert rc == -1 and "61 for 60 chunks" in msg, (rc, msg)     # 600 samples / L 10 = 60 chunks
rc, msg = mb(K=0); assert rc == -1, (rc, msg)
rc, msg = mb(mode=0, K=601); assert rc == -1 and "601 for 600 samples" in msg, (rc, msg)
rc, msg = mb(mode=0, K=4, mbs=151); assert rc == -1 and "151 samples" in msg, (rc, msg)
rc, msg = mb(mode=0, K=4, mbs=-1); assert rc == -1, (rc, msg)
rc, msg = mb(mode=1, mbs=5); assert rc == -1 and "feed-forward" in msg, (rc, msg)
rc, msg = mb(mode=2, K=25); assert rc == -1 and "25 for 24 columns" in msg, (rc, msg)
rc, msg = mb(mode=2, K=5); assert rc == -1 and "not divisible" in msg, (rc, msg)
rc, msg = mb(k=4); assert rc == -1 and "mini_batch 4 of 4" in msg, (rc, msg)
rc, msg = mb(k=-1); assert rc == -1, (rc, msg)
rc, msg = mb(E=0); assert rc == -1, (rc, msg)
rc, msg = mb(T=1 << 16, B=1 << 15, N=1); assert rc == -1 and "2^31" in msg, (rc, msg)
rc, msg = mb(mode=0, K=4, mbs=150); assert rc == -2, (rc, msg)                     # 4 x 150 = 600: accepted
rc, msg = mb(mode=1, K=60, L=10, k=59); assert rc == -2, (rc, msg)
rc, msg = mb(mode=1, K=7, L=7); assert rc == -2, (rc, msg)                          # T % L != 0: accepted
rc, msg = mb(mode=2, K=24, k=23); assert rc == -2, (rc, msg)
rc, msg = mb(mode=0, K=600, L=0); assert rc == -2, (rc, msg)                        # L is a recurrent option
"""


def test_entry_points_refuse_before_touching_a_device(lib):
    """In a child process that sees no CUDA device: a refusal that came after the device is selected would read
    FM_ERR_CUDA (-2), which is what an accepted call gets there."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = subprocess.run([sys.executable, "-c", _REFUSALS], cwd=ROOT, env=env, capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr


def test_python_generators_refuse_cpu_buffers_and_bad_arguments(monkeypatch):
    from fair_marl_b200.rollout import DeviceRolloutBuffer
    b = DeviceRolloutBuffer(25, 8, 3, 9, device="cpu")
    adv = torch.zeros(25, 8, 3, 1)
    for call in (lambda: b.advantages(), lambda: b.feed_forward_generator(adv, 4), lambda: b.recurrent_generator(adv, 4, 10),
                 lambda: b.naive_recurrent_generator(adv, 4)):
        with pytest.raises(ValueError, match="CUDA buffer"):
            call()
    # the argument checks, with the buffer taken for a CUDA one (nothing reaches a device: each raises before the draw)
    monkeypatch.setattr(DeviceRolloutBuffer, "_require_cuda", lambda self, what: None)
    for call, msg in ((lambda: b.recurrent_generator(adv, 4, 0), "data_chunk_length 0"),
                      (lambda: b.recurrent_generator(adv, 61, 10), "61 for 60 chunks"),
                      (lambda: b.feed_forward_generator(adv, 601), "601 for 600 samples"),
                      (lambda: b.feed_forward_generator(adv, 4, 151), "151 samples"),
                      (lambda: b.feed_forward_generator(adv), "num_mini_batch is required"),
                      (lambda: b.naive_recurrent_generator(adv, 5), "not divisible"),
                      (lambda: b.naive_recurrent_generator(adv, 25), "25 for 24 columns"),
                      (lambda: b.naive_recurrent_generator(adv, 0), "0 for 24 columns"),
                      (lambda: b.recurrent_generator(torch.zeros(25, 8, 3), 4, 10), "advantages")):
        with pytest.raises(ValueError, match=msg):
            call()
