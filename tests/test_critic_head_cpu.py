"""CPU-side checks of the wide critic head (fm_critic_head) and the k-node gather (fm_gnn_gather): the packed weight blob
plus a numpy twin of the kernel's algebra reproduce the dense modules, the ctypes mirror of FmCriticHeadConfig matches the
header as gcc lays it out, and both entry points refuse bad input before any device is touched."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
H = 64


@pytest.fixture(scope="module")
def lib():
    import fair_marl_b200
    fair_marl_b200.build_library()
    from fair_marl_b200 import _lib
    return _lib.load()


def _ln(x, g, b):
    m = x.mean(-1, keepdims=True)
    c = x - m
    return c / np.sqrt((c * c).mean(-1, keepdims=True) + np.float32(1e-5)) * g + b


def critic_head_packed(blob, D, cent, rows_per_env, nbd, rnn, mask, *, layers, recurrent, feat_norm, relu):
    """What critic_head_kernel computes from the blob (include/fairmarl.h FmCriticHeadConfig), in float32 numpy."""
    blob = np.asarray(blob, np.float32)
    Dp = (D + 31) // 32 * 32
    o = 0

    def take(n):
        nonlocal o
        x = blob[o:o + n]
        o += n
        return x

    def quads(rows, cols):                                  # [rows / 4][cols][4] -> W^T [rows][cols]
        return take(rows * cols).reshape(rows // 4, cols, 4).transpose(0, 2, 1).reshape(rows, cols)
    act = (lambda v: np.maximum(v, 0)) if relu else np.tanh
    gfn, bfn = take(Dp), take(Dp)
    W1, b1, g1, be1 = quads(Dp, H), take(H), take(H), take(H)
    hidden = [(quads(H, H), take(H), take(H), take(H)) for _ in range(layers)]
    if recurrent:
        Wih, Whh, bih, bhh, gr, br = quads(H, 3 * H), quads(H, 3 * H), take(3 * H), take(3 * H), take(H), take(H)
    Wo, bo = take(8 * H).reshape(8, H), take(8)
    assert o == blob.size and not W1[D:].any() and not Wo[1:].any()
    M = nbd.shape[0]
    x = nbd if cent is None else np.concatenate([np.repeat(cent, rows_per_env, axis=0), nbd], axis=1)   # env m // rows_per_env
    if feat_norm:
        x = _ln(x, gfn[:D], bfn[:D])
    h = _ln(act(x @ W1[:D] + b1), g1, be1)
    for W, b, g, be in hidden:
        h = _ln(act(h @ W + b), g, be)
    hn = None
    if recurrent:
        p = rnn.reshape(M, H) * mask.reshape(M, 1)
        gi, gh = h @ Wih + bih, p @ Whh + bhh
        sig = lambda v: 1 / (1 + np.exp(-v))
        r, z = sig(gi[:, :H] + gh[:, :H]), sig(gi[:, H:2 * H] + gh[:, H:2 * H])
        n = np.tanh(gi[:, 2 * H:] + r * gh[:, 2 * H:])
        hn = (1 - z) * n + z * p
        h = _ln(hn, gr, br)
    return h @ Wo[0] + bo[0], hn


@pytest.mark.parametrize("N,obs_dim,cent,node,layers,recurrent,feat_norm,relu", [
    (3, 7, True, False, 1, True, True, True),          # D = 37
    (3, 7, False, True, 0, False, True, False),        # D = 48
    (7, 11, True, True, 2, True, False, True),         # D = 189 (formation, the widest)
    (16, 7, True, True, 1, True, True, False),         # D = 368
    (32, 7, True, True, 2, False, True, True),         # D = 736 (navigation, the widest)
])
def test_packed_blob_and_kernel_algebra_match_the_dense_modules(N, obs_dim, cent, node, layers, recurrent, feat_norm, relu):
    import fair_marl_b200 as fm
    cfg = fm.PolicyConfig(num_agents=N, obs_dim=obs_dim, use_cent_obs=cent, critic_graph_aggr="node" if node else "global",
                          layer_N=layers, use_recurrent_policy=recurrent, use_feature_normalization=feat_norm, use_ReLU=relu)
    torch.manual_seed(N)
    net = fm.DenseGraphCritic(cfg).eval()
    with torch.no_grad():
        for p in net.parameters():
            p.add_(0.3 * torch.randn_like(p))
    assert net.critic_head_supported()
    D = net._head_in
    B = 6
    M = B * N
    g = torch.Generator().manual_seed(1)
    c = 2 * torch.randn(B, N * obs_dim, generator=g) if cent else None
    nbd = 2 * torch.randn(M, 16 * (N if node else 1), generator=g)
    rnn, mask = torch.randn(M, 1, H, generator=g), (torch.rand(M, 1, generator=g) < 0.7).float()
    with torch.no_grad():
        x = nbd if c is None else torch.cat([c.repeat_interleave(N, 0), nbd], dim=1)
        x = net.base(x)
        hn = None
        if net.recurrent:
            x, hn = net.rnn(x, rnn, mask)
        ref = net.v_out(x)[:, 0].numpy()
        blob = net.pack_head_weights((D + 31) // 32 * 32).numpy()
    out, h = critic_head_packed(blob, D, None if c is None else c.numpy(), N, nbd.numpy(), rnn.numpy(), mask.numpy(),
                                layers=layers, recurrent=net.recurrent, feat_norm=feat_norm, relu=relu)
    assert np.abs(out - ref).max() / max(1.0, np.abs(ref).max()) < 2e-5
    if recurrent:
        assert np.abs(h - hn[:, 0].numpy()).max() < 2e-5


def test_weight_floats_match_the_packer(lib):
    import fair_marl_b200 as fm
    from fair_marl_b200 import _lib
    for N, cent, node, layers, rec in [(3, True, False, 1, True), (32, True, True, 2, False), (5, False, True, 0, True)]:
        cfg = fm.PolicyConfig(num_agents=N, use_cent_obs=cent, critic_graph_aggr="node" if node else "global", layer_N=layers,
                              use_recurrent_policy=rec)
        net = fm.DenseGraphCritic(cfg)
        c = _lib.FmCriticHeadConfig(num_rows=N, cent_dim=7 * N if cent else 0, rows_per_env=N,
                                    nbd_dim=16 * (N if node else 1), layers=layers, recurrent=int(rec))
        assert lib.fm_critic_head_weight_floats(ctypes.byref(c)) == net.pack_head_weights((net._head_in + 31) // 32 * 32).numel()


def test_critic_head_config_layout_matches_header(tmp_path):
    from fair_marl_b200 import _lib
    cls = _lib.FmCriticHeadConfig
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "fairmarl.h"', 'int main(void) {',
             '  printf("size %zu\\n", sizeof(FmCriticHeadConfig));']
    lines += [f'  printf("{f} %zu\\n", offsetof(FmCriticHeadConfig, {f}));' for f, _ in cls._fields_]
    lines += ['  return 0;', '}']
    src, exe = tmp_path / "layout.c", tmp_path / "layout"
    src.write_text("\n".join(lines))
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(got["size"]) == ctypes.sizeof(cls) == 32
    for f, _ in cls._fields_:
        assert int(got[f]) == getattr(cls, f).offset, f


_REFUSALS = """
import ctypes
from fair_marl_b200 import _lib
lib = _lib.load()
fake = ctypes.c_void_p(256)                  # never dereferenced: every refused call below is refused first
def gather(E=9, k=3, mapping=0, aggr=0, aid=fake, NF=11, convs=3):
    c = _lib.FmGnnConfig(num_graphs=4, graphs_per_adj=1, num_entities=E, node_feat_dim=NF, embed_layers=1, conv_layers=convs,
                         aggr=aggr, relu=1, layer_norm=1, mapping=mapping, max_edge_dist=1.0)
    return lib.fm_gnn_gather(0, ctypes.byref(c), k, fake, fake, fake, aid, fake, None), lib.fm_last_error().decode()
rc, msg = gather(k=0); assert rc == -1 and "k 0" in msg, (rc, msg)
rc, msg = gather(k=10); assert rc == -1 and "k 10" in msg, (rc, msg)
rc, msg = gather(aid=None); assert rc == -1 and "null" in msg, (rc, msg)
rc, msg = gather(aggr=1); assert rc == -1 and "aggr 1" in msg, (rc, msg)
rc, msg = gather(E=35, k=16, mapping=1); assert rc == -3 and "mapping 1" in msg, (rc, msg)
rc, msg = gather(E=65, k=16); assert rc == -3, (rc, msg)
rc, msg = gather(mapping=3); assert rc == -1, (rc, msg)
rc, msg = gather(convs=9); assert rc == -3 and "conv_layers 9" in msg, (rc, msg)
rc, msg = gather(E=64, k=64, mapping=2); assert rc == -2, (rc, msg)     # accepted: fails at the device
rc, msg = gather(E=9, k=9, mapping=1); assert rc == -2, (rc, msg)
def head(rows=6, cent=21, per=3, nbd=48, layers=1, rec=1, c_ptr=fake, rnn=fake, value=fake):
    c = _lib.FmCriticHeadConfig(num_rows=rows, cent_dim=cent, rows_per_env=per, nbd_dim=nbd, layers=layers, recurrent=rec,
                                feature_norm=1, relu=1)
    return lib.fm_critic_head(0, ctypes.byref(c), fake, c_ptr, fake, rnn, fake, fake, value, None), lib.fm_last_error().decode()
rc, msg = head(cent=224, nbd=545); assert rc == -3 and "769 input features" in msg, (rc, msg)
rc, msg = head(layers=3); assert rc == -3 and "layers 3" in msg, (rc, msg)
rc, msg = head(layers=-1); assert rc == -3, (rc, msg)
rc, msg = head(c_ptr=None); assert rc == -1, (rc, msg)
rc, msg = head(value=None); assert rc == -1 and "null" in msg, (rc, msg)
rc, msg = head(rnn=None); assert rc == -1 and "recurrent" in msg, (rc, msg)
rc, msg = head(rows=7); assert rc == -1 and "whole number" in msg, (rc, msg)
rc, msg = head(per=0); assert rc == -1, (rc, msg)
rc, msg = head(nbd=0); assert rc == -1, (rc, msg)
rc, msg = head(cent=224, nbd=544); assert rc == -2, (rc, msg)           # D = 768, the cap: accepted
rc, msg = head(cent=0, per=0, c_ptr=None, rec=0, rnn=None); assert rc == -2, (rc, msg)
"""


def test_new_entry_points_refuse_before_touching_a_device(lib):
    """In a child process that sees no CUDA device: a refusal that came after the device is selected would read
    FM_ERR_CUDA (-2), which is what an accepted configuration gets there."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = subprocess.run([sys.executable, "-c", _REFUSALS], cwd=ROOT, env=env, capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
