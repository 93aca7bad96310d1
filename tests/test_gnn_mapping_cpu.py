"""CPU-side checks of the graph-network mapping choice (fm_gnn_mapping, FmGnnConfig.mapping): which E values are fused
and by which kernel, the refusals of fm_gnn_forward (given before any device is touched), and the struct layout."""
import ctypes
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import fair_marl_b200
    fair_marl_b200.build_library()
    from fair_marl_b200 import _lib
    return _lib.load()


def test_gnn_mapping_over_entity_counts(lib):
    """1 where the warp-per-graph kernel is compiled, 2 for every other 2 <= E <= 64, 0 outside; 0 for node rows outside
    2..17 features."""
    warp = {E for E in range(0, 71) if lib.fm_gnn_supported(E, 11)}
    assert warp and warp <= set(range(2, 65))
    for E in range(0, 71):
        want = 1 if E in warp else (2 if 2 <= E <= 64 else 0)
        for nf in (2, 11, 13, 17):
            assert lib.fm_gnn_mapping(E, nf) == want, (E, nf)
        assert lib.fm_gnn_mapping(E, 1) == 0 and lib.fm_gnn_mapping(E, 18) == 0


_REFUSALS = """
import ctypes
from fair_marl_b200 import _lib
lib = _lib.load()
fake = ctypes.c_void_p(256)                  # never dereferenced: every call below is refused first
def call(E, mapping, NF=11):
    c = _lib.FmGnnConfig(num_graphs=4, graphs_per_adj=1, num_entities=E, node_feat_dim=NF, embed_layers=1, conv_layers=3,
                         aggr=0, relu=1, layer_norm=1, mapping=mapping, max_edge_dist=1.0)
    return lib.fm_gnn_forward(0, ctypes.byref(c), fake, fake, fake, None, fake, None), lib.fm_last_error().decode()
rc, msg = call(35, 1); assert rc == -3 and "mapping 1" in msg, (rc, msg)       # warp kernel not compiled for E = 35
rc, msg = call(65, 2); assert rc == -3 and "65 entities" in msg, (rc, msg)     # beyond the CTA-per-graph kernel
rc, msg = call(65, 0); assert rc == -3, (rc, msg)
rc, msg = call(1, 2); assert rc == -3, (rc, msg)
rc, msg = call(35, 2, NF=18); assert rc == -3, (rc, msg)
rc, msg = call(9, 5); assert rc == -1 and "mapping 5" in msg, (rc, msg)
rc, msg = call(9, -1); assert rc == -1, (rc, msg)
# an accepted configuration gets as far as selecting the device, which fails with a CUDA error
rc, msg = call(35, 2); assert rc == -2, (rc, msg)
"""


def test_gnn_forward_refuses_before_touching_a_device(lib):
    """Runs in a child process that sees no CUDA device: a refusal that came after the device is selected would read
    FM_ERR_CUDA (-2), which is what an accepted configuration gets there."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = subprocess.run([sys.executable, "-c", _REFUSALS], cwd=ROOT, env=env, capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr


def test_gnn_config_layout_matches_header(tmp_path):
    """sizeof / offsetof of FmGnnConfig and FmHeadConfig as gcc lays out include/fairmarl.h == the ctypes mirror."""
    from fair_marl_b200 import _lib
    structs = {"FmGnnConfig": _lib.FmGnnConfig, "FmHeadConfig": _lib.FmHeadConfig}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "fairmarl.h"', 'int main(void) {']
    for name, cls in structs.items():
        lines.append(f'  printf("{name} %zu\\n", sizeof({name}));')
        for field, _ in cls._fields_:
            lines.append(f'  printf("{name}.{field} %zu\\n", offsetof({name}, {field}));')
    lines += ['  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    for name, cls in structs.items():
        assert int(got[name]) == ctypes.sizeof(cls), name
        for field, _ in cls._fields_:
            assert int(got[f"{name}.{field}"]) == getattr(cls, field).offset, f"{name}.{field}"
    assert _lib.FmGnnConfig.mapping.offset == 36 and ctypes.sizeof(_lib.FmGnnConfig) == 48
