"""CPU-side checks of the C ABI: the library builds for sm_100a, loads, exports every symbol
include/fairmarl.h declares, and refuses to work without a GPU (no fallback)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib_path():
    import fair_marl_b200
    return fair_marl_b200.build_library()


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "fairmarl.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(fm_[a-z_0-9]+)\s*\(", text)))


def test_header_symbols_are_exported(lib_path):
    lib = ctypes.CDLL(lib_path)
    declared = _declared_symbols()
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/fairmarl.h but not exported"


def test_binding_covers_header(lib_path):
    from fair_marl_b200 import _lib
    assert sorted(_lib.EXPORTED_SYMBOLS) == _declared_symbols()
    lib = _lib.load()
    assert lib.fm_abi_version() == 6
    assert lib.fm_stats_len(3) == 47


def test_struct_layouts_match_header(tmp_path):
    """sizeof / offsetof of every struct as gcc lays out include/fairmarl.h == the ctypes mirror."""
    import subprocess
    from fair_marl_b200 import _lib
    structs = {"FmConfig": _lib.FmConfig, "FmOutputs": _lib.FmOutputs, "FmState": _lib.FmState,
               "FmFormationConfig": _lib.FmFormationConfig, "FmFormationState": _lib.FmFormationState}
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
    assert ctypes.sizeof(_lib.FmOutputs) == 6 * 8 and ctypes.sizeof(_lib.FmState) == 19 * 8
    assert ctypes.sizeof(_lib.FmFormationState) == 23 * 8       # fm_abi.cu walks it as 23 pointers


def test_library_is_sm100a_only(lib_path):
    import subprocess
    out = subprocess.run(["cuobjdump", "-lelf", lib_path], capture_output=True, text=True).stdout
    assert "sm_100a" in out and "sm_90" not in out and "sm_80" not in out


_NO_CPU_FALLBACK = """
import ctypes
import fair_marl_b200
from fair_marl_b200 import _lib
try:
    fair_marl_b200.B200GraphVecEnv(fair_marl_b200.SimConfig(), num_envs=4)
    raise SystemExit("B200GraphVecEnv was created without a CUDA device")
except _lib.FairMarlError:
    pass
# the C entry point itself reports "no device" instead of computing anything
lib = _lib.load()
cfg = _lib.FmConfig(num_envs=4, num_agents=3, num_obstacles=3, episode_length=25)
h = ctypes.c_void_p()
rc = lib.fm_create(ctypes.byref(cfg), 0, ctypes.byref(h))
assert rc == -4 and b"no CUDA device" in lib.fm_last_error(), (rc, lib.fm_last_error())
"""


def test_no_cpu_fallback(lib_path):
    """Runs in a child process that sees no CUDA device, so the check holds on GPU machines too."""
    import subprocess
    import sys
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = subprocess.run([sys.executable, "-c", _NO_CPU_FALLBACK], cwd=ROOT, env=env, capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr


def test_invalid_config_is_rejected(lib_path):
    from fair_marl_b200 import _lib
    lib = _lib.load()
    h = ctypes.c_void_p()
    cfg = _lib.FmConfig(num_envs=0, num_agents=3, num_obstacles=3, episode_length=25)
    assert lib.fm_create(ctypes.byref(cfg), 0, ctypes.byref(h)) == -1
    cfg = _lib.FmConfig(num_envs=4, num_agents=33, num_obstacles=3, episode_length=25)
    assert lib.fm_create(ctypes.byref(cfg), 0, ctypes.byref(h)) == -1
    assert b"num_agents" in lib.fm_last_error()


def test_formation_entry_points_reject_bad_configs_and_have_no_cpu_path(lib_path):
    import torch
    from fair_marl_b200 import _lib
    lib = _lib.load()
    h = ctypes.c_void_p()
    cfg = _lib.FmFormationConfig(num_envs=4, num_agents=8, num_obstacles=3, episode_length=25)
    assert lib.fm_formation_create(ctypes.byref(cfg), 0, ctypes.byref(h)) == -3 and b"num_agents" in lib.fm_last_error()
    cfg = _lib.FmFormationConfig(num_envs=4, num_agents=3, num_obstacles=9, episode_length=25)
    assert lib.fm_formation_create(ctypes.byref(cfg), 0, ctypes.byref(h)) == -1
    if not torch.cuda.is_available():
        cfg = _lib.FmFormationConfig(num_envs=4, num_agents=3, num_obstacles=3, episode_length=25)
        assert lib.fm_formation_create(ctypes.byref(cfg), 0, ctypes.byref(h)) == -4
        import fair_marl_b200
        with pytest.raises(_lib.FairMarlError):
            fair_marl_b200.B200FormationVecEnv(fair_marl_b200.FormationSimConfig(), num_envs=4)


def test_formation_config_from_reference_namespace():
    from argparse import Namespace
    from fair_marl_b200 import FormationSimConfig
    a = Namespace(num_agents=3, num_landmarks=3, num_obstacles=3, world_size=2, max_speed=2, collision_rew=30, goal_rew=30,
                  min_dist_thresh=0.05, min_obs_dist=0.5, episode_length=25, fair_rew=1.0, zeroshift=5.0, collaborative=False,
                  num_walls=0, num_scripted_agents=0, graph_feat_type="relative",
                  scenario_name="nav_fairassign_nofairrew_formation_graph")
    c = FormationSimConfig.from_args(a)
    assert not c.fairness_reward and c.num_entities == 9 and c.goal_rew == 30
    a.scenario_name = "navigation_graph"
    with pytest.raises(NotImplementedError):
        FormationSimConfig.from_args(a)
    a.scenario_name, a.num_walls = "nav_fairassign_fairrew_formation_graph", 1
    c = FormationSimConfig.from_args(a)
    assert c.num_walls == 1 and c.num_entities == 10 and c.fairness_reward
    a.num_scripted_agents = 1
    with pytest.raises(NotImplementedError):
        FormationSimConfig.from_args(a)


def test_config_from_reference_namespace():
    from argparse import Namespace
    from fair_marl_b200 import SimConfig
    a = Namespace(num_agents=3, num_landmarks=3, num_obstacles=3, world_size=2, max_speed=2, collision_rew=30,
                  goal_rew=30, min_dist_thresh=0.05, episode_length=25, fair_rew=1, zeroshift=5, max_edge_dist=1,
                  collaborative=False, num_walls=0, graph_feat_type="relative", num_scripted_agents=0,
                  scenario_name="navigation_graph", use_dones=False, fair_wt=1)
    c = SimConfig.from_args(a)
    assert c.num_entities == 9 and c.goal_rew == 30 and c.fairness_reward
    a.scenario_name = "nav_graph_goalassign_noFair"
    assert not SimConfig.from_args(a).fairness_reward
    a.num_walls = 1
    assert SimConfig.from_args(a).num_entities == 10            # walls close the entity list
    a.graph_feat_type = "global"
    with pytest.raises(NotImplementedError):                     # no global features for wall entities
        SimConfig.from_args(a)
    a.graph_feat_type, a.num_walls = "relative", 3
    with pytest.raises(ValueError):
        SimConfig.from_args(a)
    a.num_walls, a.num_scripted_agents = 0, 1
    with pytest.raises(NotImplementedError):
        SimConfig.from_args(a)


def test_shard_range_partitions():
    from fair_marl_b200 import shard_range
    for total, world in [(65536, 8), (10, 3), (1, 1), (7, 8)]:
        spans = [shard_range(total, world, r) for r in range(world)]
        assert spans[0][0] == 0 and sum(c for _, c in spans) == total
        for (o1, c1), (o2, _) in zip(spans, spans[1:]):
            assert o1 + c1 == o2


def test_integration_doc_stub_matches_binding():
    """The raw ctypes stub shown to maintainers in INTEGRATION.md must declare FmConfig exactly like the binding
    (a shorter struct would make fm_create read past it)."""
    import re
    from fair_marl_b200 import _lib
    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    block = text[text.index("class FmConfig(C.Structure):"):text.index("class FmOutputs(C.Structure):")]
    doc_fields = re.findall(r'\("(\w+)", C\.(c_\w+)\)', block)
    lib_fields = [(name, ctype.__name__) for name, ctype in _lib.FmConfig._fields_]
    # ctypes aliases: c_int32 is c_int, c_int64 is c_long, ... compare through the types themselves
    import ctypes as C
    assert [(n, getattr(C, t)) for n, t in doc_fields] == list(_lib.FmConfig._fields_), (doc_fields, lib_fields)


def test_integration_doc_formation_stub_matches_binding():
    import ctypes as C
    import re
    from fair_marl_b200 import _lib
    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    block = text[text.index("class FmFormationConfig(C.Structure):"):text.index("fcfg = FmFormationConfig(")]
    doc_fields = re.findall(r'\("(\w+)", C\.(c_\w+)\)', block)
    assert [(n, getattr(C, t)) for n, t in doc_fields] == list(_lib.FmFormationConfig._fields_)


def _load_bench():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_bench_dump_outputs_is_float_bounded_and_reproducible(tmp_path, monkeypatch):
    import numpy as np
    bench = _load_bench()
    B = 1000
    rng = np.random.default_rng(1)
    per_env = {"obs": rng.random((B, 3, 7), dtype=np.float32), "done": rng.integers(0, 2, (B, 3)).astype(np.uint8)}
    whole = {"episode_stats": rng.random(47)}
    bench.dump_outputs(str(tmp_path / "full"), per_env, whole)
    got = {p.stem: np.load(p) for p in (tmp_path / "full").iterdir()}
    assert sorted(got) == ["done", "episode_stats", "obs"]
    assert got["obs"].dtype == np.float32 and got["done"].dtype == np.float32 and got["episode_stats"].dtype == np.float64
    assert np.array_equal(got["obs"], per_env["obs"]) and np.array_equal(got["done"], per_env["done"])
    limit = 20000
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", limit)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), per_env, whole)
    a = {p.stem: np.load(p) for p in (tmp_path / "a").iterdir()}
    b = {p.stem: np.load(p) for p in (tmp_path / "b").iterdir()}
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= limit
    assert 0 < a["obs"].shape[0] < B and a["obs"].shape[0] == a["done"].shape[0]
    rows = [int(np.flatnonzero((per_env["obs"] == r).all(axis=(1, 2)))[0]) for r in a["obs"]]
    assert rows == sorted(rows) and np.array_equal(a["done"], per_env["done"][rows])      # same env rows in every array
    assert all(np.array_equal(a[k], b[k]) for k in a)                                      # the same sample every run
    assert np.array_equal(a["episode_stats"], whole["episode_stats"])


def test_bench_reports_ncu_traffic_only_for_the_matching_kernel():
    """roofline.traffic comes from the ncu capture of the SAME kernel at the SAME size (profiles/step_kernel_traffic.json)."""
    import json
    bench = _load_bench()
    table = json.load(open(os.path.join(ROOT, "profiles", "step_kernel_traffic.json")))
    assert bench.lookup_traffic(table, "fm::aw_kernel<3,3,0> (agent-warp)", 65536, 0) == 13900800
    c3 = bench.lookup_traffic(table, "fm::step_kernel<8> (group-per-env)", 262144, 0)
    alg = table["by_kernel"]["fm::step_kernel<8>"]["algorithmic_bytes_per_launch"]
    assert c3 is not None and 0.9 < c3 / alg < 1.1                       # no wasted re-reads
    assert bench.lookup_traffic(table, "fm::step_kernel<8> (group-per-env)", 4096, 0) is None
    assert bench.lookup_traffic(table, "fm::step_kernel<8> (group-per-env)", 262144, 2) is None
    assert bench.lookup_traffic(table, "fm::step_kernel<8, true> (group-per-env)", 262144, 2) is not None
