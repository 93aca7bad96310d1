"""In-tree build of ``libfairmarl.so`` with nvcc for sm_100a (no JIT cache, no torch linkage).

Every ``csrc/*.cu`` is compiled to an object under ``build/`` (in parallel, only when it or a header changed) and the
objects are linked into one shared library next to this file."""
from __future__ import annotations

import os
import shutil
import subprocess
from concurrent.futures import ThreadPoolExecutor

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "csrc")
_OBJ = os.path.join(_HERE, "build")
SOURCES = ["fm_kernels.cu", "fm_aw.cu", "fm_roll.cu", "fm_formation.cu", "fm_form_image.cu", "fm_edges.cu", "fm_soa.cu", "fm_policy.cu", "fm_lsap.cu", "fm_buffer.cu", "fm_abi.cu"]
HEADERS = ["fm_device.cuh", "fm_launch.h", "fm_small.cuh", "fm_aw.cuh", "fm_form.cuh",
           os.path.join("..", "..", "include", "fairmarl.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC"]


def library_path() -> str:
    return os.path.join(_HERE, "libfairmarl.so")


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    raise RuntimeError("nvcc not found: fair_marl_b200 needs the CUDA toolkit to build libfairmarl.so")


def _sources():
    return [s for s in SOURCES if os.path.isfile(os.path.join(_CSRC, s))]


def _headers_mtime() -> float:
    return max(os.path.getmtime(os.path.join(_CSRC, h)) for h in HEADERS if os.path.isfile(os.path.join(_CSRC, h)))


def _stale() -> bool:
    lib = library_path()
    if not os.path.isfile(lib):
        return True
    t = os.path.getmtime(lib)
    return _headers_mtime() > t or any(os.path.getmtime(os.path.join(_CSRC, f)) > t for f in _sources())


def build_library(force: bool = False, verbose: bool = False) -> str:
    """Compile the CUDA sources if the library is missing or older than them.  Returns its path."""
    if not force and not _stale():
        return library_path()
    extra = os.environ.get("FM_NVCC_EXTRA", "").split()      # diagnostics only, e.g. FM_NVCC_EXTRA="-G" for compute-sanitizer runs
    os.makedirs(_OBJ, exist_ok=True)
    nvcc, hdr_t = _nvcc(), _headers_mtime()
    tag = os.path.join(_OBJ, "flags.txt")                    # objects are only reused under the same flags
    flags = " ".join(NVCC_FLAGS + extra)
    same_flags = os.path.isfile(tag) and open(tag).read() == flags

    def compile_one(src: str):
        path, obj = os.path.join(_CSRC, src), os.path.join(_OBJ, src[:-3] + ".o")
        if (not force and same_flags and os.path.isfile(obj)
                and os.path.getmtime(obj) > max(os.path.getmtime(path), hdr_t)):
            return obj, ""
        cmd = [nvcc] + NVCC_FLAGS + extra + (["-Xptxas=-v"] if verbose else []) + ["-c", path, "-o", obj]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
        return obj, res.stderr

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as pool:
        results = list(pool.map(compile_one, _sources()))
    with open(tag, "w") as f:
        f.write(flags)
    if verbose:
        for _, log in results:
            print(log)
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a"] + [o for o, _ in results] + ["-o", library_path()]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc link failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    return library_path()
