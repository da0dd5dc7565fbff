"""Builds the CUDA extension in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m hironaka_b200.build [--force] [--verbose]

Output: hironaka_b200/_lib/libhironaka_b200.so (git-ignored; travels to the GPU box with the
gpurun snapshot).  The library is a plain C-ABI shared object (include/hironaka_b200.h); it is
loaded with ctypes by hironaka_b200._lib and has no Python or torch dependency.  The kernels are
spread over several translation units that compile in parallel and are linked into one library.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "_lib")
OBJ_DIR = os.path.join(OUT_DIR, "obj")
OUT = os.path.join(OUT_DIR, "libhironaka_b200.so")
SOURCES = ["hk_capi.cu", "hk_small_i32_step.cu", "hk_small_i32_obs.cu", "hk_small_f32_step.cu", "hk_small_f32_obs.cu",
           "hk_generic_i32_plain_obs.cu", "hk_generic_f32_plain_obs.cu", "hk_sched_i32.cu", "hk_sched_f32.cu", "hk_sched_i32_obs.cu", "hk_sched_f32_obs.cu", "hk_rows_i32.cu", "hk_rows_f32.cu",
           "hk_small_i32_rec.cu", "hk_small_f32_rec.cu", "hk_generic_i32_rec.cu", "hk_generic_f32_rec.cu",
           "hk_small_i32_thr.cu", "hk_small_f32_thr.cu", "hk_generic_i32_thr.cu", "hk_generic_f32_thr.cu",
           "hk_search.cu"]
HEADERS = ["hk_common.cuh", "hk_census.cuh", "hk_small.cuh", "hk_generic.cuh", "hk_experience.cuh", "hk_value.cuh", "hk_launch.cuh",
           "hk_small_launch.inl", "hk_generic_launch.inl", "hk_sched.cuh", "hk_sched_launch.inl", "hk_rows.cuh", "hk_rows_launch.inl", "hk_sortnet.inc", "hk_search.cuh", "hk_minimax.cuh", "hk_lines.cuh", "hk_labels.cuh", os.path.join("..", "..", "include", "hironaka_b200.h")]

ARCH_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMPILE_FLAGS = ARCH_FLAGS + ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-c"]
LINK_FLAGS = ARCH_FLAGS + ["-shared", "-Xcompiler", "-fPIC", "-cudart", "static"]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def _newest_header() -> float:
    return max(os.path.getmtime(os.path.join(CSRC, h)) for h in HEADERS)


def is_stale() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return _newest_header() > t or any(os.path.getmtime(os.path.join(CSRC, s)) > t for s in SOURCES)


def _compile(nvcc: str, src: str, verbose: bool):
    obj = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
    cmd = [nvcc] + COMPILE_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", obj, os.path.join(CSRC, src)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    return src, obj, r, cmd


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return OUT
    os.makedirs(OBJ_DIR, exist_ok=True)
    nvcc = nvcc_path()
    hdr_t = _newest_header()
    todo, objs = [], []
    for src in SOURCES:
        obj = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        objs.append(obj)
        fresh = os.path.exists(obj) and os.path.getmtime(obj) > max(hdr_t, os.path.getmtime(os.path.join(CSRC, src)))
        if force or not fresh:
            todo.append(src)
    with ThreadPoolExecutor(max_workers=min(len(todo) or 1, os.cpu_count() or 1)) as pool:
        for src, obj, r, cmd in pool.map(lambda s: _compile(nvcc, s, verbose), todo):
            if verbose or r.returncode != 0:
                sys.stderr.write(r.stdout + r.stderr)
            if r.returncode != 0:
                raise RuntimeError("nvcc failed: " + " ".join(cmd))
    r = subprocess.run([nvcc] + LINK_FLAGS + ["-o", OUT] + objs, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("link failed")
    return OUT


def build_variant(name: str, defines, sources=None) -> str:
    """A tuning variant of the library: every source compiled with extra -D macros into
    hironaka_b200/_lib/variants/<name>/ (load it with HIRONAKA_B200_LIB=<path>)."""
    vdir = os.path.join(OUT_DIR, "variants", name)
    os.makedirs(vdir, exist_ok=True)
    nvcc = nvcc_path()
    flags = [f"-D{d}" for d in defines]

    def one(src):
        obj = os.path.join(vdir, src.replace(".cu", ".o"))
        r = subprocess.run([nvcc] + COMPILE_FLAGS + flags + ["-o", obj, os.path.join(CSRC, src)], capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError(f"nvcc failed on {src}")
        return obj
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as pool:
        objs = list(pool.map(one, SOURCES))
    out = os.path.join(vdir, "libhironaka_b200.so")
    r = subprocess.run([nvcc] + LINK_FLAGS + ["-o", out] + objs, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("link failed")
    for o in objs:
        os.remove(o)
    return out


if __name__ == "__main__":
    if "--variant" in sys.argv:  # python -m hironaka_b200.build --variant NAME MACRO=VALUE ...
        i = sys.argv.index("--variant")
        print(build_variant(sys.argv[i + 1], sys.argv[i + 2:]))
    else:
        print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
