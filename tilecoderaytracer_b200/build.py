"""Build recipes (no JIT cache: everything lands in-tree so it travels with the repo snapshot).

  build_lib()     nvcc/g++ -> tilecoderaytracer_b200/libtcrt.so   (the product: CUDA kernels for
                  sm_100a + C ABI + host construction API)
  build_oracle()  gcc      -> oracle/_build/liboracle.so          (test infrastructure only)
  build_ref()     oracle/build_ref.sh -> oracle/_ref/*            (the reference itself; only when
                  /root/reference is present)
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "tilecoderaytracer_b200")
CSRC = os.path.join(PKG, "csrc")
LIB_PATH = os.path.join(PKG, "libtcrt.so")
ORACLE_LIB_PATH = os.path.join(ROOT, "oracle", "_build", "liboracle.so")

NVCC = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"

# -fmad=false: the reference's arithmetic is unfused binary32 (SURVEY §8c); contraction
# would change results.  IEEE division and square root are nvcc's defaults
# (-prec-div=true -prec-sqrt=true, -ftz=false) and are stated explicitly.
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-fmad=false", "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-Wall,-Wno-unused-function",
]
CXX_FLAGS = ["-std=c++17", "-O2", "-fPIC", "-ffp-contract=off", "-Wall"]
INCLUDES = ["-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "scenes")]

CUDA_SOURCES = ["tcrt_render.cu", "tcrt_render_grid.cu", "tcrt_render_wave.cu", "tcrt_render_pool.cu", "tcrt_hits.cu", "tcrt_adaptive.cu", "tcrt_format.cu", "tcrt_api.cu", "tcrt_bvh.cpp", "tcrt_cluster.cpp"]
HOST_SOURCES = ["host_scene.cpp", "host_capi.cpp"]


def _run(cmd: list[str], quiet: bool = False) -> None:
    if not quiet:
        print("+", " ".join(cmd), file=sys.stderr, flush=True)
    subprocess.run(cmd, check=True)


def _digest(sources: list[str], extra: str = "") -> str:
    h = hashlib.sha256(extra.encode())
    for s in sorted(sources):
        h.update(os.path.relpath(s, ROOT).encode())
        with open(s, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def _stale(target: str, sources: list[str], extra: str = "") -> bool:
    """Is `target` older than what it is built from?  By CONTENT: the digest of the sources (and flags) a target was
    built from sits next to it in <target>.srchash.  A repo snapshot copied to another machine does not keep
    modification times, and a rebuild there for nothing costs a minute of every test run; without a digest file
    (a target built by hand) modification times decide."""
    if not os.path.exists(target):
        return True
    try:
        with open(target + ".srchash") as f:
            return f.read().strip() != _digest(sources, extra)
    except OSError:
        t = os.path.getmtime(target)
        return any(os.path.getmtime(s) > t for s in sources)


def _stamp(target: str, sources: list[str], extra: str = "") -> None:
    with open(target + ".srchash", "w") as f:
        f.write(_digest(sources, extra) + "\n")


def _deps() -> list[str]:
    deps = []
    for d in (CSRC, os.path.join(ROOT, "include"), os.path.join(ROOT, "scenes")):
        for f in os.listdir(d):
            if f.endswith((".cu", ".cuh", ".cpp", ".h", ".hpp", ".inc")):  # .cuh: shared device helpers
                deps.append(os.path.join(d, f))
    deps.append(os.path.abspath(__file__))
    return deps


def build_lib(force: bool = False, verbose_ptxas: bool = False, defines: tuple = (), out: str | None = None) -> str:
    """Compile libtcrt.so for sm_100a (cross-compiles without a GPU).  `defines`/`out` build a
    developer variant (e.g. ("TCRT_MIN_BLOCKS=3",) -> libtcrt_mb3.so) for A/B timing."""
    lib_path = out or LIB_PATH
    flags = " ".join([*NVCC_FLAGS, *CXX_FLAGS, *defines])
    if not force and not _stale(lib_path, _deps(), flags):
        return lib_path
    objdir = os.path.join(PKG, "build", os.path.basename(lib_path))
    os.makedirs(objdir, exist_ok=True)
    objs = []
    for src in CUDA_SOURCES:
        obj = os.path.join(objdir, src + ".o")
        cmd = [NVCC, *NVCC_FLAGS, *INCLUDES, *[f"-D{d}" for d in defines], "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose_ptxas:
            cmd[1:1] = ["-Xptxas", "-v"]
        _run(cmd)
        objs.append(obj)
    for src in HOST_SOURCES:
        obj = os.path.join(objdir, src + ".o")
        _run(["g++", *CXX_FLAGS, *INCLUDES, "-c", os.path.join(CSRC, src), "-o", obj])
        objs.append(obj)
    # static cudart: the library has no run-time dependency beyond libcuda (the driver)
    _run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-cudart", "static",
          *objs, "-o", lib_path, "-lpthread"])
    _stamp(lib_path, _deps(), flags)
    return lib_path


def build_oracle(force: bool = False) -> str:
    src = os.path.join(ROOT, "oracle", "tcrt_oracle.c")
    deps = [src, os.path.join(ROOT, "include", "tcrt.h")]
    if not force and not _stale(ORACLE_LIB_PATH, deps):
        return ORACLE_LIB_PATH
    os.makedirs(os.path.dirname(ORACLE_LIB_PATH), exist_ok=True)
    _run(["gcc", "-std=gnu11", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-Wall",
          src, "-o", ORACLE_LIB_PATH, "-lm"])
    _stamp(ORACLE_LIB_PATH, deps)
    return ORACLE_LIB_PATH


def build_ref() -> bool:
    """Builds oracle/_ref from /root/reference when it is present; keeps a prebuilt one otherwise."""
    script = os.path.join(ROOT, "oracle", "build_ref.sh")
    ref_bin = os.path.join(ROOT, "oracle", "_ref", "ref_render")
    cnt_bin = os.path.join(ROOT, "oracle", "_ref", "ref_count")
    have_ref = os.path.isdir(os.environ.get("TCRT_REFERENCE_DIR", "/root/reference"))
    srcs = [script, os.path.join(ROOT, "oracle", "ref_harness.cpp"), os.path.join(ROOT, "scenes", "scene_builders.inc")]
    if have_ref and (_stale(ref_bin, srcs) or _stale(cnt_bin, srcs)):
        _run(["bash", script])
        _stamp(ref_bin, srcs)
        _stamp(cnt_bin, srcs)
    return os.path.exists(ref_bin) and os.path.exists(cnt_bin)


if __name__ == "__main__":
    build_lib(force="--force" in sys.argv, verbose_ptxas="-v" in sys.argv)
    build_oracle(force="--force" in sys.argv)
    build_ref()
