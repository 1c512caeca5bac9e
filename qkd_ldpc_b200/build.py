"""In-tree build of libqkdldpc_b200.so (hand-written sm_100a CUDA + the C-ABI) and of the host C++ programs.

Everything is compiled with explicit nvcc / g++ command lines; artefacts land in qkd_ldpc_b200/lib/ and
qkd_ldpc_b200/bin/ (git-ignored, but they travel to the GPU box with the gpurun snapshot).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
ROOT = PKG.parent
CSRC = PKG / "csrc"
HOST = PKG / "host"
LIB_DIR = PKG / "lib"
BIN_DIR = PKG / "bin"
LIB_PATH = LIB_DIR / "libqkdldpc_b200.so"
SIM_PATH = BIN_DIR / "qkd_ldpc_b200_sim"

NVCC = os.environ.get("NVCC", shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc")
# /usr/bin/g++ links libstdc++ dynamically; the image's $CXX wrapper links it statically, which breaks when the .so
# is loaded into a Python process that already holds libstdc++.so.6.
HOST_CXX = "/usr/bin/g++" if Path("/usr/bin/g++").exists() else (shutil.which("g++") or "g++")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-ccbin", HOST_CXX, "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall", *os.environ.get("QLB_NVCC_EXTRA", "").split(),
]


def _newer(target: Path, sources) -> bool:
    if not target.exists():
        return False
    t = target.stat().st_mtime
    return all(Path(s).stat().st_mtime <= t for s in sources)


def _run(cmd, log: Path):
    proc = subprocess.run([str(c) for c in cmd], capture_output=True, text=True)
    log.write_text(proc.stdout + proc.stderr)
    if proc.returncode != 0:
        sys.stderr.write(proc.stdout + proc.stderr)
        raise RuntimeError(f"build failed: {' '.join(str(c) for c in cmd)}")


TRANSLATION_UNITS = ["qlb_api.cu", "qlb_tu_generic.cu", "qlb_tu_resident_f32.cu", "qlb_tu_stream.cu", "qlb_tu_resident_f64.cu",
                     "qlb_rate.cu"]


def build_library(force: bool = False, verbose_ptxas: bool = True, out: Path = LIB_PATH, extra_flags=()) -> Path:
    """One object per translation unit, compiled in parallel, linked into `out` (default: libqkdldpc_b200.so).
    `extra_flags`: more nvcc flags, e.g. the -D knobs of a variant library; a library other than the default keeps its objects
    and logs in a directory of its own beside it."""
    from concurrent.futures import ThreadPoolExecutor
    out = Path(out)
    work = LIB_DIR if out == LIB_PATH else out.parent / (out.stem + "_build")
    obj_dir = work / "obj"
    obj_dir.mkdir(parents=True, exist_ok=True)
    headers = sorted(CSRC.glob("*.cuh")) + sorted(CSRC.glob("*.hpp")) + [ROOT / "include" / "qkd_ldpc_b200.h"]
    sources = [CSRC / tu for tu in TRANSLATION_UNITS]
    if not force and _newer(out, sources + headers):
        return out
    flags = [*NVCC_FLAGS, *extra_flags]

    def compile_tu(src: Path) -> Path:
        obj = obj_dir / (src.stem + ".o")
        if force or not _newer(obj, [src] + headers):
            cmd = [NVCC, *flags, "-c", "-o", obj, src]
            if verbose_ptxas:
                cmd += ["-Xptxas", "-v"]
            _run(cmd, work / f"build_{src.stem}.log")
        return obj

    with ThreadPoolExecutor(max_workers=len(sources)) as pool:
        objs = list(pool.map(compile_tu, sources))
    _run([NVCC, *flags, "-shared", "-o", out, *objs, "-ldl"], work / "build_link.log")
    (work / "build_lib.log").write_text("".join((work / f"build_{src.stem}.log").read_text() for src in sources
                                                if (work / f"build_{src.stem}.log").exists()))
    return out


def build_host(force: bool = False) -> Path | None:
    """The host-side C++ mirror of the reference API + the config.json-driven simulation binary."""
    srcs = sorted(HOST.glob("*.cpp"))
    if not srcs:
        return None
    BIN_DIR.mkdir(exist_ok=True)
    deps = srcs + sorted(HOST.glob("*.hpp")) + [ROOT / "include" / "qkd_ldpc_b200.h", LIB_PATH]
    if not force and _newer(SIM_PATH, deps):
        return SIM_PATH
    cmd = [HOST_CXX, "-std=c++20", "-O2", "-Wall", "-pthread", f"-I{ROOT / 'include'}", f"-I{HOST}", "-o", SIM_PATH, *srcs,
           f"-L{LIB_DIR}", "-lqkdldpc_b200", f"-Wl,-rpath,{LIB_DIR}", "-Wl,-rpath,$ORIGIN/../lib", "-ldl"]
    _run(cmd, LIB_DIR / "build_host.log")
    return SIM_PATH


def build_all(force: bool = False) -> None:
    build_library(force)
    build_host(force)


if __name__ == "__main__":
    build_all(force="--force" in sys.argv)
    print(LIB_PATH)
