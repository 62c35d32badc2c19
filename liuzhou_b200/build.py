"""Build libliuzhou_b200.so (hand-written sm_100a kernels + C ABI) in-tree with nvcc.

    python -m liuzhou_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU; the resulting .so travels to the GPU box with the repo snapshot.
"""
from __future__ import annotations

import argparse
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

CSRC = Path(__file__).resolve().parent / "csrc"
LIB = CSRC / "libliuzhou_b200.so"
INCLUDE = Path(__file__).resolve().parents[1] / "include"

NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr",
]


def nvcc() -> str:
    """nvcc from PATH, else from $CUDA_HOME or the toolkit's default location."""
    found = shutil.which("nvcc")
    if found:
        return found
    for home in (os.environ.get("CUDA_HOME"), "/usr/local/cuda"):
        if home and (Path(home) / "bin" / "nvcc").is_file():
            return str(Path(home) / "bin" / "nvcc")
    raise RuntimeError("nvcc not found: put the CUDA toolkit's bin directory on PATH or set CUDA_HOME")


def sources() -> list[Path]:
    return sorted(CSRC.glob("*.cu"))


def _deps() -> list[Path]:
    return sources() + sorted(CSRC.glob("*.cuh")) + sorted(INCLUDE.glob("*.h"))


def needs_build() -> bool:
    if not LIB.exists():
        return True
    t = LIB.stat().st_mtime
    return any(p.stat().st_mtime > t for p in _deps())


def build(force: bool = False, verbose: bool = False) -> Path:
    if not force and not needs_build():
        return LIB
    objs = []
    cmds = []
    for src in sources():
        obj = src.with_suffix(".o")
        objs.append(str(obj))
        cmd = [nvcc(), *NVCC_FLAGS, f"-I{INCLUDE}", "-c", str(src), "-o", str(obj)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        cmds.append(cmd)

    def run(cmd):
        res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if res.returncode != 0 or verbose:
            sys.stderr.write(res.stdout)
        if res.returncode != 0:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))

    with ThreadPoolExecutor(max_workers=8) as pool:
        list(pool.map(run, cmds))
    run([nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", *objs, "-o", str(LIB)])
    return LIB


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--force", action="store_true")
    ap.add_argument("--verbose", action="store_true")
    a = ap.parse_args()
    print(build(a.force, a.verbose))
