"""Build libsod_b200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

The .so lands next to this file so it travels with the repo snapshot to the GPU box; it is
git-ignored.  `python -m sod_b200.build` or `__graft_entry__.build()` run this.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
CSRC = PKG_DIR.parent / "csrc"
LIB_PATH = PKG_DIR / "libsod_b200.so"
OBJ_DIR = PKG_DIR / "_obj"

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
]


LINK_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-lcudart_static", "-ldl", "-lrt",
              "-lpthread"]


def _nvcc() -> str:
    cand = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(cand):
        raise RuntimeError("nvcc not found: the CUDA path has no fallback")
    return cand


def _sources() -> list[Path]:
    return sorted(CSRC.glob("*.cu"))


def _digest() -> str:
    h = hashlib.sha256()
    for p in sorted(list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) +
                    [PKG_DIR.parent.parent / "include" / "sod.h"]):
        h.update(p.name.encode())
        h.update(p.read_bytes())
    h.update(" ".join(NVCC_FLAGS + LINK_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> Path:
    stamp = OBJ_DIR / "digest.txt"
    digest = _digest()
    if not force and LIB_PATH.exists() and stamp.exists() and stamp.read_text() == digest:
        return LIB_PATH
    OBJ_DIR.mkdir(exist_ok=True)
    nvcc = _nvcc()

    def compile_one(src: Path) -> Path:
        obj = OBJ_DIR / (src.stem + ".o")
        cmd = [nvcc, *NVCC_FLAGS, "-c", str(src), "-o", str(obj)]
        r = subprocess.run(cmd, capture_output=True, text=True)
        (OBJ_DIR / (src.stem + ".ptxas.log")).write_text(r.stderr)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src.name}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=4) as ex:
        objs = list(ex.map(compile_one, _sources()))
    cmd = [nvcc, "-o", str(LIB_PATH), *map(str, objs), *LINK_FLAGS]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    stamp.write_text(digest)
    return LIB_PATH


def build_variant(name: str, defines: list[str]) -> Path:
    """Kernel experiments: the same sources with extra -D flags -> libsod_b200.<name>.so next to the
    shipped library (select it with SOD_B200_LIB; never loaded by default)."""
    nvcc = _nvcc()
    out = PKG_DIR / f"libsod_b200.{name}.so"
    cmd = [nvcc, *NVCC_FLAGS, *defines, *map(str, _sources()), "-o", str(out), *LINK_FLAGS]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed for variant {name}:\n{r.stdout}\n{r.stderr}")
    return out


if __name__ == "__main__":
    if "--variant" in sys.argv:    # python -m sod_b200.build --variant checked -DSOD_DEVICE_CHECKS
        i = sys.argv.index("--variant")
        print(build_variant(sys.argv[i + 1], [a for a in sys.argv[i + 2:] if a.startswith("-D")]))
    else:
        print(build(force="--force" in sys.argv, verbose=True))
