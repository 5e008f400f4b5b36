"""Builds libcudf_b200.so in-tree with nvcc for sm_100a (no JIT cache; the .so travels with gpurun)."""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

HERE = Path(__file__).resolve().parent
CSRC = HERE / "csrc"
OBJ = HERE / "build"
LIB = HERE / "libcudf_b200.so"
STAMP = HERE / "libcudf_b200.stamp"
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC,-fvisibility=hidden,-O3", "--expt-relaxed-constexpr", "-DNDEBUG",
]


def _digest(paths) -> str:
    h = hashlib.sha256()
    for p in sorted(paths):
        h.update(p.name.encode())
        h.update(p.read_bytes())
    h.update(" ".join(FLAGS).encode())
    return h.hexdigest()


def _inputs():
    return sorted(CSRC.glob("*.cu")), sorted(CSRC.glob("*.cuh")) + [HERE.parent / "include" / "cudf_b200.h"]


def _up_to_date() -> bool:
    sources, headers = _inputs()
    return LIB.exists() and STAMP.exists() and STAMP.read_text() == _digest(sources + headers)


def build(force: bool = False, verbose: bool = False) -> Path:
    # an up-to-date library is used as it is, without writing to the tree (which may be read-only)
    if not force and _up_to_date():
        return LIB
    # several ranks of a torchrun job may call build() at once: serialise them on a lock file
    import fcntl

    OBJ.mkdir(exist_ok=True)
    with open(OBJ / ".lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            return _build_locked(force, verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(force: bool, verbose: bool) -> Path:
    if not force and _up_to_date():  # another rank built it while this one waited for the lock
        return LIB
    sources, headers = _inputs()
    digest = _digest(sources + headers)
    hdr_digest = _digest(headers)

    def compile_one(src: Path):
        obj = OBJ / (src.stem + ".o")
        key = OBJ / (src.stem + ".key")
        k = hashlib.sha256(src.read_bytes() + hdr_digest.encode()).hexdigest()
        if not force and obj.exists() and key.exists() and key.read_text() == k:
            return obj
        cmd = [NVCC, *FLAGS, "-c", str(src), "-o", str(obj)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src.name}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            print(r.stderr)
        key.write_text(k)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(sources))) as ex:
        objs = list(ex.map(compile_one, sources))
    cmd = [NVCC, "-shared", "-o", str(LIB), *map(str, objs), "-lcudart", "-ldl"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    STAMP.write_text(digest)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
