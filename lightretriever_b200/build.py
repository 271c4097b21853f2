"""In-tree build of liblr_b200.so (sm_100a only, nvcc; no JIT cache, no torch extension machinery).

`python -m lightretriever_b200.build` or `__graft_entry__.build()`.  The shared object is written next to this
file so that it travels with the repository snapshot to the GPU box.
"""
from __future__ import annotations

import fcntl
import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
CSRC = PKG_DIR / "csrc"
LIB_PATH = PKG_DIR / "liblr_b200.so"
OBJ_DIR = PKG_DIR / "csrc" / "_obj"
DIGEST_PATH = PKG_DIR / "liblr_b200.srcdigest"  # digest of the sources the library was built from (travels with it)

SOURCES = [
    "api.cu",
    "embbag.cu",
    "flatip_topk.cu",
    "topk_merge.cu",
    "sparse_head.cu",
    "sparse_score.cu",
    "fuse_topk.cu",
    "query_counts.cu",
    "doc_filter.cu",
]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC",
    
]


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: liblr_b200.so cannot be built")
    return exe


def _dep_files() -> list[Path]:
    files = [CSRC / s for s in SOURCES] + sorted(CSRC.glob("*.cuh")) + [PKG_DIR.parent / "include" / "lr_b200.h"]
    return [f for f in files if f.exists()]


def source_digest() -> str:
    """sha1 over the sources and the compiler flags.  Staleness is decided on content, not on mtimes: the snapshot that
    carries the built library to the GPU box does not preserve them."""
    h = hashlib.sha1()
    h.update(" ".join(NVCC_FLAGS).encode())
    for f in _dep_files():
        h.update(f.name.encode())
        h.update(f.read_bytes())
    return h.hexdigest()


def is_stale() -> bool:
    if not LIB_PATH.exists() or not DIGEST_PATH.exists():
        return True
    return DIGEST_PATH.read_text().strip() != source_digest()


def build(force: bool = False, verbose: bool = False) -> Path:
    if not force and not is_stale():
        return LIB_PATH
    nvcc = _nvcc()
    OBJ_DIR.mkdir(parents=True, exist_ok=True)
    srcs = [s for s in SOURCES if (CSRC / s).exists()]
    missing = sorted(set(SOURCES) - set(srcs))
    if missing:
        raise RuntimeError(f"missing CUDA sources: {missing}")
    # One builder at a time (every rank of a one-process-per-GPU launch may find the library stale at once); whoever gets
    # the lock second finds it fresh.  Objects are written under per-process names and renamed into place.
    with open(OBJ_DIR / ".build.lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        if not force and not is_stale():
            return LIB_PATH
        digest = source_digest()
        tag = f".{os.getpid()}"

        def compile_one(src: str) -> Path:
            obj = OBJ_DIR / (Path(src).stem + ".o")
            tmp_obj = OBJ_DIR / (Path(src).stem + tag + ".o")
            cmd = [nvcc, *NVCC_FLAGS, "-c", str(CSRC / src), "-o", str(tmp_obj)]
            if verbose:
                cmd.insert(1, "-Xptxas")
                cmd.insert(2, "-v")
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
            if verbose:
                sys.stderr.write(r.stderr)
            os.replace(tmp_obj, obj)
            return obj

        with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
            objs = list(ex.map(compile_one, srcs))
        tmp = LIB_PATH.with_suffix(f".so{tag}.tmp")
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(tmp), *map(str, objs)]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
        os.replace(tmp, LIB_PATH)
        DIGEST_PATH.write_text(digest + "\n")
    return LIB_PATH


if __name__ == "__main__":
    p = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(p)
