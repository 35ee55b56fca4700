"""In-tree build of libfoodrec_b200.so (nvcc, sm_100a only).

``python -m foodrec_b200._build`` or ``foodrec_b200._build.build()``.  Each translation
unit is compiled to an object in parallel, then linked.  The .so is git-ignored but
travels to the GPU box with the repo snapshot.
"""
from __future__ import annotations

import concurrent.futures as cf
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "libfoodrec_b200.so")
SOURCES = ["sort.cu", "train_fwd.cu", "train_seg.cu", "train_shard.cu", "eval.cu", "catalog.cu", "catalog_gemm.cu", "sampler.cu", "api.cu", "api_shard.cu",
           "eval_shard.cu"]
HEADERS = ["common.cuh", "internal.h", "train.cuh", "optim.cuh", "ctx.h", "catalog.cuh", "tc05.cuh",
           os.path.join("..", "..", "include", "foodrec_b200.h")]
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC"]


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: cannot build libfoodrec_b200.so")


def sources():
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def source_hash() -> str:
    """sha256 over every source and header (names + bytes) and the compiler flags: what a .so was built from."""
    import hashlib
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    for f in sorted(sources() + [os.path.join(CSRC, x) for x in HEADERS]):
        if os.path.exists(f):
            h.update(os.path.basename(f).encode()); h.update(open(f, "rb").read())
    return h.hexdigest()[:16]


STAMP = LIB + ".stamp"        # source_hash() of the sources the in-tree .so was linked from (travels with it)
LAST = {}                     # what the last build() call did: {"action": "compiled" | "reused", "hash": ..., "objects": n}


def needs_build(lib=LIB) -> bool:
    """The library is rebuilt unless it exists AND its stamp equals the hash of the current sources (mtimes do not
    survive a snapshot; a stale or foreign .so must never be picked up silently)."""
    if not os.path.exists(lib):
        return True
    if lib == LIB:
        return not (os.path.exists(STAMP) and open(STAMP).read().strip() == source_hash())
    t = os.path.getmtime(lib)
    deps = sources() + [os.path.join(CSRC, h) for h in HEADERS]
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def _compile(out_lib, defines=(), verbose=False, tag="") -> str:
    objdir = os.path.join(CSRC, "build" + tag)
    os.makedirs(objdir, exist_ok=True)
    nvcc = _nvcc()
    extra = [f"-D{d}" for d in defines] + (["-Xptxas", "-v"] if verbose else [])
    hdr_t = max(os.path.getmtime(os.path.join(CSRC, h)) for h in HEADERS if os.path.exists(os.path.join(CSRC, h)))

    def one(src):
        obj = os.path.join(objdir, os.path.basename(src)[:-3] + ".o")
        if os.path.exists(obj) and os.path.getmtime(obj) > max(os.path.getmtime(src), hdr_t) and not verbose:
            return obj, ""
        cmd = [nvcc] + NVCC_FLAGS + extra + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        return obj, r.stderr

    with cf.ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 4)) as ex:
        res = list(ex.map(one, sources()))
    if verbose:
        sys.stderr.write("".join(e for _, e in res))
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", out_lib] + [o for o, _ in res]
    r = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    return out_lib


def build(force: bool = False, verbose: bool = False) -> str:
    hsh = source_hash()
    if not force and not verbose and not needs_build():
        LAST.update(action="reused", hash=hsh, lib=LIB)
        return LIB
    if force or not os.path.exists(STAMP) or open(STAMP).read().strip() != hsh:
        # objects are keyed by mtime inside one checkout only: sources that differ from the stamped build start clean
        if force:
            shutil.rmtree(os.path.join(CSRC, "build"), ignore_errors=True)
    out = _compile(LIB, verbose=verbose)
    with open(STAMP, "w") as f:
        f.write(hsh + "\n")
    LAST.update(action="compiled", hash=hsh, lib=LIB)
    return out


def build_variant(name: str, defines) -> str:
    """A/B build of the same sources with extra -D flags -> csrc/libfoodrec_b200_<name>.so
    (selected at run time with FOODREC_B200_LIB=<path>)."""
    return _compile(os.path.join(CSRC, f"libfoodrec_b200_{name}.so"), defines=defines, tag="_" + name)


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
