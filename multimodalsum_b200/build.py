"""In-tree build of libmmsum_b200.so (nvcc, sm_100a only).

`python -m multimodalsum_b200.build` or `__graft_entry__.build()`.  The .so is git-ignored but travels
to the GPU box with the repo snapshot; nothing is JIT-compiled at run time.
"""
import hashlib
import json
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libmmsum_b200.so")
INFO = LIB + ".buildinfo.json"      # written next to the library by build(); git-ignored like the .so, travels with the snapshot
SOURCES = ["gemm_sm100.cu", "attention_sm100.cu", "decode_sm100.cu", "beam_sm100.cu", "sample_sm100.cu", "rowwise.cu", "optim.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O3", "--expt-relaxed-constexpr",
]


def _dep_files():
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    return srcs, srcs + [os.path.join(CSRC, "common.cuh"), os.path.join(HERE, "..", "include", "mmsum_b200.h")]


def source_digest():
    """sha256 over the sources, the shared headers and the compiler flags the library is built from: what ties a shipped
    libmmsum_b200.so to the tree it sits in (file mtimes do not survive the snapshot to the GPU box)."""
    h = hashlib.sha256()
    for f in _dep_files()[1]:
        h.update(os.path.basename(f).encode() + b"\0")
        with open(f, "rb") as fh:
            h.update(hashlib.sha256(fh.read()).digest())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def read_build_info():
    try:
        with open(INFO) as f:
            return json.load(f)
    except (OSError, ValueError):
        return None


def is_current():
    """True when the library exists and its build record matches the sources in this tree (None: no record to compare)."""
    if not os.path.exists(LIB):
        return False
    info = read_build_info()
    if info is None:
        return None
    return info.get("source_digest") == source_digest()


def build(force=False, verbose=False):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    srcs, deps = _dep_files()
    if not force and is_current():
        return LIB
    if not force and is_current() is None and os.path.exists(LIB) and not os.path.exists(nvcc):
        return LIB                                  # a shipped library without a record, and nothing to rebuild it with
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found and %s is missing or stale" % LIB)
    objs = []
    procs = []
    for s in srcs:
        o = os.path.join(CSRC, os.path.basename(s).replace(".cu", ".o"))
        objs.append(o)
        extra = ["-DMMSUM_ATTN_TRACE"] if os.environ.get("MMSUM_TRACE") else []
        cmd = [nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out)
        if p.returncode != 0:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
    subprocess.check_call(cmd)
    ver = subprocess.run([nvcc, "--version"], stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()
    with open(INFO, "w") as f:
        json.dump({"source_digest": source_digest(), "nvcc": ver[-2].strip() if len(ver) >= 2 else "", "flags": NVCC_FLAGS,
                   "arch": "sm_100a", "sources": SOURCES, "trace_build": bool(os.environ.get("MMSUM_TRACE"))}, f, indent=1)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
