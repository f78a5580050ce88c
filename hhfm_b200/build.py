"""Build libhhfm_sm100.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m hhfm_b200.build [--force] [--verbose]

The shared library is git-ignored but travels to the GPU box with the repo snapshot.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libhhfm_sm100.so")
OBJ = os.path.join(HERE, "build")
SOURCES = ["host.cu", "fm.cu", "fm_bn.cu", "pairrank.cu", "opt.cu", "topn.cu", "afm.cu", "afm_fused_tc.cu", "afm_topn.cu", "cars2.cu", "dfm.cu", "dfm_tc.cu", "p2p.cu", "sampler.cu", "topn_tc.cu", "wd.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-O3", "--expt-relaxed-constexpr"]


def _sources():
    return [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _digest():
    h = hashlib.sha256()
    names = sorted(os.listdir(CSRC)) + ["../../include/hhfm_sm100.h"]
    for n in names:
        p = os.path.join(CSRC, n)
        if os.path.isfile(p):
            h.update(n.encode())
            h.update(open(p, "rb").read())
    h.update(" ".join(FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    stamp = os.path.join(OBJ, "digest.txt")
    dig = _digest()
    if not force and os.path.exists(OUT) and os.path.exists(stamp) and open(stamp).read() == dig:
        return OUT
    if not os.path.exists(NVCC):
        raise RuntimeError("nvcc not found at %s; cannot build libhhfm_sm100.so" % NVCC)

    def compile_one(src):
        obj = os.path.join(OBJ, src.replace(".cu", ".o"))
        cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        objs = list(ex.map(compile_one, _sources()))
    cmd = [NVCC, "-shared", "-o", OUT] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    open(stamp, "w").write(dig)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
