"""Test builds of the CUDA library: decoy.cu recompiled with extra -D flags (smaller round entries, fewer hash bits, other
repair-loop constants, device-side checks) and linked with the other objects of the regular build.

Each variant is cached under the system temp directory, keyed by a hash of the csrc sources, the public header and the
flags, so the test processes that share a variant compile it once."""
import hashlib
import os
import shutil
import subprocess
import tempfile
from multiprocessing.pool import ThreadPool

import pytest

import maxdecoy

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "max-decoy_b200", "csrc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
FLAGS = ARCH + ["-O3", "-std=c++17", "-Xcompiler", "-fPIC,-fvisibility=hidden", "--expt-relaxed-constexpr", "-cudart", "static"]
OTHERS = ("api.o", "comm.o", "digest.o", "index.o", "exhaustive.o", "score.o")


def _nvcc():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("no nvcc to make the test build")
    return nvcc


def _key(defines):
    h = hashlib.sha256()
    sources = sorted(f for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h")) or f == "Makefile")
    for path in [os.path.join(CSRC, f) for f in sources] + [os.path.join(ROOT, "include", "maxdecoy.h")]:
        h.update(os.path.basename(path).encode() + b"\0")
        with open(path, "rb") as fh:
            h.update(fh.read())
    h.update("\0".join(FLAGS + list(defines)).encode())
    return h.hexdigest()[:20]


def library(defines):
    """Path of the shared library built with `defines` (e.g. ["-DMD_ROUND_ATTEMPTS=64"]); compiled on first use."""
    others = [os.path.join(CSRC, f) for f in OTHERS]
    missing = [f for f in others if not os.path.exists(f)]
    if missing:
        raise FileNotFoundError("the regular build's objects are missing (run __graft_entry__.build() first): %s" % missing)
    cache = os.path.join(tempfile.gettempdir(), "maxdecoy-testbuild-%d" % os.getuid())
    so = os.path.join(cache, "libmaxdecoy_%s.so" % _key(defines))
    if os.path.exists(so):
        return so
    os.makedirs(cache, exist_ok=True)
    nvcc = _nvcc()
    work = tempfile.mkdtemp(dir=cache)
    try:
        obj, tmp_so = os.path.join(work, "decoy.o"), os.path.join(work, "lib.so")
        subprocess.check_call([nvcc] + FLAGS + list(defines) + ["-c", os.path.join(CSRC, "decoy.cu"), "-o", obj])
        subprocess.check_call([nvcc] + ARCH + ["-shared", "-cudart", "static", "-o", tmp_so, obj] + others + ["-ldl"])
        os.replace(tmp_so, so)       # atomic: a concurrent builder of the same variant leaves the same file
    finally:
        shutil.rmtree(work, ignore_errors=True)
    return so


def libraries(variants):
    """library() of several variants, compiled in parallel."""
    with ThreadPool(max(1, len(variants))) as pool:
        return pool.map(library, variants)


def engine(defines):
    """An Engine on the test build with `defines`."""
    return maxdecoy.Engine(lib=maxdecoy.load(library(defines)))
