"""Builds libqpskcuda.so in-tree with nvcc for sm_100a (no torch extension machinery needed:
the library is a plain C-ABI shared object, exactly what the C# P/Invoke layer loads)."""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
OBJDIR = os.path.join(HERE, "build")
LIB = os.path.join(LIBDIR, "libqpskcuda.so")

SOURCES = ["core.cu", "fir.cu", "util.cu", "loops.cu", "eq.cu", "fll_duo.cu", "fll_lane.cu", "modulator.cu", "demod.cu", "chain.cu", "stream.cu", "channel.cu", "comm.cu"]

# serial-loop kernels restate C# arithmetic in which RyuJIT never fuses a*b+c: no FMA contraction there
PER_FILE_FLAGS = {"loops.cu": ["--fmad=false"], "eq.cu": ["--fmad=false"], "fll_duo.cu": ["--fmad=false"], "fll_lane.cu": ["--fmad=false"], "demod.cu": ["--fmad=false"], "chain.cu": ["--fmad=false"], "channel.cu": ["--fmad=false"]}

NVCC_FLAGS = [
    "-std=c++17", "-O3",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-fvisibility=hidden,-Wall",
]


def _nvcc() -> str:
    for c in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


def _sha(parts) -> str:
    h = hashlib.sha256()
    for p in parts:
        h.update(p if isinstance(p, bytes) else p.encode())
        h.update(b"\0")
    return h.hexdigest()


def _read(path: str) -> bytes:
    with open(path, "rb") as f:
        return f.read()


def _headers():
    hs = sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h")))
    hs.append(os.path.join(HERE, "..", "include", "qpskcuda.h"))
    return hs


def _nvcc_version(nvcc: str) -> str:
    try:
        out = subprocess.run([nvcc, "--version"], capture_output=True, text=True).stdout
        return out.strip().splitlines()[-1]
    except Exception:
        return "unknown"


def source_id(nvcc_version: str | None = None) -> str:
    """Build stamp: a hash of every csrc/ source and header, include/qpskcuda.h, the nvcc flags (global and per file) and
    the compiler version.  It is compiled into the library (`qpsk_build_id()`); `build()` rebuilds when the library's stamp
    differs from the tree's, and `_native.lib()` refuses a library whose stamp is not the tree's — so a binary shipped with
    the snapshot cannot pass as the build of newer sources (file mtimes do not survive the copy to the GPU box)."""
    if nvcc_version is None:
        nvcc_version = _nvcc_version(_nvcc())
    parts = [nvcc_version, " ".join(NVCC_FLAGS), repr(sorted(PER_FILE_FLAGS.items()))]
    for s in SOURCES:
        parts += [s, _read(os.path.join(CSRC, s))]
    for h in _headers():
        parts += [os.path.basename(h), _read(h)]
    return _sha(parts)[:16]


_MARK = b"QPSK_BUILD_ID="


def library_id(path: str = LIB) -> str | None:
    """The stamp embedded in a built library, read from the file (no dlopen)."""
    if not os.path.exists(path):
        return None
    data = _read(path)
    i = data.find(_MARK)
    if i < 0:
        return None
    j = i + len(_MARK)
    return data[j:j + 16].decode("ascii", "replace")


def build(force: bool = False, verbose: bool = False, ptxas_v: bool = False) -> str:
    os.makedirs(LIBDIR, exist_ok=True)
    os.makedirs(OBJDIR, exist_ok=True)
    nvcc = _nvcc()
    ver = _nvcc_version(nvcc)
    bid = source_id(ver)
    hdr_blob = [_read(h) for h in _headers()]
    jobs = []
    keys = {}
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        obj = os.path.join(OBJDIR, s.replace(".cu", ".o"))
        flags = NVCC_FLAGS + PER_FILE_FLAGS.get(s, [])
        if s == "core.cu":
            flags = flags + [f'-DQPSK_BUILD_ID_STR="{bid}"']     # core.cu carries the stamp, so it rebuilds whenever anything changes
        key = _sha([ver, " ".join(flags), _read(src)] + hdr_blob)
        keys[obj] = key
        old = _read(obj + ".key").decode() if os.path.exists(obj + ".key") else None
        if force or ptxas_v or old != key or not os.path.exists(obj):
            cmd = [nvcc] + flags + (["-Xptxas", "-v"] if ptxas_v else []) + ["-c", src, "-o", obj]
            jobs.append((s, cmd, obj))

    def run(job):
        name, cmd, obj = job
        if os.path.exists(obj + ".key"):
            os.remove(obj + ".key")
        r = subprocess.run(cmd, capture_output=True, text=True)
        return name, r, obj

    with ThreadPoolExecutor(max_workers=max(1, min(len(jobs), os.cpu_count() or 1))) as ex:
        for name, r, obj in ex.map(run, jobs):
            if verbose or ptxas_v or r.returncode != 0:
                sys.stderr.write(f"--- {name}\n{r.stdout}{r.stderr}\n")
            if r.returncode != 0:
                raise RuntimeError(f"nvcc failed on {name}")
            with open(obj + ".key", "w") as f:
                f.write(keys[obj])
    objs = [os.path.join(OBJDIR, s.replace(".cu", ".o")) for s in SOURCES]
    if force or jobs or library_id() != bid:
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs + ["-lcudart_static", "-lpthread", "-ldl", "-lrt"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("link failed")
        if library_id() != bid:
            raise RuntimeError(f"built library carries stamp {library_id()}, expected {bid}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True, ptxas_v="--ptxas-v" in sys.argv))
    print("build id", library_id())
