"""
Builds ``matten_b200/lib/libmatten_b200.so`` (the C ABI of include/matten_b200.h) with
nvcc for sm_100a, in-tree.  nvcc cross-compiles without a GPU.

    python -m matten_b200.build [--force] [-j N]
"""
from __future__ import annotations

import argparse
import concurrent.futures as cf
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
OBJDIR = os.path.join(HERE, "lib", "obj")
LIBNAME = "libmatten_b200.so"

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
    "-Xptxas", "-v",
]

PLAIN_SOURCES = ["api.cu", "graph_ops.cu", "node_ops.cu", "train_ops.cu", "norm_ops.cu", "conv.cu", "conv_fwd_tc.cu", "conv_bwd.cu"]
CONV_INST = [(t, hp) for t in ("float", "double") for hp in (8, 16, 32, 64)]


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


def _deps_hash(paths) -> str:
    h = hashlib.sha256()
    for p in sorted(paths):
        with open(p, "rb") as f:
            h.update(p.encode())
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def _all_headers():
    out = []
    for root, _, files in os.walk(CSRC):
        for f in files:
            if f.endswith((".cuh", ".h")):
                out.append(os.path.join(root, f))
    out.append(os.path.join(HERE, "..", "include", "matten_b200.h"))
    return out


def _compile(job):
    src, obj, extra, log = job
    cmd = [_nvcc()] + NVCC_FLAGS + extra + ["-c", src, "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    with open(log, "w") as f:
        f.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed for {src}:\n{r.stderr[-4000:]}")
    return obj


def build(force: bool = False, jobs: int | None = None, verbose: bool = True) -> str:
    os.makedirs(OBJDIR, exist_ok=True)
    gen = os.path.join(CSRC, "generated", "cg_gen.cuh")
    if not os.path.exists(gen):
        from .codegen import gen_tables

        gen_tables.main()
    headers = _all_headers()
    stamp_path = os.path.join(OBJDIR, "stamp")
    srcs = [os.path.join(CSRC, s) for s in os.listdir(CSRC) if s.endswith(".cu")]
    stamp = _deps_hash(srcs + headers)
    lib = os.path.join(LIBDIR, LIBNAME)
    if not force and os.path.exists(lib) and os.path.exists(stamp_path) and open(stamp_path).read() == stamp:
        return lib
    work = []
    for s in PLAIN_SOURCES:
        work.append((os.path.join(CSRC, s), os.path.join(OBJDIR, s[:-3] + ".o"), [],
                     os.path.join(OBJDIR, s[:-3] + ".log")))
    for t, hp in CONV_INST:
        name = f"conv_fwd_{t}_{hp}"
        work.append((os.path.join(CSRC, "conv_fwd_inst.cu"), os.path.join(OBJDIR, name + ".o"),
                     [f"-DMT_INST_T={t}", f"-DMT_INST_HP={hp}"], os.path.join(OBJDIR, name + ".log")))
    jobs = jobs or min(len(work), os.cpu_count() or 4)
    if verbose:
        print(f"[matten_b200.build] compiling {len(work)} units with {jobs} jobs ...", file=sys.stderr)
    with cf.ThreadPoolExecutor(max_workers=jobs) as ex:
        objs = list(ex.map(_compile, work))
    cmd = [_nvcc(), "-shared", "-o", lib] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stderr[-4000:]}")
    with open(stamp_path, "w") as f:
        f.write(stamp)
    if verbose:
        print(f"[matten_b200.build] wrote {lib}", file=sys.stderr)
    return lib


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--force", action="store_true")
    ap.add_argument("-j", type=int, default=None)
    a = ap.parse_args()
    print(build(force=a.force, jobs=a.j))
