"""Builds libsbv2_b200.so in-tree with nvcc for sm_100a (no other architecture, no fallback)."""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
HOST = os.path.join(HERE, "host")
OUT_DIR = os.path.join(HERE, "sbv2_b200")
OBJ_DIR = os.path.join(HERE, "build")
LIB = os.path.join(OUT_DIR, "libsbv2_b200.so")

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC,-Wall,-Wno-unused-function",
         "--expt-relaxed-constexpr", "-I", os.path.join(HERE, "..", "include"), "-I", CSRC, "-I", HOST]


def sources():
    out = []
    for d in (CSRC, HOST):
        if not os.path.isdir(d):
            continue
        for f in sorted(os.listdir(d)):
            if f.endswith((".cu", ".cpp")):
                out.append(os.path.join(d, f))
    return out


def _digest(path: str) -> str:
    h = hashlib.sha1()
    for d in (CSRC, HOST, os.path.join(HERE, "..", "include")):
        if not os.path.isdir(d):
            continue
        for f in sorted(os.listdir(d)):
            if f.endswith((".h", ".cuh", ".hpp")):
                h.update(open(os.path.join(d, f), "rb").read())
    h.update(open(path, "rb").read())
    h.update(" ".join(FLAGS).encode())
    return h.hexdigest()


# Debug hooks (sbv2_debug_conv_compare / _conv_trace / _pair_compare / _attn_trace, the MMA micro-benchmarks, the
# attention / spline / duration / decoder-layer / DeBERTa hooks of debug_kernels.cu) are compiled only with -DSBV2_DEBUG_HOOKS and
# linked only into libsbv2_b200_debug.so, which the kernel unit tests and tools/ load.
# The product library libsbv2_b200.so carries the C ABI of include/sbv2_b200.h and nothing else.
DEBUG_ONLY = {"umma_microbench.cu", "debug_kernels.cu"}     # whole file is a debug facility
DEBUG_VARIANT = {"umma_decoder.cu", "flow_attention_tc.cu", "bert_attention_tc.cu"}  # contain #ifdef SBV2_DEBUG_HOOKS sections
DEBUG_LIB = os.path.join(OUT_DIR, "libsbv2_b200_debug.so")


def build(verbose: bool = False, force: bool = False) -> str:
    os.makedirs(OBJ_DIR, exist_ok=True)
    os.makedirs(os.path.join(OBJ_DIR, "debug"), exist_ok=True)
    objs, dbg_objs, jobs = [], [], []

    def plan(src, obj, flags):
        stamp = obj + ".sha1"
        dig = _digest(src) + " " + " ".join(flags)
        if not force and os.path.exists(obj) and os.path.exists(stamp) and open(stamp).read() == dig:
            return
        extra = ["-x", "cu"] if src.endswith(".cpp") else []
        jobs.append((src, obj, stamp, dig, [NVCC] + FLAGS + flags + (["-Xptxas", "-v"] if verbose else []) + extra + ["-c", src, "-o", obj]))

    for src in sources():
        base = os.path.basename(src)
        obj = os.path.join(OBJ_DIR, base + ".o")
        if os.path.dirname(src) == HOST:
            # the host restatement of the assist-text blend must round like the device kernel: no fused multiply-add
            plan(src, obj, ["-Xcompiler", "-ffp-contract=off"])
            objs.append(obj)
            dbg_objs.append(obj)
            continue
        if base in DEBUG_ONLY or base in DEBUG_VARIANT:
            dobj = os.path.join(OBJ_DIR, "debug", base + ".o")
            plan(src, dobj, ["-DSBV2_DEBUG_HOOKS"])
            dbg_objs.append(dobj)
            if base in DEBUG_ONLY:
                continue
        else:
            dbg_objs.append(obj)
        plan(src, obj, [])
        objs.append(obj)

    def run(job):
        src, obj, stamp, dig, cmd = job
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        open(stamp, "w").write(dig)
        return src

    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        list(ex.map(run, jobs))
    for lib, lst in ((LIB, objs), (DEBUG_LIB, dbg_objs)):
        if jobs or not os.path.exists(lib):
            cmd = [NVCC, "-shared", "-o", lib] + lst + ["-lcudart", "-ldl", "-Xlinker", "-rpath,/usr/local/cuda/lib64"]
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv, force="-f" in sys.argv))
