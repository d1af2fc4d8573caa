"""Builds libsrl_b200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo).

    python -m srl_b200.build [--force] [--verbose]
"""
from __future__ import annotations

import argparse
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")
LIB = os.path.join(HERE, "libsrl_b200.so")
SOURCES = ["api.cu", "gae_scan.cu", "gae_scan_tma.cu", "gae_scan_ws.cu", "ppo_loss.cu", "ppo_loss_dense.cu", "ppo_loss_gather.cu",
           "ppo_loss_pack.cu", "ppo_loss_pair.cu", "ppo_loss_gaussian.cu", "stats.cu", "perm.cu", "gather.cu", "xchg.cu", "nstep.cu", "gae_general.cu", "host_copy.cu", "rnn_chunk.cu", "blosc_decode.cu"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",  # B200 only; no PTX for other archs, no fallback
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
]
# The GAE scan reproduces the reference's float64 rounding sequence operation by operation: no FMA contraction
# there (its roundings are explicit __dmul_rn / __dadd_rn as well; the flag is the belt to those braces).  The
# loss kernels are compared at 1e-5, so they keep nvcc's default contraction (ncu: FMUL + FADD pairs were a
# quarter of their instructions).
FILE_FLAGS = {"gae_scan.cu": ["-fmad=false"], "gae_scan_tma.cu": ["-fmad=false"], "gae_scan_ws.cu": ["-fmad=false"], "stats.cu": ["-fmad=false"],
              "nstep.cu": ["-fmad=false"], "gae_general.cu": ["-fmad=false"]}


def find_nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def _stale() -> bool:
    if not os.path.isfile(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(INCLUDE, "srl_b200.h"), __file__]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, out: str = LIB, extra_flags=()) -> str:
    """`out` / `extra_flags` (e.g. -DSRL_LOSS_UNROLL=2) build tuning variants next to the product library; load one
    with SRL_B200_LIB=<path> (profiles/ scripts only)."""
    if out == LIB and not force and not _stale():
        return LIB
    from concurrent.futures import ThreadPoolExecutor
    nvcc = find_nvcc()
    objdir = os.path.join(HERE, "build", os.path.basename(out) + ".o")
    os.makedirs(objdir, exist_ok=True)

    def compile_one(src):
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + FILE_FLAGS.get(src, []) + list(extra_flags) + (["-Xptxas", "-v"] if verbose else [])
        cmd += ["-I", INCLUDE, "-c", "-o", obj, os.path.join(CSRC, src)]
        proc = subprocess.run(cmd, capture_output=True, text=True)
        return src, obj, cmd, proc

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 4)) as ex:
        results = list(ex.map(compile_one, SOURCES))
    for src, obj, cmd, proc in results:
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
            print(proc.stderr, file=sys.stderr)
        if proc.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src} ({proc.returncode}):\n{proc.stdout}\n{proc.stderr}")
    link = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", out] + [r[1] for r in results]
    proc = subprocess.run(link, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError(f"link failed ({proc.returncode}):\n{proc.stdout}\n{proc.stderr}")
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--force", action="store_true")
    ap.add_argument("--verbose", action="store_true")
    ap.add_argument("--out", default=LIB)
    ap.add_argument("flags", nargs="*", help="extra nvcc flags after --, e.g. -- -DSRL_LOSS_UNROLL=2")
    a = ap.parse_args()
    print(build(force=a.force, verbose=a.verbose, out=a.out, extra_flags=a.flags))
