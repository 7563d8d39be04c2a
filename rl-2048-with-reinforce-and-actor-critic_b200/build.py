"""In-tree build of libb2048.so (hand-written CUDA for sm_100a, explicit nvcc, no JIT cache).

The shared library is git-ignored but travels to the GPU box with the repo snapshot."""
from __future__ import annotations

import os
import shutil
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libb2048.so")
SOURCES = ["b2048_capi.cu", "b2048_env.cu", "b2048_policy.cu", "b2048_policy_tc.cu", "b2048_learn.cu", "b2048_learn_tc.cu", "b2048_learn_hp.cu", "b2048_mlp_gen.cu",
           "b2048_lookahead.cu"]
# -cudart shared: torch already loads libcudart; a statically linked runtime would also embed every runtime entry-point
# name in the shipped binary.
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-cudart", "shared"]
OBJ_DIR = os.path.join(PKG_DIR, "build")


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libb2048.so cannot be built")


def sources() -> list[str]:
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(PKG_DIR, "..", "include", "b2048.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB_PATH
    # one nvcc -c per translation unit, in parallel (the units are independent: no relocatable device code), then a link
    os.makedirs(OBJ_DIR, exist_ok=True)
    nvcc = _nvcc()
    hdr_time = max(os.path.getmtime(os.path.join(CSRC, f)) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h")))
    hdr_time = max(hdr_time, os.path.getmtime(os.path.join(PKG_DIR, "..", "include", "b2048.h")))
    procs, objs = [], []
    for src in sources():
        obj = os.path.join(OBJ_DIR, os.path.basename(src)[:-3] + ".o")
        objs.append(obj)
        if not force and os.path.exists(obj) and os.path.getmtime(obj) > max(os.path.getmtime(src), hdr_time):
            continue
        procs.append((src, subprocess.Popen([nvcc] + NVCC_FLAGS + ["-c", "-o", obj, src], cwd=CSRC, stdout=subprocess.PIPE,
                                            stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            print(f"---- {os.path.basename(src)}\n{out}")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed building libb2048.so")
    res = subprocess.run([nvcc, "-shared", "-cudart", "shared", "-o", LIB_PATH] + objs, cwd=CSRC, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout)
        print(res.stderr)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed linking libb2048.so")
    return LIB_PATH


if __name__ == "__main__":
    print(build(force=True, verbose=True))
