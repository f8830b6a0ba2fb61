"""Build libdiffnet_fem.so (sm_100a only) in-tree with nvcc.

    python -m diffnet_b200.build [--force] [-j N]

One object per translation unit, compiled in parallel.  The variants of each fused-kernel family
(csrc/fem*_combos.h) are split into slices: csrc/fem*_inst.cu is compiled once per (lane width V,
Dirichlet variant MK) for the general families and once per MK for the streaming ones.  This file is
the only list of the slices: one left out leaves the library with an undefined symbol, and it fails
to load.  The library has NO torch dependency: its boundary is the C ABI of include/diffnet_fem.h.
"""
from __future__ import annotations

import argparse
import concurrent.futures as cf
import hashlib
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
OBJ = os.environ.get("DN_BUILD_DIR", os.path.join(PKG, "build"))
LIB = os.environ.get("DN_BUILD_LIB", os.path.join(PKG, "lib", "libdiffnet_fem.so"))

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O2",
    "-DDN_BUILD=1",
] + os.environ.get("DN_NVCC_EXTRA", "").split()

VS = (4, 1)                     # lane widths of the general families (16-byte / scalar row loads)
MKS = (0, 1, 2, 3, 4)           # Dirichlet variants of every family (dn_launch.h: mk_nmasks)
MKS_OP = (5, 6, 7)              # streaming families only: operator apply (mask_input = 0)


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; libdiffnet_fem needs the CUDA 12.9 toolkit to build")


def units() -> list[tuple[str, str, list[str]]]:
    """(source, object name, defines) of every translation unit."""
    out = [(os.path.join(CSRC, n), n[:-3], []) for n in
           ("dn_api.cu", "fem2d_dispatch.cu", "fem2d_tma_dispatch.cu", "fem3d_dispatch.cu", "fem3d_tma_dispatch.cu",
            "gp_eval.cu", "input_grads.cu", "peer.cu", "producers.cu")]
    for dim in (2, 3):
        src = os.path.join(CSRC, f"fem{dim}d_inst.cu")
        out += [(src, f"fem{dim}d_v{v}_mk{mk}", [f"-DDN_V={v}", f"-DDN_MK={mk}"]) for v in VS for mk in MKS]
    for dim in (2, 3):
        src = os.path.join(CSRC, f"fem{dim}d_tma_inst.cu")
        out += [(src, f"fem{dim}dt_mk{mk}", [f"-DDN_MK={mk}"]) for mk in MKS + MKS_OP]
    return out


def _deps_digest() -> str:
    h = hashlib.sha1()
    hdrs = [os.path.join(CSRC, n) for n in sorted(os.listdir(CSRC)) if n.endswith((".cuh", ".h"))]
    hdrs.append(os.path.join(ROOT, "include", "diffnet_fem.h"))
    for p in hdrs:
        h.update(open(p, "rb").read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def _compile_one(args):
    nvcc, src, defines, obj, stamp, digest = args
    key = hashlib.sha1(open(src, "rb").read() + " ".join(defines).encode() + digest.encode()).hexdigest()
    if os.path.exists(obj) and os.path.exists(stamp) and open(stamp).read() == key:
        return obj, 0, "cached"
    cmd = [nvcc, *NVCC_FLAGS, *defines, "-I", os.path.join(ROOT, "include"), "-c", src, "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode == 0:
        with open(stamp, "w") as fh:
            fh.write(key)
    return obj, r.returncode, (r.stdout + r.stderr).strip()


def build(force: bool = False, jobs: int | None = None, verbose: bool = True) -> str:
    nvcc = nvcc_path()
    os.makedirs(OBJ, exist_ok=True)
    os.makedirs(os.path.dirname(LIB), exist_ok=True)
    digest = _deps_digest()
    work = []
    for src, base, defines in units():
        obj, stamp = os.path.join(OBJ, base + ".o"), os.path.join(OBJ, base + ".stamp")
        if force and os.path.exists(stamp):
            os.remove(stamp)
        work.append((nvcc, src, defines, obj, stamp, digest))
    jobs = jobs or min(len(work), max(1, os.cpu_count() or 1))
    rebuilt = 0
    with cf.ThreadPoolExecutor(max_workers=jobs) as ex:
        for obj, rc, msg in ex.map(_compile_one, work):
            if rc != 0:
                raise RuntimeError(f"nvcc failed on {os.path.basename(obj)}:\n{msg}")
            if msg != "cached":
                rebuilt += 1
                if verbose:
                    print(f"[diffnet_b200.build] compiled {os.path.basename(obj)}", flush=True)
    objs = [w[3] for w in work]
    if rebuilt or not os.path.exists(LIB):
        # cudart is linked statically (nvcc default): the library then does not care which
        # libcudart the host process (e.g. torch 2.11+cu128) has loaded; streams are shared
        # through the primary context.
        cmd = [nvcc, "-shared", "-o", LIB, *objs, "-Xlinker", "-soname=libdiffnet_fem.so"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}{r.stderr}")
        if verbose:
            print(f"[diffnet_b200.build] linked {os.path.relpath(LIB, ROOT)} "
                  f"({os.path.getsize(LIB) / 1e6:.1f} MB)", flush=True)
    return LIB


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--force", action="store_true")
    ap.add_argument("-j", type=int, default=None)
    a = ap.parse_args()
    print(build(force=a.force, jobs=a.j))
