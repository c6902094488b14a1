"""Builds libalice_codec.so (sm_100a only) in-tree with nvcc.

    python alice-codec_b200/build.py            # product library  -> alice-codec_b200/lib/libalice_codec.so
    python alice-codec_b200/build.py --emul     # dev-only CPU SIMT emulation of the same sources
                                                #   -> tests/emul/_build/libalice_codec_emul.so (never loaded by the package)
"""
from __future__ import annotations

import argparse
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
SOURCES = ["k_forward.cu", "k_fwd_fused.cu", "k_inv_fused.cu", "k_inverse.cu", "k_rans.cu", "k_generic.cu", "k_wavelet_i32.cu", "k_rdo.cu", "k_rate.cu", "k_synth.cu", "engine.cu", "lossless.cu", "capi.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
              "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr", "-cudart", "static"]


def _digest(paths):
    h = hashlib.sha256()
    for p in sorted(paths):
        with open(p, "rb") as f:
            h.update(p.encode() + b"\0" + f.read())
    return h.hexdigest()


def _inputs():
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h"))]
    srcs.append(os.path.join(ROOT, "include", "alice_codec.h"))
    return srcs


def lib_path():
    return os.path.join(HERE, "lib", "libalice_codec.so")


def build(force=False, verbose=False, variant=None, defines=()):
    """variant/defines: experiment builds (lib/libalice_codec_<variant>.so compiled with extra -D flags); the product
    library is the plain build."""
    out_dir = os.path.join(HERE, "lib")
    obj_dir = os.path.join(out_dir, "obj" + ("_" + variant if variant else ""))
    os.makedirs(obj_dir, exist_ok=True)
    stamp = os.path.join(out_dir, "build" + ("_" + variant if variant else "") + ".sha256")
    digest = _digest(_inputs() + [os.path.abspath(__file__)]) + "".join(defines)
    so = lib_path() if not variant else os.path.join(out_dir, f"libalice_codec_{variant}.so")
    if not force and os.path.exists(so) and os.path.exists(stamp) and open(stamp).read().strip() == digest:
        return so
    if not os.path.exists(NVCC):
        raise RuntimeError(f"nvcc not found at {NVCC}; libalice_codec has no CPU build")

    def compile_one(src):
        obj = os.path.join(obj_dir, src.replace(".cu", ".o"))
        cmd = ([NVCC] + NVCC_FLAGS + ["-D" + d for d in defines] + (["-Xptxas", "-v"] if verbose else []) +
               ["-c", os.path.join(CSRC, src), "-o", obj])
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [NVCC, "-shared", "-o", so] + objs + ["-cudart", "static", "-Xlinker", "--exclude-libs,ALL"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(stamp, "w") as f:
        f.write(digest)
    return so


def emul_lib_path():
    return os.path.join(ROOT, "tests", "emul", "_build", "libalice_codec_emul.so")


def build_emul(force=False, variant=None, defines=()):
    """variant/defines: emulator builds of experiment variants (tests/emul/_build/<variant>/)."""
    out_dir = os.path.dirname(emul_lib_path())
    if variant:
        out_dir = os.path.join(out_dir, variant)
    os.makedirs(out_dir, exist_ok=True)
    stamp = os.path.join(out_dir, "build.sha256")
    emul_h = os.path.join(ROOT, "tests", "emul", "cuda_emul.h")
    digest = _digest(_inputs() + [emul_h, os.path.abspath(__file__)]) + "".join(defines)
    so = os.path.join(out_dir, os.path.basename(emul_lib_path()))
    if not force and os.path.exists(so) and os.path.exists(stamp) and open(stamp).read().strip() == digest:
        return so
    flags = ["-O1", "-g", "-std=c++17", "-fPIC", "-fwrapv", "-DALICE_EMUL", "-x", "c++", "-Wno-unknown-pragmas",
             "-I", os.path.join(ROOT, "tests", "emul"), "-fvisibility=hidden"] + ["-D" + d for d in defines]

    def compile_one(src):
        obj = os.path.join(out_dir, src.replace(".cu", ".o"))
        r = subprocess.run(["g++"] + flags + ["-c", os.path.join(CSRC, src), "-o", obj], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"g++ (emul) failed on {src}:\n{r.stdout}\n{r.stderr}")
        return obj

    with ThreadPoolExecutor(max_workers=8) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    r = subprocess.run(["g++", "-shared", "-o", so] + objs, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link (emul) failed:\n{r.stdout}\n{r.stderr}")
    with open(stamp, "w") as f:
        f.write(digest)
    return so


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--emul", action="store_true")
    ap.add_argument("--force", action="store_true")
    ap.add_argument("-v", "--verbose", action="store_true")
    ap.add_argument("--variant", default=None, help="experiment build name (lib/libalice_codec_<variant>.so)")
    ap.add_argument("-D", dest="defines", action="append", default=[])
    a = ap.parse_args()
    print(build_emul(a.force, a.variant, tuple(a.defines)) if a.emul else build(a.force, a.verbose, a.variant, tuple(a.defines)))
