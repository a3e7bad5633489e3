"""Compile ``libbdg.so`` (the C-ABI library) for sm_100a with nvcc, in-tree.

``python -m bodge_b200.build`` or ``__graft_entry__.build()``.  nvcc cross-compiles without a
GPU, so this runs in the CPU-only build container; the resulting ``.so`` travels to the GPU box.
"""

from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libbdg.so")
PACK = os.path.join(PKG, "_bdgpack.so")  # host-side dict packer (CPython API, no CUDA): csrc/pack_dict.c
SOURCES = ["assemble.cu", "scan.cu", "cheb.cu", "cheb_ell.cu", "cheb_pair.cu", "cheb_cube.cu", "formats.cu", "observables.cu", "multi.cu"]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; libbdg.so cannot be built")


def is_stale() -> bool:
    if not os.path.exists(LIB):
        return True
    built = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if not f.endswith(".c")] + [os.path.join(ROOT, "include", "bdg.h")]
    return any(os.path.getmtime(d) > built for d in deps)


def build_packer(force: bool = False) -> str:
    """gcc -shared csrc/pack_dict.c -> _bdgpack.so (resolves the CPython symbols from the running interpreter)."""
    import sysconfig

    src = os.path.join(CSRC, "pack_dict.c")
    if not force and os.path.exists(PACK) and os.path.getmtime(PACK) >= os.path.getmtime(src):
        return PACK
    cc = os.environ.get("CC") or shutil.which("gcc") or shutil.which("cc")
    if not cc:
        raise RuntimeError("no C compiler found for csrc/pack_dict.c")
    subprocess.run([cc, "-O2", "-Wall", "-shared", "-fPIC", "-I", sysconfig.get_paths()["include"], "-o", PACK, src], check=True)
    return PACK


def build(force: bool = False, verbose: bool = False, defines=(), out: str | None = None) -> str:
    """``defines`` / ``out``: development builds of kernel variants (``-DNAME``) into another file, loaded by
    setting ``BDG_LIB`` (``_native.load``); the product is always ``libbdg.so`` without defines."""
    target = out or LIB
    build_packer(force)
    if not force and not defines and not is_stale():
        return LIB
    cmd = [
        nvcc_path(), "-O3", "-std=c++17", "-lineinfo", "--threads", "0",
        "-gencode", "arch=compute_100a,code=sm_100a",
        "-Xcompiler", "-fPIC,-O2,-Wall", "-shared",
        "-I", os.path.join(ROOT, "include"), "-I", CSRC,
        "-o", target, "-ldl",
    ] + [f"-D{d}" for d in defines] + [os.path.join(CSRC, s) for s in SOURCES]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
        print(" ".join(cmd), file=sys.stderr)
    subprocess.run(cmd, check=True)
    return target


if __name__ == "__main__":
    defs = [a[2:] for a in sys.argv[1:] if a.startswith("-D")]
    outs = [a[2:] for a in sys.argv[1:] if a.startswith("-o")]
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, defines=defs, out=outs[0] if outs else None))
