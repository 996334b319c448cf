"""ctypes binding of libtexpose_b200.so (the C-ABI declared in include/texpose_b200.h).

Prototypes are parsed from the header so the Python side can never drift from the ABI.  There is no
CPU fallback: if the shared library is missing, or a call returns non-zero, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes
import os
import re
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(_HERE)
HEADER = os.path.join(ROOT, "include", "texpose_b200.h")
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.environ.get("TEXPOSE_B200_LIB") or os.path.join(_HERE, "libtexpose_b200.so")      # override: A/B builds
SOURCES = ["api.cu", "rays.cu", "mask.cu", "composite.cu", "mlp_simt.cu", "mlp_tc.cu", "mlp_tc_split.cu", "mlp_tc_bwd.cu", "mlp_tc_chain.cu", "loss.cu", "peer.cu", "raster.cu"]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]

_ERRORS = {-1: "bad argument", -2: "bad shape", -3: "misaligned pointer", -4: "device is not sm_100",
           -5: "workspace too small"}

_lib = None


def sources():
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = sources() + [HEADER] + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """nvcc cross-compiles for sm_100a without a GPU; the .so is built in-tree so it travels with the repo."""
    if not force and not needs_build():
        return LIB_PATH
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    extra = os.environ.get("TEXPOSE_NVCC_EXTRA", "").split()      # e.g. -DTP_CHAIN_PROF for scripts/chain_prof.py
    cmd = [nvcc] + NVCC_FLAGS + extra + sources() + ["-o", LIB_PATH]
    if verbose:
        print(" ".join(cmd), file=sys.stderr)
    subprocess.run(cmd, check=True, cwd=CSRC)
    return LIB_PATH


_CTYPE = {"int": ctypes.c_int, "int64_t": ctypes.c_int64, "uint64_t": ctypes.c_uint64, "float": ctypes.c_float,
          "int32_t": ctypes.c_int32, "uint32_t": ctypes.c_uint32}


def declared_prototypes():
    """[(return_type, name, [arg type strings])] for every function declared in the header."""
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    out = []
    for m in re.finditer(r"\b(int|int64_t)\s+(tp_\w+)\s*\(([^)]*)\)\s*;", text):
        ret, name, args = m.group(1), m.group(2), m.group(3).strip()
        arg_types = []
        if args and args != "void":
            for a in args.split(","):
                a = " ".join(a.split())
                arg_types.append(a)
        out.append((ret, name, arg_types))
    return out


def _to_ctype(arg: str):
    if "*" in arg:
        return ctypes.c_void_p
    toks = [t for t in arg.split() if t != "const"]
    return _CTYPE[toks[0]]


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(texpose_b200 has no CPU fallback)")
    lib = ctypes.CDLL(LIB_PATH)
    for ret, name, args in declared_prototypes():
        fn = getattr(lib, name)     # AttributeError here == header/library drift
        fn.restype = _CTYPE[ret]
        fn.argtypes = [_to_ctype(a) for a in args]
    _lib = lib
    return lib


def check(code: int, name: str):
    if code == 0:
        return
    if code < 0:
        raise RuntimeError(f"{name}: {_ERRORS.get(code, 'error')} ({code})")
    raise RuntimeError(f"{name}: CUDA error {code}")


launch_counts = {}      # C-ABI call counts by entry point (bench.py reports them as `gpu_launches`)


def call(name: str, *args):
    lib = load()
    check(getattr(lib, name)(*args), name)
    launch_counts[name] = launch_counts.get(name, 0) + 1
