"""ctypes binding of libcvad_b200.so (the C ABI declared in include/cvad_b200.h).

The prototypes are parsed from the header itself so the binding cannot drift from the ABI.  There is NO fallback:
if the shared library is missing or does not export a declared symbol, importing this module raises.
"""
from __future__ import annotations

import ctypes
import os
import re
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG_DIR)
HEADER = os.path.join(ROOT, "include", "cvad_b200.h")
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libcvad_b200.so")
# development only: A/B a library built from another branch (tools/build_variant.sh) without touching the in-tree one
LOAD_PATH = os.environ.get("CVAD_B200_LIB", LIB_PATH)

# a login shell often lacks the toolkit's bin directory on PATH
NVCC = shutil.which("nvcc") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
              "-Xcompiler", "-fvisibility=hidden", "-I", os.path.join(ROOT, "include"), "-I", CSRC]


class ConvDesc(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int) for n in ("N", "Cin", "Din", "Hin", "Win", "Cout", "Dout", "Hout", "Wout",
                                             "kD", "kH", "kW", "sD", "sH", "sW", "pD", "pH", "pW")] + \
               [("xs", ctypes.c_longlong * 5), ("ys", ctypes.c_longlong * 5)]


class OptState(ctypes.Structure):
    _fields_ = [("gradsq", ctypes.c_double), ("nonfinite", ctypes.c_double), ("last_gradnorm", ctypes.c_double),
                ("step", ctypes.c_longlong * 8), ("skipped", ctypes.c_longlong), ("lr_device", ctypes.c_double)]


def sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = sources() + [HEADER] + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = True) -> str:
    """Compile every csrc/*.cu for sm_100a into libcvad_b200.so (in-tree).  nvcc cross-compiles without a GPU."""
    if not force and not needs_build():
        return LIB_PATH
    objs = []
    os.makedirs(os.path.join(PKG_DIR, "build"), exist_ok=True)
    procs = []
    for src in sources():
        obj = os.path.join(PKG_DIR, "build", os.path.basename(src)[:-3] + ".o")
        objs.append(obj)
        if (not force and os.path.exists(obj) and os.path.getmtime(obj) > os.path.getmtime(src)
                and os.path.getmtime(obj) > os.path.getmtime(HEADER)
                and all(os.path.getmtime(obj) > os.path.getmtime(os.path.join(CSRC, f)) for f in os.listdir(CSRC) if f.endswith(".cuh"))):
            continue
        cmd = [NVCC] + NVCC_FLAGS + ["-c", src, "-o", obj]
        if verbose:
            print("[cvad_b200.build]", " ".join(cmd), flush=True)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{out}")
    cmd = [NVCC, "-shared", "--cudart", "shared", "-o", LIB_PATH] + objs
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    return LIB_PATH


_CTYPE = {"int": ctypes.c_int, "float": ctypes.c_float, "long long": ctypes.c_longlong, "double": ctypes.c_double}


def parse_header(path: str = HEADER):
    """Return {name: (restype, [argtypes])} for every function prototype in the header."""
    text = open(path).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    text = re.sub(r"//[^\n]*", "", text)
    protos = {}
    for m in re.finditer(r"\b(int|long long)\s+(cvad_\w+)\s*\(([^;{}]*?)\)\s*;", text, flags=re.S):
        ret, name, args = m.group(1), m.group(2), m.group(3)
        argtypes = []
        for a in [x.strip() for x in args.replace("\n", " ").split(",") if x.strip()]:
            if a == "void":
                continue
            if "*" in a:
                argtypes.append(ctypes.c_void_p)
            else:
                base = re.sub(r"\bconst\b", "", a).strip()
                base = " ".join(base.split()[:-1])  # drop the parameter name
                argtypes.append(_CTYPE[base])
        protos[name] = (_CTYPE[ret], argtypes)
    return protos


def load():
    if not os.path.exists(LOAD_PATH):
        raise ImportError(
            f"{LOAD_PATH} is missing: the CUDA extension must be built first (python -c 'import __graft_entry__ as g; g.build()'). "
            "There is no CPU fallback.")
    lib = ctypes.CDLL(LOAD_PATH)
    for name, (ret, argtypes) in parse_header().items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise ImportError(f"libcvad_b200.so does not export {name} declared in include/cvad_b200.h") from e
        fn.restype = ret
        fn.argtypes = argtypes
    return lib


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = load()
    return _lib


class CvadError(RuntimeError):
    pass


def check(status: int, what: str) -> None:
    if status != 0:
        # cudaErrorMemoryAllocation == 2: keep torch's wording so callers matching "out of memory" (cad:702-703) still work
        msg = "CUDA out of memory" if status == 2 else f"CUDA error {status}"
        raise CvadError(f"{what}: {msg}")


if __name__ == "__main__":
    build(force="--force" in sys.argv)
    print(LIB_PATH, "exports", len(parse_header()), "symbols")
