"""TEST INFRASTRUCTURE ONLY: the CPU oracle stepped with the two-relaxation-time collision (trt_reference.c).

The library is compiled on first use into a temporary directory, with the flags of oracle/Makefile, so that
running the tests writes nothing into the tree."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile
from pathlib import Path

from oracle import oracle as O

HERE = Path(__file__).resolve().parent
CFLAGS = ["-O3", "-march=x86-64-v3", "-ffp-contract=off", "-fopenmp", "-fPIC", "-Wall", "-Wextra", "-Wno-unused-function"]
_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        cc = "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else "gcc"
        tmp = Path(tempfile.mkdtemp(prefix="trt_reference_"))
        atexit.register(shutil.rmtree, tmp, True)
        src = str(HERE / "trt_reference.c")
        subprocess.run([cc, *CFLAGS, "-DREAL=float", "-DSUF=_f32", "-c", src, "-o", str(tmp / "f32.o")], check=True)
        subprocess.run([cc, *CFLAGS, "-DREAL=double", "-DSUF=_f64", "-DORC_IS_DOUBLE", "-c", src, "-o", str(tmp / "f64.o")],
                       check=True)
        subprocess.run([cc, "-shared", "-fopenmp", "-o", str(tmp / "libtrt_reference.so"), str(tmp / "f32.o"),
                        str(tmp / "f64.o"), "-lm"], check=True)
        _lib = C.CDLL(str(tmp / "libtrt_reference.so"))
        for suf in ("_f32", "_f64"):
            getattr(_lib, "trt_step" + suf).argtypes = [C.c_void_p, C.c_int, C.c_double]
    return _lib


def step(o: O.Oracle, n: int, magic: float):
    """n TRT steps of the oracle handle `o` (it must not be stepped with Oracle.step in between)"""
    getattr(lib(), "trt_step" + o.suf)(o._h, int(n), float(magic))
