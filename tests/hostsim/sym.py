"""Host build of csrc/ac_sym.cuh (test infrastructure): canonical forms and group tables on the CPU."""
import ctypes as C
import os
import subprocess

import numpy as np

from . import CSRC, HERE

SO = os.path.join(HERE, "libsym_host.so")
_SRCS = [os.path.join(HERE, "sym_host.cpp"), os.path.join(HERE, "core_host.cpp")] + [
    os.path.join(CSRC, f) for f in ("ac_core.cuh", "ac_pack.cuh", "ac_keys.cuh", "ac_sym.cuh")]
_lib = None


def _load():
    global _lib
    if _lib is None:
        if not os.path.exists(SO) or any(os.path.getmtime(s) > os.path.getmtime(SO) for s in _SRCS):
            subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++",
                                   "-I/usr/local/cuda/include", "-I" + CSRC, _SRCS[0], "-o", SO])
        _lib = C.CDLL(SO)
        _lib.hostsim_canonical.argtypes = [C.c_void_p] * 4 + [C.c_int64, C.c_int]
        _lib.hostsim_sym_tables.argtypes = [C.c_void_p] * 3
    return _lib


def canonical(rows, apply=None):
    """-> (rows, elements): the canonical forms of int8 rows [n, 2*mrl] and their elements, or with
    ``apply`` (one element per row) the images apply[r].row r."""
    s = np.ascontiguousarray(rows, np.int8)
    n, w = s.shape
    out = np.empty_like(s)
    elem = np.zeros(n, np.uint8)
    a = None if apply is None else np.ascontiguousarray(apply, np.uint8)
    rc = _load().hostsim_canonical(s.ctypes.data, None if a is None else a.ctypes.data, out.ctypes.data,
                                   elem.ctypes.data, n, w // 2)
    assert rc == 0
    return out, elem


def tables():
    """-> (mul [16, 16], inv [16], pi [16, 12]) as the header computes them."""
    mul, inv, pi = np.zeros((16, 16), np.uint8), np.zeros(16, np.uint8), np.zeros((16, 12), np.uint8)
    _load().hostsim_sym_tables(mul.ctypes.data, inv.ctypes.data, pi.ctypes.data)
    return mul, inv, pi
