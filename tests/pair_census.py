"""The census pairs of tests/test_striped_parity.py (oracle/parasail_striped.c: ps_make_pair) as Python data, so that
the device tests of fadegpu_align_pairs replay exactly the pairs the CPU fuzz checks.

Test infrastructure: tests/native/pair_census.c is compiled on first use into a temporary directory."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_lib = None


def lib():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="fade_pair_census_"), "libpaircensus.so")
        ora = os.path.join(ROOT, "oracle")
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-fopenmp", "-std=gnu11", "-shared", "-I", ora, "-o", out,
                               os.path.join(ROOT, "tests", "native", "pair_census.c"),
                               os.path.join(ora, "fade_oracle.c"), os.path.join(ora, "fade_oracle_simd.c")])
        L = C.CDLL(out)
        L.pc_gen_pairs.argtypes = [C.c_uint64, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p]
        L.pc_gen_pairs.restype = C.c_int
        _lib = L
    return _lib


def gen_pairs(seed: int, first: int, n: int, qmax: int = 72, tmax: int = 160):
    """(query buffer, query offsets[n+1], target buffer, target offsets[n+1]) of census pairs first .. first+n-1"""
    q = np.zeros(max(n, 1) * qmax, np.uint8)
    t = np.zeros(max(n, 1) * tmax, np.uint8)
    qo = np.zeros(n + 1, np.int64)
    to = np.zeros(n + 1, np.int64)
    if lib().pc_gen_pairs(seed, first, n, qmax, tmax, q.ctypes.data, qo.ctypes.data, t.ctypes.data, to.ctypes.data):
        raise ValueError("pc_gen_pairs: bad arguments")
    return q[:qo[n]].copy(), qo, t[:to[n]].copy(), to


def strings(buf: np.ndarray, off: np.ndarray) -> list[bytes]:
    b = buf.tobytes()
    return [b[off[k]:off[k + 1]] for k in range(len(off) - 1)]
