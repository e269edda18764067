"""CPU restatement of the SSSP tree (sssp_tree_ref.cpp) for the tests, compiled with g++ on first use into a
per-user temporary directory, so the repository tree is never written.

It lives beside the tests rather than in oracle/: oracle.cpp restates the reference's own CPU algorithms line by line
and is pinned against them (tests/test_oracle.py, the golden vectors), and the reference has no SSSP tree to restate
or pin against. This restatement is checked instead against an independent numpy one (tests/test_sssp_tree_oracle.py).

    pred, status = sssp_tree(off, col, w, src, dist)

status is OK (pred is the tree) or the first kind of violation found, in the order of STATUS."""
import ctypes
import hashlib
import os
import subprocess
import tempfile
from ctypes import c_int, c_int32, c_int64, c_void_p

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "sssp_tree_ref.cpp")
OK, INVALID_ENTRY, SOURCE_NOT_ZERO, RELAXABLE_EDGE, ORPHAN = range(5)
STATUS = {OK: "ok", INVALID_ENTRY: "NaN, negative or infinite entry", SOURCE_NOT_ZERO: "source distance is not 0",
          RELAXABLE_EDGE: "relaxable edge", ORPHAN: "reached vertex without a tight path from the source"}
_lib = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        with open(_SRC, "rb") as f:
            tag = hashlib.sha256(f.read()).hexdigest()[:16]
        d = os.path.join(tempfile.gettempdir(), f"essentials-b200-tests-{os.getuid()}")
        os.makedirs(d, exist_ok=True)
        so = os.path.join(d, f"sssp_tree_ref-{tag}.so")
        if not os.path.exists(so):
            tmp = f"{so}.{os.getpid()}"
            subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-o", tmp,
                                   _SRC])
            os.replace(tmp, so)
        L = ctypes.CDLL(so)
        L.sssp_tree_ref.restype = c_int
        L.sssp_tree_ref.argtypes = [c_int64, c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_void_p]
        _lib = L
    return _lib


def sssp_tree(off, col, w, src: int, dist):
    off = np.ascontiguousarray(off, np.int64)
    col = np.ascontiguousarray(col, np.int32)
    w = None if w is None else np.ascontiguousarray(w, np.float32)
    dist = np.ascontiguousarray(dist, np.float32)
    n = off.size - 1
    pred = np.empty(n, np.int32)
    ptr = lambda a: None if a is None else a.ctypes.data_as(c_void_p)
    status = lib().sssp_tree_ref(n, ptr(off), ptr(col), ptr(w), int(src), ptr(dist), ptr(pred))
    return pred, int(status)
