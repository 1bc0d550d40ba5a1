"""ctypes front-end of the CPU ORACLE of calculate_pairwise_differences (stats.rs:4106-4231, parity unpinned;
test infrastructure, NOT product code).

tests/pairwise_oracle.c is compiled on first use into a per-user temporary directory (the source tree stays
untouched, so it may be read-only).  Variants are oracle.pyoracle.Variants (the sparse CompressedGenotypes
layout)."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "pairwise_oracle.c")
_lib = None


def _build() -> str:
    src = open(_SRC, "rb").read()
    tag = hashlib.sha256(src).hexdigest()[:16]
    out_dir = os.path.join(tempfile.gettempdir(), f"ferromic_pairwise_oracle_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, f"pairwise_oracle_{tag}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        cc = os.environ.get("CC", "gcc")
        subprocess.check_call([cc, "-O2", "-fPIC", "-std=c11", "-Wall", "-Wextra", "-shared", "-o", tmp, _SRC,
                               "-lpthread"])
        os.replace(tmp, so)
    return so


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(_build())
        vp, sz = C.c_void_p, C.c_size_t
        L.pw_pairwise_differences.argtypes = [vp, sz, vp, vp, vp, vp]
        L.pw_pairwise_differences.restype = None
        L.pw_pairwise_differences_mt.argtypes = [vp, sz, vp, vp, C.c_int]
        L.pw_pairwise_differences_mt.restype = None
        _lib = L
    return _lib


def _ptr(a):
    return None if a is None else a.ctypes.data


def pairwise_differences(vs, sample_count: int, threads: int = 0):
    """(differences, comparable, pair_start, positions) over the pairs i < j of 0 .. sample_count-1 in pdist
    order.  threads > 0 runs the threaded rows form and returns counts only (pair_start and positions are None)."""
    n = int(sample_count)
    n_pairs = n * (n - 1) // 2
    diff = np.zeros(n_pairs, dtype=np.uint32)
    comp = np.zeros(n_pairs, dtype=np.uint32)
    v = C.addressof(vs._c)
    if threads > 0:
        lib().pw_pairwise_differences_mt(v, n, _ptr(diff), _ptr(comp), threads)
        return diff, comp, None, None
    start = np.zeros(n_pairs + 1, dtype=np.uint64)
    lib().pw_pairwise_differences(v, n, _ptr(diff), _ptr(comp), _ptr(start), None)
    pos = np.zeros(max(int(start[-1]), 1), dtype=np.int64)
    lib().pw_pairwise_differences(v, n, _ptr(diff), _ptr(comp), _ptr(start), _ptr(pos))
    return diff, comp, start, pos[:int(start[-1])]
