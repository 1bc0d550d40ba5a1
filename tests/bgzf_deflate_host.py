"""ctypes front-end of tests/bgzf_deflate_host.cpp, the CPU build of the BGZF encoder (and decoder) under
AddressSanitizer and UBSan (test infrastructure, not product code).  Built like tests/bgzf_host.py: on first use,
into a per-user temporary directory; `bgzf_host.run_in_child` runs code that loads it.  `sanitize=False` builds an
optimised copy of the same code that loads into any interpreter: the GPU tests compare the device's bytes with it."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

from tests import bgzf_host

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRCS = [os.path.join(_HERE, "bgzf_deflate_host.cpp"), os.path.join(_HERE, "bgzf_host.cpp"),
         os.path.join(os.path.dirname(_HERE), "ferromic_b200", "csrc", "fm_bgzf.cuh"),
         os.path.join(os.path.dirname(_HERE), "ferromic_b200", "csrc", "fm_deflate.cuh")]


def build(sanitize: bool = True) -> str:
    tag = hashlib.sha256(b"".join(open(p, "rb").read() for p in _SRCS)).hexdigest()[:16] + ("" if sanitize else "_O2")
    out_dir = os.path.join(tempfile.gettempdir(), f"ferromic_bgzf_host_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, f"bgzf_deflate_host_{tag}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        flags = ["-O1", "-g", *bgzf_host.SAN_FLAGS] if sanitize else ["-O2"]
        subprocess.check_call([bgzf_host._compiler(), *flags, "-fPIC", "-std=c++17", "-Wall", "-Wextra", "-shared",
                               "-o", tmp, _SRCS[0]])
        os.replace(tmp, so)
    return so


_libs = {}


def lib(sanitize: bool = True):
    if sanitize not in _libs:
        L = C.CDLL(build(sanitize))
        vp, sz = C.c_void_p, C.c_size_t
        L.bh_deflate.argtypes = [C.c_char_p, sz, C.c_int, vp, sz, C.POINTER(C.c_uint64)]
        L.bh_walk.argtypes = [C.c_char_p, sz, C.POINTER(C.c_uint64)]
        L.bh_inflate.argtypes = [C.c_char_p, sz, vp, sz, C.POINTER(C.c_uint64), C.POINTER(C.c_int64)]
        for f in (L.bh_deflate, L.bh_walk, L.bh_inflate):
            f.restype = C.c_int
        _libs[sanitize] = L
    return _libs[sanitize]


def deflate(data: bytes, eof: bool = True, sanitize: bool = True) -> bytes:
    """The BGZF stream the device writes for `data`."""
    L, total = lib(sanitize), C.c_uint64()
    L.bh_deflate(data, len(data), int(eof), None, 0, C.byref(total))
    out = C.create_string_buffer(max(total.value, 1))
    L.bh_deflate(data, len(data), int(eof), out, total.value, C.byref(total))
    return out.raw[:total.value]


def walk(gz: bytes, sanitize: bool = True):
    """(status, members) of the member walk."""
    n = C.c_uint64()
    return lib(sanitize).bh_walk(gz, len(gz), C.byref(n)), n.value


def inflate(gz: bytes, sanitize: bool = True):
    """(status, bad member, inflated bytes) from the project's decoder."""
    L, total, bad = lib(sanitize), C.c_uint64(), C.c_int64()
    st = L.bh_inflate(gz, len(gz), None, 0, C.byref(total), C.byref(bad))
    if st:
        return st, bad.value, b""
    out = C.create_string_buffer(max(total.value, 1))
    st = L.bh_inflate(gz, len(gz), out, total.value, C.byref(total), C.byref(bad))
    return st, bad.value, out.raw[:total.value]
