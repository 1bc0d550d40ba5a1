"""ctypes front-end of tests/bgzf_host.cpp, the CPU build of the BGZF decoder under AddressSanitizer and UBSan
(test infrastructure, not product code).

The harness is compiled on first use into a per-user temporary directory (the source tree stays untouched, so it
may be read-only) as a shared object; `run_in_child` preloads the sanitizer runtime into a child interpreter,
because a sanitized library cannot be loaded into an interpreter started without it."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import sys
import tempfile

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "bgzf_host.cpp")
_HDR = os.path.join(os.path.dirname(_HERE), "ferromic_b200", "csrc", "fm_bgzf.cuh")
SAN_FLAGS = ["-fsanitize=address,undefined", "-fno-sanitize-recover=all", "-fno-omit-frame-pointer"]


def _compiler() -> str:
    """The first C++ compiler that ships the AddressSanitizer runtime ($CXX may be a toolchain without it)."""
    for cxx in (os.environ.get("CXX"), "g++", "/usr/bin/g++", "clang++"):
        if not cxx:
            continue
        try:
            lib = subprocess.check_output([cxx, "-print-file-name=libasan.so"], text=True).strip()
        except (OSError, subprocess.CalledProcessError):
            continue
        if os.path.isabs(lib) and os.path.exists(lib):
            return cxx
    raise RuntimeError("no C++ compiler with the AddressSanitizer runtime (libasan.so) found")


def build() -> str:
    tag = hashlib.sha256(open(_SRC, "rb").read() + open(_HDR, "rb").read()).hexdigest()[:16]
    out_dir = os.path.join(tempfile.gettempdir(), f"ferromic_bgzf_host_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, f"bgzf_host_{tag}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.check_call([_compiler(), "-O1", "-g", "-fPIC", "-std=c++17", "-Wall", "-Wextra", *SAN_FLAGS, "-shared",
                               "-o", tmp, _SRC])
        os.replace(tmp, so)
    return so


def sanitizer_preload() -> str:
    """The ASan runtime the compiler links against, for LD_PRELOAD of the child interpreter."""
    return subprocess.check_output([_compiler(), "-print-file-name=libasan.so"], text=True).strip()


_lib = None


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        vp, sz = C.c_void_p, C.c_size_t
        L.bh_inflate.argtypes = [C.c_char_p, sz, vp, sz, C.POINTER(C.c_uint64), C.POINTER(C.c_int64)]
        L.bh_inflate.restype = C.c_int
        _lib = L
    return _lib


def inflate(gz: bytes):
    """(status, bad member, inflated bytes)."""
    total, bad = C.c_uint64(), C.c_int64()
    st = lib().bh_inflate(gz, len(gz), None, 0, C.byref(total), C.byref(bad))
    if st:
        return st, bad.value, b""
    out = C.create_string_buffer(max(total.value, 1))
    st = lib().bh_inflate(gz, len(gz), out, total.value, C.byref(total), C.byref(bad))
    return st, bad.value, out.raw[:total.value]


def run_in_child(code: str) -> subprocess.CompletedProcess:
    """Runs `code` in a fresh interpreter with the sanitizer runtime preloaded (leak checks off: the interpreter
    itself keeps memory until exit)."""
    env = dict(os.environ)
    env["LD_PRELOAD"] = sanitizer_preload()
    env["ASAN_OPTIONS"] = "detect_leaks=0:abort_on_error=0:exitcode=86"
    env["UBSAN_OPTIONS"] = "print_stacktrace=1:halt_on_error=1:exitcode=87"
    env["PYTHONPATH"] = os.path.dirname(_HERE) + os.pathsep + env.get("PYTHONPATH", "")
    return subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
