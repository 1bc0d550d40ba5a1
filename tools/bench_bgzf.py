"""Times BGZF input on the device (fm_bgzf_inflate kernel, fm_vcf_parse_bgzf) against the raw-text chain and against
host inflate.  Prints one JSON line per corpus:
  - gt_gq: synth_text(20000, 2504) from tools/bench_vcf.py (GT:GQ sample fields, 352 MB);
  - gt_only: the same sites with 'a|b' fields only (1000 Genomes-shaped; without GQ in FORMAT every line is an
    error line under the reference's rules, so this corpus times inflate + line index + the fixed-field pass).
Each corpus is BGZF-compressed here at level 6 in 0xff00-byte members, as bgzip writes it.
usage: python tools/bench_bgzf.py [--lines N] [--samples S] [--reps R] [--corpus gt_gq,gt_only]"""
import argparse
import ctypes as C
import json
import os
import struct
import subprocess
import sys
import time
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.bench_vcf import synth_text  # noqa: E402

BGZF_HEAD = b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0"
BGZF_EOF = BGZF_HEAD + struct.pack("<H", 27) + b"\x03\x00" + b"\0" * 8


def _member(chunk: bytes, level: int) -> bytes:
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 8)
    raw = c.compress(chunk) + c.flush()
    return BGZF_HEAD + struct.pack("<H", len(raw) + 25) + raw + struct.pack("<II", zlib.crc32(chunk), len(chunk))


def bgzf_compress(data: bytes, level: int = 6, size: int = 0xff00, threads: int = 0) -> bytes:
    """BGZF as bgzip writes it: members of `size` inflated bytes, then the EOF member (zlib releases the GIL)."""
    with ThreadPoolExecutor(threads or os.cpu_count() or 1) as ex:
        parts = list(ex.map(lambda o: _member(data[o:o + size], level), range(0, len(data), size)))
    return b"".join(parts) + BGZF_EOF


def host_inflate(gz: bytes, threads: int) -> bytes:
    """The host baseline: every member's raw deflate data through zlib on `threads` threads."""
    spans, off = [], 0
    while off < len(gz):
        bsize = struct.unpack_from("<H", gz, off + 16)[0] + 1
        spans.append((off + 18, off + bsize - 8))
        off += bsize
    with ThreadPoolExecutor(threads) as ex:
        return b"".join(ex.map(lambda s: zlib.decompress(gz[s[0]:s[1]], -15), spans))


def gt_only(text: bytes, n_samples: int) -> bytes:
    """synth_text's lines with FORMAT GT and 'a|b' sample fields (the ':QQ' of every field dropped)."""
    out = []
    for line in text.split(b"\n")[:-1]:
        fixed, samples = line.split(b"GT:GQ\t", 1)
        f = np.frombuffer(samples + b"\t", dtype=np.uint8).reshape(n_samples, 7)
        out.append(fixed + b"GT\t" + f[:, [0, 1, 2, 6]].tobytes()[:-1])
    return b"\n".join(out) + b"\n"


def card() -> dict:
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        s = subprocess.check_output(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], text=True)
        return dict(zip(("gpu", "power_limit", "max_sm_clock", "sm_clock_now"), (x.strip() for x in s.split(","))))
    except (OSError, subprocess.CalledProcessError):
        import torch
        return {"gpu": torch.cuda.get_device_name(0)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lines", type=int, default=20000)
    ap.add_argument("--samples", type=int, default=2504)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--corpus", default="gt_gq,gt_only")
    a = ap.parse_args()
    import torch

    from ferromic_b200 import _lib, vcf
    L = _lib.lib()
    kept = np.arange(9, 9 + a.samples, dtype=np.uint32)
    reg = np.array([[0, 1 << 40]], dtype=np.int64)
    p = lambda x: x.ctypes.data_as(C.c_void_p)
    nth = os.cpu_count() or 1
    base = synth_text(a.lines, a.samples)
    info_card = card()

    def pin(b: bytes):
        t = torch.empty(len(b), dtype=torch.uint8).pin_memory()
        t.numpy()[:] = np.frombuffer(b, dtype=np.uint8)
        return t

    def parse(fn, head):
        h = C.c_void_p()
        t0 = time.perf_counter()
        _lib.check(fn(*head, b"1", p(reg), 1, p(kept), len(kept), 30, 0, None, 0, 0, None, 0, 2, C.byref(h)))
        wall = (time.perf_counter() - t0) * 1e3
        return vcf.VcfBatch(h, "1", int(kept[-1])), wall

    for name in a.corpus.split(","):
        text = base if name == "gt_gq" else gt_only(base, a.samples)
        gz = bgzf_compress(text)
        pt, pg = pin(text), pin(gz)
        text_head = (C.cast(pt.data_ptr(), C.c_char_p), len(text))
        gz_head = (C.c_void_p(pg.data_ptr()), len(gz), 0)
        r = {}
        # kernel time: the whole stream as one chunk, so one fm_k_inflate_members launch inside the CUDA events
        os.environ["FM_VCF_CHUNK_MB"] = "4000"
        for rep in range(a.reps + 1):
            b, _ = parse(L.fm_vcf_parse_bgzf, gz_head)
            if rep:
                r["inflate_kernel_ms"] = min(r.get("inflate_kernel_ms", 1e9), float(b.info.inflate_ms))
        del os.environ["FM_VCF_CHUNK_MB"]
        # end to end, default chunking: the BGZF chain against the text chain from page-locked memory
        for rep in range(a.reps + 1):
            bt, wt = parse(L.fm_vcf_parse, text_head)
            bg, wg = parse(L.fm_vcf_parse_bgzf, gz_head)
            if rep and wg < r.get("bgzf_chain_ms", 1e9):
                r.update(bgzf_chain_ms=wg, bgzf_h2d_ms=float(bg.info.h2d_ms), bgzf_inflate_ms=float(bg.info.inflate_ms),
                         bgzf_index_ms=float(bg.info.index_ms), bgzf_parse_ms=float(bg.info.parse_ms))
            if rep and wt < r.get("text_chain_ms", 1e9):
                r.update(text_chain_ms=wt, text_h2d_ms=float(bt.info.h2d_ms))
        parity = (bt.stats() == bg.stats() and bt.errors == bg.errors and np.array_equal(bt.positions, bg.positions)
                  and np.array_equal(bt.flags, bg.flags) and np.array_equal(bt.genotypes(), bg.genotypes())
                  and int(bt.info.n_lines) == int(bg.info.n_lines) == a.lines)
        # fm_bgzf_inflate as a call: compressed bytes up, inflated bytes down
        out = torch.empty(len(text), dtype=torch.uint8).pin_memory()
        tot = C.c_uint64()
        for rep in range(a.reps + 1):
            t0 = time.perf_counter()
            _lib.check(L.fm_bgzf_inflate(C.c_void_p(pg.data_ptr()), len(gz), C.c_void_p(out.data_ptr()), len(text),
                                         C.byref(tot)))
            dt = (time.perf_counter() - t0) * 1e3
            if rep:
                r["bgzf_inflate_call_ms"] = min(r.get("bgzf_inflate_call_ms", 1e9), dt)
        parity = parity and bytes(out.numpy()) == text
        # host baseline: zlib over all host threads, then the text chain
        host = 1e9
        for _ in range(3):
            t0 = time.perf_counter()
            inflated = host_inflate(gz, nth)
            host = min(host, (time.perf_counter() - t0) * 1e3)
        parity = parity and inflated == text
        mb_in, mb_out = len(gz) / 1e6, len(text) / 1e6
        res = {"what": "BGZF on the device vs raw text vs host inflate", "corpus": name, "lines": a.lines,
               "samples": a.samples, "n_variants": int(bg.info.n_variants), "n_errors": int(bg.info.n_errors),
               "compressed_MB": round(mb_in, 3), "inflated_MB": round(mb_out, 3),
               "ratio": round(mb_out / mb_in, 3), **{k: round(v, 3) for k, v in r.items()},
               "inflate_kernel_GBps": round(mb_out / 1e3 / (r["inflate_kernel_ms"] / 1e3), 2),
               "bgzf_h2d_GBps": round(mb_in / 1e3 / (r["bgzf_h2d_ms"] / 1e3), 2),
               "host_inflate_ms": round(host, 3), "host_threads": nth,
               "host_inflate_plus_text_chain_ms": round(host + r["text_chain_ms"], 3),
               "speedup_vs_text_chain": round(r["text_chain_ms"] / r["bgzf_chain_ms"], 3),
               "speedup_vs_host_inflate_chain": round((host + r["text_chain_ms"]) / r["bgzf_chain_ms"], 2),
               "parity": bool(parity), **info_card}
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
