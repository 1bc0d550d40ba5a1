"""Times BGZF deflate on the device (fm_bgzf_deflate, fm_falsta_tracks_bgzf) on two corpora and prints one JSON line
per corpus:

- falsta: the tools/bench_falsta.py shape (6 FST tracks over a 5 Mb region, 150k records, ~94 MB of text).  The
  compressed render call is set against the text render call (fm_falsta_tracks), that call plus host zlib level 6 in
  BGZF members on all host threads, and the writer's default gzip level 9 pass over the whole text.
- vcf: synth_text(20000, 2504), 352 MB of GT:GQ text, through fm_bgzf_deflate.

Kernel time is the sum of fm_k_deflate_members' device time in torch.profiler (CUDA activity) records of one warmed
call.  Ratios are next to zlib level 1 and level 6 in the same 0xff00 members.  Every output is checked by a round
trip.  The device name, power limit and SM clocks are read in the same run."""
import ctypes as C
import gzip
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def best_ms(f, reps):
    best = None
    for _ in range(reps):
        t0 = time.perf_counter()
        f()
        dt = (time.perf_counter() - t0) * 1e3
        best = dt if best is None or dt < best else best
    return best


def kernel_ms(f):
    """Device time of fm_k_deflate_members during one call of f."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        f()
        torch.cuda.synchronize()
    total = 0.0
    for e in prof.events():
        if "fm_k_deflate_members" in e.name:
            total += getattr(e, "device_time", None) or getattr(e, "cuda_time", 0.0)
    return total / 1e3 if total else None


def device_info():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def zlib_bgzf(data, level):
    from tools.bench_bgzf import bgzf_compress
    t0 = time.perf_counter()
    gz = bgzf_compress(data, level=level)
    return gz, (time.perf_counter() - t0) * 1e3


def main():
    import torch
    torch.cuda.init()
    from ferromic_b200 import _lib, falsta, vcf
    L = _lib.lib()
    reps = int(os.environ.get("REPS", "5"))
    info = device_info()
    threads = os.cpu_count()

    # ---------------------------------------------------------------- falsta
    rng = np.random.default_rng(5)
    region_len, n, T = 5_000_000, 150_000, 6
    pos = np.sort(rng.choice(np.arange(1, region_len + 1), size=n, replace=False)).astype(np.int64)
    vals = rng.random((T, n))
    vals[rng.random((T, n)) < 0.1] = np.nan
    vals[rng.random((T, n)) < 0.1] = 0.0
    vals = np.ascontiguousarray(vals)
    heads = [f">track_{t}_chr_1_start_1_end_{region_len}\n" for t in range(T)]
    c_heads = (C.c_char_p * T)(*[h.encode() for h in heads])
    pp, vp = pos.ctypes.data_as(C.c_void_p), vals.ctypes.data_as(C.c_void_p)
    cap = 120_000_000
    buf = np.empty(cap, dtype=np.uint8)
    lens = (C.c_size_t * T)()
    size = C.c_size_t(0)

    def render():
        _lib.check(L.fm_falsta_tracks(pp, vp, n, T, 1, region_len, falsta.FST, buf.ctypes.data_as(C.c_void_p), cap,
                                      lens, C.byref(size)))

    def render_bgzf():
        _lib.check(L.fm_falsta_tracks_bgzf(pp, vp, n, T, 1, region_len, falsta.FST, C.cast(c_heads, C.c_void_p),
                                           buf.ctypes.data_as(C.c_void_p), cap, C.byref(size)))

    for f in (render, render_bgzf):
        f()
    render_ms = best_ms(render, reps)
    lines = falsta.track_lines(pos, vals, 1, region_len, falsta.FST)
    text = b"".join(h.encode() + line + b"\n" for h, line in zip(heads, lines))
    bgzf_ms = best_ms(render_bgzf, reps)
    members = buf[:size.value].tobytes()
    ok = gzip.decompress(members) == text and vcf.bgzf_inflate(members) == text
    krn = kernel_ms(render_bgzf)
    z1, _ = zlib_bgzf(text, 1)
    host6 = None
    for _ in range(2):
        t0 = time.perf_counter()
        render()
        z6 = zlib_bgzf(buf[:size.value].tobytes(), 6)[0]
        dt = (time.perf_counter() - t0) * 1e3
        host6 = dt if host6 is None or dt < host6 else host6
    t0 = time.perf_counter()
    g9 = gzip.compress(text, 9)
    gzip9_ms = (time.perf_counter() - t0) * 1e3
    print(json.dumps({
        "corpus": "falsta: 6 FST tracks, 5 Mb region, 150k records", **info, "text_bytes": len(text),
        "members_bytes": len(members), "ratio": len(text) / len(members),
        "ratio_zlib1_bgzf": len(text) / len(z1), "ratio_zlib6_bgzf": len(text) / len(z6),
        "ratio_gzip9_whole": len(text) / len(g9), "size_vs_zlib1": len(members) / (len(z1) - 28),
        "deflate_kernel_ms": krn, "deflate_kernel_GBps": len(text) / krn / 1e6 if krn else "not measured",
        "fm_falsta_tracks_bgzf_ms": bgzf_ms, "fm_falsta_tracks_ms": render_ms,
        "fm_falsta_tracks_plus_host_zlib6_ms": host6, "host_threads": threads,
        "writer_gzip9_ms": gzip9_ms, "round_trip_ok": ok}), flush=True)

    # ---------------------------------------------------------------- vcf
    from tools.bench_vcf import synth_text
    text = synth_text(20000, 2504)
    out = np.empty(len(text) + len(text) // 1000 + 4096, dtype=np.uint8)

    def deflate():
        _lib.check(L.fm_bgzf_deflate(text, len(text), _lib.FM_BGZF_EOF, out.ctypes.data_as(C.c_void_p), out.size,
                                     C.byref(size)))

    deflate()
    call_ms = best_ms(deflate, reps)
    gz = out[:size.value].tobytes()
    ok = vcf.bgzf_inflate(gz) == text
    krn = kernel_ms(deflate)
    z1, z1_ms = zlib_bgzf(text, 1)
    z6, z6_ms = zlib_bgzf(text, 6)
    print(json.dumps({
        "corpus": "vcf: synth_text(20000, 2504) GT:GQ", **info, "text_bytes": len(text), "bgzf_bytes": len(gz),
        "ratio": len(text) / len(gz), "ratio_zlib1_bgzf": len(text) / len(z1), "ratio_zlib6_bgzf": len(text) / len(z6),
        "size_vs_zlib1": len(gz) / len(z1), "deflate_kernel_ms": krn,
        "deflate_kernel_GBps": len(text) / krn / 1e6 if krn else "not measured", "fm_bgzf_deflate_ms": call_ms,
        "host_zlib1_bgzf_ms": z1_ms, "host_zlib6_bgzf_ms": z6_ms, "host_threads": threads, "round_trip_ok": ok}),
        flush=True)


if __name__ == "__main__":
    main()
