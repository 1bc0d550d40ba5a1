#!/usr/bin/env python
"""Device-resident timing of the other BASELINE.json configs (bench.py measures configs[1]):
  cfg1  100k sites x 5008 haplotypes, one group, no bitmap: S + pi + theta (summary pass)
  cfg3  Hudson FST/Dxy between two populations (fused two-group pass), sites per GPU of the 8-GPU shard
  cfg4  W&C over 26 subpopulations (27 count passes once, then K4 on cached counts)
  cfg5  biobank shard: 200k haplotypes, 1% missing, two populations, 100 kb windows
One JSON line per config on stdout.  usage: bench_configs.py [cfg1 cfg3 cfg4 cfg5] [--scale F]"""
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import bench  # noqa: E402
from ferromic_b200 import _lib  # noqa: E402
from tools.wc_timing import membership  # noqa: E402

PEAK = 6553.3
try:
    PEAK = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
except Exception:
    pass


def group_handle(L, m, haps):
    idx = np.asarray([h[0] for h in haps], dtype=np.uint64)
    side = np.asarray([h[1] for h in haps], dtype=np.uint8)
    h = C.c_void_p()
    _lib.check(L.fm_group_create(m, idx.ctypes.data, side.ctypes.data, len(haps), C.byref(h)))
    return h


def matrix(L, V, S, seed, dev, missing):
    pos = bench.make_positions(V, seed)
    d_data, d_bitmap = bench.gen_device(V, S, seed, dev, missing_rate=missing)
    torch.cuda.synchronize()
    m = C.c_void_p()
    _lib.check(L.fm_matrix_create_device(d_data.data_ptr(), d_bitmap.data_ptr() if missing > 0 else None, V, S, 2, 1,
                                         pos.ctypes.data, C.byref(m)))
    return m, pos, (d_data, d_bitmap)


def line(name, V, H, ms, bytes_per_launch, extra=None):
    out = {"config": name, "sites": V, "haplotypes": H, "ms_per_pass": ms, "genotypes_per_s": V * H / (ms * 1e-3),
           "algorithmic_GBps": bytes_per_launch / (ms * 1e-3) / 1e9,
           "frac_of_measured_peak": bytes_per_launch / (ms * 1e-3) / 1e9 / PEAK}
    out.update(extra or {})
    print(json.dumps(out), flush=True)


def cfg1(L, dev, scale):
    V, S = 100_000, 2504
    m, pos, keep = matrix(L, V, S, 102_504, dev, 0.0)
    g = group_handle(L, m, [(s, k) for s in range(S) for k in (0, 1)])
    arr = (C.c_void_p * 1)(g.value)
    res = _lib.BenchResult()
    for it in (50, 200):
        _lib.check(L.fm_bench_diversity(arr, 1, 0, None, 0, it, None, C.byref(res), None, None))
    line("cfg1 summary (S, pi, theta), one group, no bitmap", V, 2 * S, res.plane_ms_avg, res.group_bytes[0],
         {"step_ms": res.step_ms_avg, "note": "latency-sized: 62.6 MB per pass, resident in the 126 MB L2"})
    L.fm_group_release(g)
    L.fm_matrix_release(m)


def cfg3(L, dev, scale):
    V, S = int(1_250_000 * scale), 2504
    m, pos, keep = matrix(L, V, S, 10_002_504, dev, 0.0)
    g1 = group_handle(L, m, [(s, k) for s in range(S // 2) for k in (0, 1)])
    g2 = group_handle(L, m, [(s, k) for s in range(S // 2, S) for k in (0, 1)])
    res = _lib.BenchResult()
    for it in (5, 30):
        _lib.check(L.fm_bench_hudson(g1, g2, it, C.byref(res)))
    line("cfg3 Hudson per-site fused two-group kernel (NG=2; kept for reference, no longer the product path)", V, 2 * S, res.plane_ms_avg,
         res.plane_bytes_per_step, {"step_ms": res.step_ms_avg})
    # the product path of fm_hudson_pair's first call: ONE sequential launch over both groups' planes
    # (counts + summary scalars cached) + the light Hudson kernel on the counts; device time by events
    o = _lib.HudsonOutcome()
    n = C.c_size_t()
    Lr = int(pos[-1] - pos[0] + 1)
    best = None
    tim = _lib.Timings()
    for rep in range(3):
        for g in (g1, g2):
            L.fm_group_release(g)
        g1 = group_handle(L, m, [(s, k) for s in range(S // 2) for k in (0, 1)])
        g2 = group_handle(L, m, [(s, k) for s in range(S // 2, S) for k in (0, 1)])
        L.fm_timings_reset()
        t0 = time.perf_counter()
        _lib.check(L.fm_hudson_pair(g1, g2, Lr, Lr, 0, 0, 0, 0, S, S, C.byref(o), None, C.byref(n)))
        dt = time.perf_counter() - t0
        L.fm_timings_get(C.byref(tim))
        if best is None or tim.stats_ms < best[0]:
            best = (tim.stats_ms, dt * 1e3, tim.kernel_launches)
    plane_bytes = res.plane_bytes_per_step
    print(json.dumps({"config": "cfg3 fm_hudson_pair first call (sequential count launch over both groups + light "
                                "Hudson kernel + reductions)", "device_ms": best[0], "wall_ms": best[1],
                      "kernel_launches": best[2], "genotypes_per_s": V * 2 * S / (best[0] * 1e-3),
                      "plane_GBps_incl_light_kernels": plane_bytes / (best[0] * 1e-3) / 1e9,
                      "fst": o.fst, "d_xy": o.d_xy}), flush=True)
    for g in (g1, g2):
        L.fm_group_release(g)
    L.fm_matrix_release(m)


def cfg4(L, dev, scale):
    V, S = int(1_000_000 * scale), 2504
    m, pos, keep = matrix(L, V, S, 10_002_504, dev, 0.01)
    left, right = membership(S)
    L.fm_timings_reset()
    ph = C.c_void_p()
    t0 = time.perf_counter()
    _lib.check(L.fm_partition_create(m, left.ctypes.data, right.ctypes.data, S, 26, C.byref(ph)))
    t_part = time.perf_counter() - t0
    w = np.array([int(pos[0]), int(pos[-1])], dtype=np.int64)
    NP = 325
    nv = np.zeros(1, dtype=np.uint64); osz = np.zeros(1, dtype=np.uint64)
    oa = np.zeros(1); ob = np.zeros(1); pa = np.zeros(NP); pb = np.zeros(NP); pn = np.zeros(NP, dtype=np.uint64)
    times = []
    tim = _lib.Timings()
    for i in range(4):
        L.fm_timings_reset()
        t0 = time.perf_counter()
        _lib.check(L.fm_wc_window_sums(ph, w.ctypes.data, 1, nv.ctypes.data, oa.ctypes.data, ob.ctypes.data,
                                       osz.ctypes.data, pa.ctypes.data, pb.ctypes.data, pn.ctypes.data))
        times.append((time.perf_counter() - t0) * 1e3)
        L.fm_timings_get(C.byref(tim))
    line("cfg4 W&C 26 populations / 325 pairs, region sums (K4 on cached counts)", V, 2 * S, min(times[1:]),
         V * 27 * 8, {"first_call_ms_incl_27_count_passes": times[0], "partition_repack_wall_ms": t_part * 1e3,
                      "bound": "fp64 pipe (divisions), not HBM", "k4_stats_ms": tim.stats_ms})
    L.fm_partition_release(ph)
    L.fm_matrix_release(m)


def cfg5(L, dev, scale):
    V, S = int(65_536 * scale), 100_000
    m, pos, keep = matrix(L, V, S, 2_100_000, dev, 0.01)
    g1 = group_handle(L, m, [(s, k) for s in range(S // 2) for k in (0, 1)])
    g2 = group_handle(L, m, [(s, k) for s in range(S // 2, S) for k in (0, 1)])
    res = _lib.BenchResult()
    for it in (3, 10):
        _lib.check(L.fm_bench_hudson(g1, g2, it, C.byref(res)))
    line("cfg5 biobank shard, 200k haplotypes, 1% missing, fused two-group pass (column-chunked rows)", V, 2 * S,
         res.plane_ms_avg, res.plane_bytes_per_step, {"step_ms": res.step_ms_avg})
    edges = np.arange(int(pos[0]), int(pos[-1]) + 1, 100_000, dtype=np.int64)
    ww = np.stack([edges, edges + 99_999], axis=1).reshape(-1).copy()
    n = len(edges)
    f = [np.zeros(n) for _ in range(5)]
    sk = np.zeros(n, dtype=np.uint64)
    _lib.check(L.fm_hudson_window_sums(g1, g2, ww.ctypes.data, n, f[0].ctypes.data, f[1].ctypes.data,
                                       f[2].ctypes.data, sk.ctypes.data, f[3].ctypes.data, f[4].ctypes.data))
    t0 = time.perf_counter()
    _lib.check(L.fm_hudson_window_sums(g1, g2, ww.ctypes.data, n, f[0].ctypes.data, f[1].ctypes.data,
                                       f[2].ctypes.data, sk.ctypes.data, f[3].ctypes.data, f[4].ctypes.data))
    print(json.dumps({"config": "cfg5 100 kb window sums from cached counts", "windows": n,
                      "wall_ms": (time.perf_counter() - t0) * 1e3}), flush=True)
    for g in (g1, g2):
        L.fm_group_release(g)
    L.fm_matrix_release(m)


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    scale = 1.0
    if "--scale" in sys.argv:
        scale = float(sys.argv[sys.argv.index("--scale") + 1])
        args = [a for a in args if a != str(scale) and a != sys.argv[sys.argv.index("--scale") + 1]]
    todo = args or ["cfg1", "cfg3", "cfg4", "cfg5"]
    dev = torch.device("cuda", 0)
    L = _lib.lib()
    _lib.check(L.fm_set_device(0))
    for name in todo:
        globals()[name](L, dev, scale)
        torch.cuda.empty_cache()
        L.fm_trim_pool()


if __name__ == "__main__":
    main()
