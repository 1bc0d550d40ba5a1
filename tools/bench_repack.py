#!/usr/bin/env python
"""K1 (u8 rows -> group bitplanes) on a device-resident matrix: the two orientation groups of
BASELINE configs[1] (every haplotype belongs to one of them) repacked by ONE launch through the
streaming-ingest-free path (fm_group_create per group = one launch each) and timed by the library's
own events (fm_timings.repack_ms).
usage: bench_repack.py [sites]"""
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import bench  # noqa: E402
from ferromic_b200 import _lib  # noqa: E402
from tools.bench_configs import group_handle, matrix  # noqa: E402


def main():
    V = int(sys.argv[1]) if len(sys.argv) > 1 else 250_000
    S = 2504
    dev = torch.device("cuda:0")
    L = _lib.lib()
    out = {"what": "K1 repack, two orientation groups covering all 5008 haplotypes", "sites": V}
    for missing in (0.01, 0.0):
        m, pos, keep = matrix(L, V, S, 1_002_504, dev, missing)
        rng = np.random.default_rng(3)
        orient = rng.integers(0, 2, size=S)
        haps1 = [(s, int(orient[s])) for s in range(S)] + [(s, k) for s in range(0, S, 3) for k in (0, 1)]
        set1 = set(haps1)
        haps2 = [(s, k) for s in range(S) for k in (0, 1) if (s, k) not in set1]
        tim = _lib.Timings()
        best = None
        best1 = None
        for rep in range(4):
            L.fm_timings_reset()
            g1 = group_handle(L, m, haps1)
            g2 = group_handle(L, m, haps2)
            L.fm_timings_get(C.byref(tim))
            L.fm_group_release(g1)
            L.fm_group_release(g2)
            if rep and (best is None or tim.repack_ms < best):
                best = tim.repack_ms
            # both groups by ONE launch (fm_groups_create)
            idx = np.asarray([h[0] for h in haps1 + haps2], dtype=np.uint64)
            side = np.asarray([h[1] for h in haps1 + haps2], dtype=np.uint8)
            sizes = (C.c_size_t * 2)(len(haps1), len(haps2))
            outg = (C.c_void_p * 2)()
            L.fm_timings_reset()
            _lib.check(L.fm_groups_create(m, idx.ctypes.data, side.ctypes.data, sizes, 2, outg))
            L.fm_timings_get(C.byref(tim))
            for h in outg:
                L.fm_group_release(C.c_void_p(h))
            if rep and (best1 is None or tim.repack_ms < best1):
                best1 = tim.repack_ms
        u8 = V * S * 2 * (1.125 if missing else 1.0)
        key = "bitmap" if missing else "no_missing"
        out[key] = {"repack_ms_two_launches": best, "u8_GBps_per_launch": 2 * u8 / (best * 1e-3) / 1e9,
                    "group_sizes": [len(set1), len(haps2)], "repack_ms_one_launch": best1,
                    "u8_GBps_one_launch": u8 / (best1 * 1e-3) / 1e9}
        L.fm_matrix_release(m)
        del keep
    print(json.dumps(out))


if __name__ == "__main__":
    main()
