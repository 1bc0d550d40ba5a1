"""Haplotype frequency benchmark (fm_haplotype_frequencies): 2504 diploid samples (n = 5008) x 10^6 sites from
fm_synth_fill (26 populations, sigma = 0.05), device-resident u8, at 0 % and 1 % missing cells, with haplotype
structure added on the device: in each block of 500 sites every haplotype copies one of 40 founder haplotypes (founder
0 with probability 0.5, the others evenly), then each cell flips with probability 0.001.  Without it every window of
the synthetic cohort would hold n distinct haplotypes and the exact run check would never see a run longer than one.
Sites are kept with max_missing 0.02 at both rates (at 1 % missing no site is fully called by 5008 haplotypes), so at
1 % missing most haplotypes have a missing cell in a window and are left out of it.  Prints JSON lines: the card; per
missing rate and run (count windows of 200 kept sites every 50, of 1000 kept sites, and 1000 position windows) the
median stage times of fm_hapfreq_info over warmed calls, hashed key words/s, sorted entries/s, the whole call, and
the mean N and K over the windows; and a parity line against the numpy restatement (tests/hapfreq_reference.py) on a
20,000-site slice with the restatement's time extrapolated to the full size."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BLOCK, FOUNDERS, TOP_P, FLIP_P = 500, 40, 0.5, 0.001


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, pl, sm, smax = [x.strip() for x in q.split(",")]
    return dict(card=name, power_limit=pl, sm_clock_sampled=sm, sm_clock_max=smax)


def add_haplotypes(torch, rows, seed):
    """rows [V, n] u8 on the device: per block of BLOCK sites each column copies a founder column, then cells flip."""
    g = torch.Generator(device=rows.device).manual_seed(seed)
    V, n = rows.shape
    p = torch.full((FOUNDERS,), (1 - TOP_P) / (FOUNDERS - 1), device=rows.device)
    p[0] = TOP_P
    for a in range(0, V, BLOCK):
        b = min(V, a + BLOCK)
        pick = torch.multinomial(p, n, replacement=True, generator=g)
        blk = rows[a:b, :FOUNDERS][:, pick]
        flip = (torch.rand((b - a, n), generator=g, device=rows.device) < FLIP_P).to(torch.uint8)
        rows[a:b] = blk ^ flip


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sites", type=int, default=1_000_000)
    ap.add_argument("--samples", type=int, default=2504)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--slice", type=int, default=20_000)
    args = ap.parse_args()
    import torch

    from ferromic_b200 import _lib
    from ferromic_b200.api import _matrix_hapfreq
    from tests import hapfreq_reference as hr
    L = _lib.lib()
    V, S = args.sites, args.samples
    n = 2 * S
    print(json.dumps(dict(kind="card", **card())), flush=True)
    pops = (np.arange(S) % 26).astype(np.uint16)
    total = V * n
    d_data = torch.empty(total, dtype=torch.uint8, device="cuda:0")
    d_miss = torch.empty((total + 63) // 64, dtype=torch.int64, device="cuda:0")
    pos = np.arange(V, dtype=np.int64) * 10
    haps = [(s, h) for s in range(S) for h in (0, 1)]
    edges = np.linspace(0, int(pos[-1]) + 1, 1001).astype(np.int64)
    windows = np.stack([edges[:-1], edges[1:] - 1], axis=1)
    mm = 0.02
    for missing in (0.0, 0.01):
        _lib.check(L.fm_synth_fill(d_data.data_ptr(), d_miss.data_ptr(), V, S, 2, 0, 2026, pops.ctypes.data, 0.05,
                                   missing))
        add_haplotypes(torch, d_data.view(V, n), 11 + int(missing * 100))
        torch.cuda.synchronize()
        h = C.c_void_p()
        _lib.check(L.fm_matrix_create_device(d_data.data_ptr(), d_miss.data_ptr() if missing else None, V, S, 2, 1,
                                             pos.ctypes.data, C.byref(h)))
        m = type("M", (), {"handle": h, "V": V, "P": 2})
        runs = (("size200_step50", dict(size=200, step=50)), ("size1000", dict(size=1000)),
                ("windows1000", dict(windows=windows)))
        for name, kw in runs:
            call = lambda: _matrix_hapfreq(m, haps, max_missing=mm, **kw)  # noqa: E731
            call()  # warm-up of the shape
            rs = []
            for _ in range(args.repeats):
                t0 = time.perf_counter()
                r = call()
                rs.append((r, (time.perf_counter() - t0) * 1e3))
            r0 = rs[0][0]
            info = r0["info"]
            med = lambda f: float(np.median([f(r["info"]) for r, _ in rs]))  # noqa: E731
            hash_ms, sort_ms = med(lambda i: i.hash_ms), med(lambda i: i.sort_ms)
            key_words = int(np.sum((r0["window_sites"].astype(np.int64) + 63) // 64)) * n
            entries = int(info.n_windows) * n
            print(json.dumps(dict(
                kind="hapfreq_timing", run=name, missing=missing, n=n, sites=V, max_missing=mm,
                n_kept=int(info.n_sites), windows=int(info.n_windows), called_plane=int(info.called_plane),
                collisions=int(info.collisions), mean_n_used=float(np.mean(r0["n_used"])),
                mean_distinct=float(np.mean(r0["distinct"])), mean_h12=float(np.nanmean(r0["h12"])),
                repeats=args.repeats, stats_ms=med(lambda i: i.stats_ms), planes_ms=med(lambda i: i.planes_ms),
                hash_ms=hash_ms, sort_ms=sort_ms, count_ms=med(lambda i: i.count_ms),
                total_ms=med(lambda i: i.total_ms), wall_ms=float(np.median([t for _, t in rs])),
                key_words=key_words, key_words_per_s=key_words / hash_ms * 1e3, sorted_entries=entries,
                sorted_entries_per_s=entries / sort_ms * 1e3, sm_clock_sampled=card()["sm_clock_sampled"])), flush=True)

        # parity on a slice of the same matrix, and the restatement's time
        sl = min(args.slice, V)
        raw = d_data.view(V, n)[:sl].cpu().numpy()
        called = np.ones_like(raw, dtype=bool)
        if missing:
            bits = np.unpackbits(d_miss.cpu().numpy().view(np.uint8), bitorder="little")[: sl * n]
            called = bits.reshape(sl, n) == 0
        region = (int(pos[0]), int(pos[sl - 1]))
        got = _matrix_hapfreq(m, haps, 200, 50, region=region, max_missing=mm, counts=True)
        t0 = time.perf_counter()
        ref = hr.haplotype_frequencies(raw, called, np.arange(n), 0.0, mm, size=200, step=50)
        t_ref = time.perf_counter() - t0
        same = lambda k: bool(np.array_equal(got[k].astype(np.int64), ref[k]))  # noqa: E731
        bits_same = all(np.array_equal(got[k].view(np.uint64), ref[k].view(np.uint64))
                        for k in ("h1", "h12", "h123", "h2_h1", "diversity"))
        co = got["count_offsets"]
        counts_same = all(got["counts"][co[w]:co[w + 1]].tolist() == c.tolist() for w, c in enumerate(ref["counts"]))
        print(json.dumps(dict(
            kind="parity", run="size200_step50", missing=missing, slice_sites=sl,
            kept_equal=got["kept"].tolist() == ref["kept"].tolist(), windows=len(ref["windows"]),
            n_used_equal=same("n_used"), distinct_equal=same("distinct"), sum_sq_equal=same("sum_sq"),
            top_counts_equal=bool(np.array_equal(got["top_counts"].astype(np.int64), ref["top"])),
            class_sizes_equal=counts_same, statistics_bit_identical=bits_same,
            restatement_s=t_ref, restatement_full_size_s_extrapolated=t_ref * V / sl)), flush=True)
        L.fm_matrix_release(h)


if __name__ == "__main__":
    main()
