"""Haplotype LD pruning benchmark (fm_haplotype_ld_prune): the cohort of tools/bench_ld.py -- 2504 diploid samples
(n = 5008) x 10^6 sites from fm_synth_fill with 26 populations (sigma = 0.05), device-resident u8, min_maf 0.01,
max_missing 0.02, at 0 % and 1 % missing cells -- with linkage added on the device: in runs of 8 sites, each site
takes every cell from the run's first site with probability 0.85, so that pruning at r^2 0.2 removes a real share of
the sites.  Prints JSON lines: the card; per missing rate M, pairs, linked pairs, the retained count and fraction, the
median stage times of fm_ld_prune_info over warmed calls, the whole prune call next to the fm_haplotype_ld call at the
same window (the two alternate in one run), the prune -> PCA chain next to PCA on every kept site, and a parity line
against the numpy restatement on a 20,000-site slice."""
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

RUN, COPY_P = 8, 0.85


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, pl, sm, smax = [x.strip() for x in q.split(",")]
    return dict(card=name, power_limit=pl, sm_clock_sampled=sm, sm_clock_max=smax)


def add_linkage(torch, rows, seed, chunk=65536):
    """rows [V, cells] u8 on the device: site v takes each cell of site v - v % RUN with probability COPY_P."""
    g = torch.Generator(device=rows.device).manual_seed(seed)
    V = rows.shape[0]
    for a in range(0, V, chunk):
        b = min(V, a + chunk)
        head = torch.arange(a, b, device=rows.device) // RUN * RUN
        mix = torch.rand((b - a, rows.shape[1]), generator=g, device=rows.device) < COPY_P
        rows[a:b] = torch.where(mix, rows[head], rows[a:b])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sites", type=int, default=1_000_000)
    ap.add_argument("--samples", type=int, default=2504)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--window", type=int, default=100)
    ap.add_argument("--threshold", type=float, default=0.2)
    ap.add_argument("--slice", type=int, default=20_000)
    args = ap.parse_args()
    import torch

    from ferromic_b200 import _lib
    from ferromic_b200.api import _matrix_ld, _matrix_ld_prune, _matrix_pca
    from tests import ld_prune_reference as lp
    from tests import pca_reference as pr
    L = _lib.lib()
    V, S, w, thr = args.sites, args.samples, args.window, args.threshold
    print(json.dumps(dict(kind="card", **card())), flush=True)
    pops = (np.arange(S) % 26).astype(np.uint16)
    total = V * S * 2
    d_data = torch.empty(total, dtype=torch.uint8, device="cuda:0")
    d_miss = torch.empty((total + 63) // 64, dtype=torch.int64, device="cuda:0")
    pos = np.arange(V, dtype=np.int64) * 10
    haps = [(s, h) for s in range(S) for h in (0, 1)]
    kw = dict(min_maf=0.01, max_missing=0.02)
    for missing in (0.0, 0.01):
        _lib.check(L.fm_synth_fill(d_data.data_ptr(), d_miss.data_ptr(), V, S, 2, 0, 2026, pops.ctypes.data, 0.05,
                                   missing))
        add_linkage(torch, d_data.view(V, S * 2), 7 + int(missing * 100))
        torch.cuda.synchronize()
        h = C.c_void_p()
        _lib.check(L.fm_matrix_create_device(d_data.data_ptr(), d_miss.data_ptr() if missing else None, V, S, 2, 1,
                                             pos.ctypes.data, C.byref(h)))
        m = type("M", (), {"handle": h, "V": V, "P": 2})

        def prune():
            return _matrix_ld_prune(m, haps, thr, w, **kw)

        def ld():
            return _matrix_ld(m, haps, w, **kw)
        prune()
        ld()  # warm-up of both shapes
        p_runs, l_runs = [], []
        for _ in range(args.repeats):  # the two calls alternate
            t0 = time.perf_counter()
            r = prune()
            p_runs.append((r["info"], (time.perf_counter() - t0) * 1e3))
            t0 = time.perf_counter()
            q = ld()
            l_runs.append((q["info"], (time.perf_counter() - t0) * 1e3))
            del q
        clk = card()
        info = p_runs[0][0]
        med = lambda runs, f: float(np.median([f(i) for i, _ in runs]))  # noqa: E731
        M, R = int(info.n_sites), int(info.n_retained)
        print(json.dumps(dict(
            kind="prune_timing", missing=missing, n=int(info.n_haplotypes), sites=V, M=M, window=w, r2_threshold=thr,
            called_plane=int(info.called_plane), pairs=int(info.pairs), linked_pairs=int(info.linked_pairs),
            n_retained=R, retained_fraction=R / M, repeats=args.repeats,
            stats_ms=med(p_runs, lambda i: i.stats_ms), planes_ms=med(p_runs, lambda i: i.planes_ms),
            band_ms=med(p_runs, lambda i: i.band_ms), scan_ms=med(p_runs, lambda i: i.scan_ms),
            prune_call_ms=med(p_runs, lambda i: i.total_ms), prune_call_wall_ms=float(np.median([t for _, t in p_runs])),
            bit_row_bytes=M * max(1, (min(w, M - 1) + 31) // 32) * 4,
            ld_call_ms=med(l_runs, lambda i: i.total_ms), ld_call_wall_ms=float(np.median([t for _, t in l_runs])),
            ld_band_ms=med(l_runs, lambda i: i.band_ms), ld_copy_ms=med(l_runs, lambda i: i.copy_ms),
            sm_clock_sampled=clk["sm_clock_sampled"])), flush=True)

        # prune -> PCA chain next to PCA on every kept site
        _matrix_pca(m, haps, 10, **kw)
        chain, full = [], []
        for _ in range(max(2, args.repeats // 2)):
            t0 = time.perf_counter()
            sites = prune()["retained"]
            pc = _matrix_pca(m, haps, 10, sites=sites, **kw)
            chain.append((time.perf_counter() - t0) * 1e3)
            t0 = time.perf_counter()
            pa = _matrix_pca(m, haps, 10, **kw)
            full.append((time.perf_counter() - t0) * 1e3)
        print(json.dumps(dict(
            kind="chain", missing=missing, pca_sites_pruned=int(pc["info"].n_sites), pca_sites_all=int(pa["info"].n_sites),
            prune_then_pca_wall_ms=float(np.median(chain)), pca_all_kept_wall_ms=float(np.median(full)),
            evr_pruned=pc["explained_variance_ratio"][:4].tolist(), evr_all=pa["explained_variance_ratio"][:4].tolist(),
            sm_clock_sampled=card()["sm_clock_sampled"])), flush=True)

        # parity on a slice of the same matrix
        sl = min(args.slice, V)
        raw = d_data.view(V, S * 2)[:sl].cpu().numpy()
        called = np.ones_like(raw, dtype=bool)
        if missing:
            bits = np.unpackbits(d_miss.cpu().numpy().view(np.uint8), bitorder="little")[: sl * S * 2]
            called = bits.reshape(sl, S * 2) == 0
        got = _matrix_ld_prune(m, haps, thr, w, region=(int(pos[0]), int(pos[sl - 1])), **kw)
        ref = lp.ld_prune(pr.rows_from_arrays(raw, called), sl, lp.lr.offsets(haps, S, 2), w, pos[:sl], thr,
                          chunk=4096, **kw)
        gi = got["info"]
        print(json.dumps(dict(
            kind="parity", missing=missing, slice_sites=sl, M=ref["M"], window=w,
            kept_equal=bool(np.array_equal(got["kept"], ref["kept"])),
            retained_equal=bool(np.array_equal(got["retained"], ref["retained"])),
            pairs_equal=int(gi.pairs) == ref["pairs"], linked_pairs_equal=int(gi.linked_pairs) == ref["linked_pairs"],
            n_retained=int(gi.n_retained))), flush=True)
        L.fm_matrix_release(h)


if __name__ == "__main__":
    main()
