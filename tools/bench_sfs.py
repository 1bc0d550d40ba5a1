"""Site frequency spectrum benchmark (fm_site_frequency_spectrum / fm_joint_site_frequency_spectrum) on the cohort of
tools/bench_ld.py: 2504 diploid samples (n = 5008) x 10^6 sites from fm_synth_fill with 26 populations (sigma = 0.05),
device-resident u8, at 0 % and 1 % missing cells.  Prints JSON lines: the card; per missing rate and run (1-D at m = n
or at a projection that keeps about 99 % of the sites, over one window and over 1000 windows; m = 20; the joint
spectrum of the two halves of the samples at (2504, 2504) or a projection keeping about 99 %), the median stage times
of the info struct over warmed calls, the counting stage's bytes and bytes/s next to the site-statistics stage of
fm_haplotype_ld (fm_k_hap_site_stats) on the same set in the same run, and a parity line against the numpy
restatement on a 20,000-site slice with the restatement's time extrapolated to the full size."""
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


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, pl, sm, smax = [x.strip() for x in q.split(",")]
    return dict(card=name, power_limit=pl, sm_clock_sampled=sm, sm_clock_max=smax)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sites", type=int, default=1_000_000)
    ap.add_argument("--samples", type=int, default=2504)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--slice", type=int, default=20_000)
    args = ap.parse_args()
    import torch

    from ferromic_b200 import _lib
    from ferromic_b200.api import _matrix_joint_sfs, _matrix_ld, _matrix_sfs
    from tests import sfs_reference as sr
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
    half1 = [(s, h) for s in range(S // 2) for h in (0, 1)]
    half2 = [(s, h) for s in range(S // 2, S) for h in (0, 1)]
    edges = np.linspace(0, int(pos[-1]) + 1, 1001).astype(np.int64)
    windows = np.stack([edges[:-1], edges[1:] - 1], axis=1)

    def median(fn, repeats):
        fn()  # warm-up of the shape
        runs = []
        for _ in range(repeats):
            t0 = time.perf_counter()
            r = fn()
            runs.append((r, (time.perf_counter() - t0) * 1e3))
        return runs

    for missing in (0.0, 0.01):
        _lib.check(L.fm_synth_fill(d_data.data_ptr(), d_miss.data_ptr(), V, S, 2, 0, 2026, pops.ctypes.data, 0.05,
                                   missing))
        torch.cuda.synchronize()
        h = C.c_void_p()
        _lib.check(L.fm_matrix_create_device(d_data.data_ptr(), d_miss.data_ptr() if missing else None, V, S, 2, 1,
                                             pos.ctypes.data, C.byref(h)))
        m = type("M", (), {"handle": h, "V": V, "P": 2})
        sl = min(args.slice, V)
        raw = d_data.view(V, n)[:sl].cpu().numpy()
        called = np.ones_like(raw, dtype=bool)
        if missing:
            bits = np.unpackbits(d_miss.cpu().numpy().view(np.uint8), bitorder="little")[: sl * n]
            called = bits.reshape(sl, n) == 0
        # projections that keep about 99 % of the sites (the 1st percentile of called on the slice)
        m_all = n if not missing else int(np.percentile(called.sum(axis=1), 1))
        m_half = S if not missing else int(min(np.percentile(called[:, :S].sum(axis=1), 0.5),
                                               np.percentile(called[:, S:].sum(axis=1), 0.5)))
        count_bytes = V * n + (V * n // 8 if missing else 0)
        ld_stats = [r["info"].stats_ms for r, _ in median(lambda: _matrix_ld(m, haps, 1), args.repeats)]
        stats_ms = float(np.median(ld_stats))
        runs = (("1d", m_all, None), ("1d_1000_windows", m_all, windows), ("1d", 20, None),
                ("joint", (m_half, m_half), None))
        for name, proj, win in runs:
            if name == "joint":
                rs = median(lambda: _matrix_joint_sfs(m, half1, half2, proj), args.repeats)
            else:
                rs = median(lambda: _matrix_sfs(m, haps, proj, windows=win), args.repeats)
            info = rs[0][0]["info"]
            med = lambda f: float(np.median([f(r["info"]) for r, _ in rs]))  # noqa: E731
            cm = med(lambda i: i.counts_ms)
            out = dict(kind="sfs_timing", run=name, missing=missing, n=n, sites=V, projection=proj,
                       windows=0 if win is None else len(win), n_sites=int(info.n_sites),
                       projected_out=int(info.projected_out), kept_fraction=int(info.n_sites) / V,
                       repeats=args.repeats, counts_ms=cm, spectrum_ms=med(lambda i: i.spectrum_ms),
                       total_ms=med(lambda i: i.total_ms), wall_ms=float(np.median([t for _, t in rs])),
                       count_bytes=count_bytes, count_GBps=count_bytes / cm / 1e6,
                       hap_site_stats_ms=stats_ms, hap_site_stats_GBps=count_bytes / stats_ms / 1e6,
                       sm_clock_sampled=card()["sm_clock_sampled"])
            if name == "joint":
                out.update(incidences=int(info.incidences), passes=int(info.passes))
            else:
                out.update(tajimas_d=float(rs[0][0]["tajimas_d"][0]))
            print(json.dumps(out), flush=True)

        # parity on a slice of the same matrix, and the restatement's time
        region = (int(pos[0]), int(pos[sl - 1]))
        for name, proj in (("1d", m_all), ("1d", 20), ("joint", (m_half, m_half))):
            t0 = time.perf_counter()
            if name == "joint":
                ref = sr.joint_sfs(raw, called, np.arange(S), np.arange(S, n), proj[0], proj[1])
                t_ref = time.perf_counter() - t0
                got = _matrix_joint_sfs(m, half1, half2, proj, region)
            else:
                ref = sr.sfs(raw, called, np.arange(n), proj)
                t_ref = time.perf_counter() - t0
                got = _matrix_sfs(m, haps, proj, region)
            xi_ref, xi = ref["spectrum"], got["spectrum"]
            ok = bool(np.all(np.abs(xi - xi_ref) <= 1e-9 * np.abs(xi_ref) + 1e-290))
            print(json.dumps(dict(
                kind="parity", run=name, missing=missing, projection=proj, slice_sites=sl,
                spectrum_within_1e9=ok, n_sites_equal=int(got["info"].n_sites) == ref["n_sites"],
                projected_out_equal=int(got["info"].projected_out) == ref["projected_out"],
                restatement_s=t_ref, restatement_full_size_s_extrapolated=t_ref * V / sl)), flush=True)
        L.fm_matrix_release(h)


if __name__ == "__main__":
    main()
