"""Times fm_pairwise_differences (calculate_pairwise_differences, stats.rs:4106-4231) on a 1000 Genomes-sized
cohort: 2504 samples x 1e6 biallelic diploid sites generated on the device (fm_synth_fill), at 0 % and 1 % missing
cells.  Prints one JSON line per cohort and a closing line with the card, its power limit and the SASS counts.

Per cohort: CUDA-event times of the transpose (zero fill + fm_k_sample_planes) and of the pair kernel
(fm_k_pairwise_counts) over warmed repeats, the end-to-end call, pair-sites/s of the pair kernel, the oracle's
threaded rows form timed on a slice and extrapolated to the full size by pair-sites, and a parity check of 64
pairs (diagonal tiles, the last partial tile, off-diagonal tiles) against the oracle over all sites."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # the card name still identifies the measurement
        out = f"unavailable ({type(e).__name__})"
    return name, out


def sass_counts(so):
    """POPC / LOP3 per pass of the inner loop body (one site word of the thread's 4 x 8 pairs)."""
    out = {}
    for hc in ("1", "0"):
        fn = f"_ZN2fm20fm_k_pairwise_countsILb{hc}EEEvPKjNS_8PwLayoutEjjjPjS4_"
        try:
            sass = subprocess.run(["cuobjdump", "-sass", "-fun", fn, so], capture_output=True, text=True,
                                  timeout=120).stdout
        except FileNotFoundError:
            sass = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", "-fun", fn, so], capture_output=True,
                                  text=True, timeout=120).stdout
        popc = sum(1 for l in sass.splitlines() if " POPC " in l)
        out["with_missing" if hc == "1" else "no_missing"] = {
            "popc_per_32_pair_sites": popc / 32.0, "popc_in_kernel": popc,
            "lop3_in_kernel": sum(1 for l in sass.splitlines() if " LOP3" in l)}
    return out


def gather_gt(d_data, d_miss, V, S, cols, v_lo=0, v_hi=None, step=100_000):
    """u8 genotypes of the listed samples with the 0xFF sentinel at missing cells, sites [v_lo, v_hi)."""
    import torch
    v_hi = V if v_hi is None else v_hi
    cidx = torch.tensor(cols, device="cuda:0")
    parts = []
    for a in range(v_lo, v_hi, step):
        b = min(v_hi, a + step)
        g = d_data.view(V, S, 2)[a:b][:, cidx, :]
        if d_miss is not None:
            e = ((torch.arange(a, b, device="cuda:0")[:, None, None] * S + cidx[None, :, None]) * 2 +
                 torch.arange(2, device="cuda:0")[None, None, :])
            miss = ((d_miss[e >> 6] >> (e & 63)) & 1).bool()
            g = torch.where(miss, torch.full_like(g, 0xFF), g)
        parts.append(g.cpu().numpy())
    return np.concatenate(parts, axis=0)


def run_cohort(V, S, missing, reps, warmup, slice_samples, slice_sites, threads):
    import torch
    from ferromic_b200 import _lib
    from oracle import pyoracle as orc
    from tests import pairwise_oracle as po
    L = _lib.lib()
    total = V * S * 2
    d_data = torch.empty(total, dtype=torch.uint8, device="cuda:0")
    d_miss = torch.empty((total + 63) // 64, dtype=torch.int64, device="cuda:0") if missing > 0 else None
    _lib.check(L.fm_set_device(0))
    _lib.check(L.fm_synth_fill(d_data.data_ptr(), d_miss.data_ptr() if d_miss is not None else None, V, S, 2, 0,
                               20261020, None, 0.05, missing))
    pos = np.arange(V, dtype=np.int64) * 3
    m = C.c_void_p()
    _lib.check(L.fm_matrix_create_device(d_data.data_ptr(), d_miss.data_ptr() if d_miss is not None else None, V, S, 2,
                                         1, pos.ctypes.data, C.byref(m)))
    n_pairs = S * (S - 1) // 2
    diff, comp = np.zeros(n_pairs, np.uint32), np.zeros(n_pairs, np.uint32)
    n_out = C.c_size_t()
    tim = _lib.Timings()
    tr, pk, e2e = [], [], []
    for r in range(warmup + reps):
        _lib.check(L.fm_timings_reset())
        t0 = time.perf_counter()
        _lib.check(L.fm_pairwise_differences(m, S, diff.ctypes.data, comp.ctypes.data, None, None, 0, C.byref(n_out)))
        t1 = time.perf_counter()
        _lib.check(L.fm_timings_get(C.byref(tim)))
        if r >= warmup:
            tr.append(tim.repack_ms)
            pk.append(tim.stats_ms)
            e2e.append((t1 - t0) * 1e3)
    pair_sites = n_pairs * V
    # parity: 64 pairs from every tile class against the oracle over all sites
    rng = np.random.default_rng(64)
    pairs = [(0, 1), (S - 2, S - 1), (0, S - 1), (63, 64), ((S - 1) // 64 * 64, S - 1)]
    while len(pairs) < 64:
        i, j = sorted(int(x) for x in rng.choice(S, size=2, replace=False))
        if len(pairs) % 3 == 0:
            b = i // 64
            i, j = b * 64 + int(rng.integers(0, 32)), b * 64 + int(rng.integers(32, 64))
            if j >= S:
                continue
        pairs.append((i, j))
    cols = sorted({c for p in pairs for c in p})
    where = {c: k for k, c in enumerate(cols)}
    gt = gather_gt(d_data, d_miss, V, S, cols)
    bad = []
    for i, j in pairs:
        od, oc, _, _ = po.pairwise_differences(orc.Variants(pos, np.ascontiguousarray(gt[:, [where[i], where[j]], :])), 2)
        k = i * (2 * S - i - 1) // 2 + j - i - 1
        if (int(diff[k]), int(comp[k])) != (int(od[0]), int(oc[0])):
            bad.append([i, j, int(diff[k]), int(od[0]), int(comp[k]), int(oc[0])])
    # CPU baseline: the oracle's threaded rows form on a slice, extrapolated by pair-sites
    sl = gather_gt(d_data, d_miss, V, S, list(range(slice_samples)), 0, slice_sites)
    vs = orc.Variants(pos[:slice_sites], np.ascontiguousarray(sl))
    t0 = time.perf_counter()
    sd, sc, _, _ = po.pairwise_differences(vs, slice_samples, threads=threads)
    cpu_s = time.perf_counter() - t0
    slice_pair_sites = slice_samples * (slice_samples - 1) // 2 * slice_sites
    L.fm_matrix_release(m)
    del d_data, d_miss
    torch.cuda.empty_cache()
    _lib.check(L.fm_trim_pool())
    pk_med = float(np.median(pk))
    cpu_full_s = cpu_s * pair_sites / slice_pair_sites
    return {
        "cohort": f"{S} samples x {V} sites, diploid biallelic, {missing:.0%} missing cells",
        "n_pairs": n_pairs, "pair_sites": pair_sites,
        "transpose_ms": {"median": float(np.median(tr)), "min": float(np.min(tr)), "max": float(np.max(tr))},
        "pair_kernel_ms": {"median": pk_med, "min": float(np.min(pk)), "max": float(np.max(pk))},
        "call_ms_median": float(np.median(e2e)),
        "pair_sites_per_s": pair_sites / (pk_med * 1e-3),
        "repeats": reps, "warmup": warmup,
        "cpu_oracle_threads": {"threads": threads, "slice": f"{slice_samples} samples x {slice_sites} sites",
                               "slice_s": cpu_s, "full_size_s": cpu_full_s, "extrapolated": True},
        "speedup_vs_cpu_extrapolated": cpu_full_s / (float(np.median(e2e)) * 1e-3),
        "parity": {"pairs": len(pairs), "sites": V, "mismatches": bad, "ok": not bad},
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--sites", type=int, default=1_000_000)
    ap.add_argument("--samples", type=int, default=2504)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--slice-samples", type=int, default=512)
    ap.add_argument("--slice-sites", type=int, default=20_000)
    ap.add_argument("--threads", type=int, default=os.cpu_count() or 1)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_pairwise.py needs a CUDA device (no CPU fallback)")
    import ferromic_b200 as fm
    ok = True
    for missing in (0.0, 0.01):
        r = run_cohort(a.sites, a.samples, missing, a.reps, a.warmup, min(a.slice_samples, a.samples),
                       min(a.slice_sites, a.sites), a.threads)
        ok = ok and r["parity"]["ok"]
        print(json.dumps(r), flush=True)
    name, power = card()
    print(json.dumps({"card": name, "power_limit_and_max_sm_clock": power, "sass": sass_counts(fm.SO_PATH),
                      "parity_ok": ok}), flush=True)
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
