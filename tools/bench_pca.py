"""Haplotype PCA benchmark (fm_haplotype_pca): 2504 diploid samples x 10^6 sites from fm_synth_fill with 26
populations (sigma = 0.05), device-resident u8, at 0 % and 1 % missing cells; k = 10, oversampling 10, q = 4.
Prints JSON lines: the card, then per missing rate the per-stage device times over warmed repeats, the FMA count
of a product (n M l) and the rate reached; a parity line against the numpy restatement on a site slice, and the
restatement's host time on that slice scaled linearly to the whole size (labelled extrapolated)."""
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
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--slice", type=int, default=50_000)
    args = ap.parse_args()
    import torch

    from ferromic_b200 import _lib
    from ferromic_b200.api import _matrix_pca
    from tests import pca_reference as pr
    L = _lib.lib()
    V, S = args.sites, args.samples
    k, os_, q = 10, 10, 4
    print(json.dumps(dict(kind="card", **card())), flush=True)
    pops = (np.arange(S) % 26).astype(np.uint16)
    total = V * S * 2
    d_data = torch.empty(total, dtype=torch.uint8, device="cuda:0")
    d_miss = torch.empty((total + 63) // 64, dtype=torch.int64, device="cuda:0")
    pos = np.arange(V, dtype=np.int64) * 10
    haps = [(s, h) for s in range(S) for h in (0, 1)]
    for missing in (0.0, 0.01):
        _lib.check(L.fm_synth_fill(d_data.data_ptr(), d_miss.data_ptr(), V, S, 2, 0, 2026, pops.ctypes.data, 0.05,
                                   missing))
        h = C.c_void_p()
        _lib.check(L.fm_matrix_create_device(d_data.data_ptr(), d_miss.data_ptr() if missing else None, V, S, 2, 1,
                                             pos.ctypes.data, C.byref(h)))
        m = type("M", (), {"handle": h, "V": V, "P": 2})
        kw = dict(max_missing=0.02, min_maf=0.01, oversampling=os_, power_iterations=q)
        _matrix_pca(m, haps, k, **kw)  # warm-up
        runs = []
        for _ in range(args.repeats):
            t0 = time.perf_counter()
            r = _matrix_pca(m, haps, k, **kw)
            wall = (time.perf_counter() - t0) * 1e3
            runs.append((r["info"], wall))
        clk = card()
        info = runs[0][0]
        n, M, l = int(info.n_haplotypes), int(info.n_sites), int(info.rank)
        fma = n * M * l

        def med(f):
            return float(np.median([f(i) for i, _ in runs]))
        zt = med(lambda i: i.zt_q_ms / i.zt_q_launches)
        zr = med(lambda i: i.z_r_ms / i.z_r_launches)
        line = dict(kind="timing", missing=missing, n=n, sites=V, M=M, l=l, k=k, q=q, repeats=args.repeats,
                    site_stats_ms=med(lambda i: i.stats_ms), transpose_ms=med(lambda i: i.planes_ms),
                    zt_q_ms_per_product=zt, z_r_ms_per_product=zr, gram_ms=med(lambda i: i.gram_ms),
                    orth_eigen_host_ms=med(lambda i: i.small_ms), call_ms=med(lambda i: i.total_ms),
                    call_wall_ms=float(np.median([w for _, w in runs])), fma_per_product=fma,
                    zt_q_tfma_s=fma / zt / 1e9, z_r_tfma_s=fma / zr / 1e9, sm_clock_sampled=clk["sm_clock_sampled"],
                    singular_values=[float(x) for x in r["singular_values"]])
        print(json.dumps(line), flush=True)
        # parity and host time on a slice of the same matrix
        sl = min(args.slice, V)
        raw = d_data.view(V, S * 2)[:sl].cpu().numpy()
        called = np.ones_like(raw, dtype=bool)
        if missing:
            bits = np.unpackbits(d_miss.cpu().numpy().view(np.uint8), bitorder="little")[: sl * S * 2]
            called = bits.reshape(sl, S * 2) == 0
        got = _matrix_pca(m, haps, k, (0, int(pos[sl - 1])), **kw)
        t0 = time.perf_counter()
        ref = pr.haplotype_pca(pr.rows_from_arrays(raw, called), sl, pr.offsets(haps, S, 2), k, chunk=8192, **kw)
        host_s = time.perf_counter() - t0
        scale = np.max(np.abs(ref["scores"]), axis=0)
        print(json.dumps(dict(
            kind="parity", missing=missing, slice_sites=sl, M=ref["M"],
            kept_equal=bool(np.array_equal(got["kept"], ref["kept"])), T_equal=got["total_variance"] == ref["T"],
            sigma_max_rel=float(np.max(np.abs(got["singular_values"] / ref["singular_values"] - 1))),
            scores_max_rel=float(np.max(np.abs(got["scores"] - ref["scores"]) / scale)),
            restatement_host_s=host_s, restatement_host_s_extrapolated_to_sites=host_s * V / sl,
            extrapolated=True, device_call_ms=line["call_ms"])), flush=True)
        L.fm_matrix_release(h)


if __name__ == "__main__":
    main()
