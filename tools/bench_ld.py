"""Haplotype LD benchmark (fm_haplotype_ld): 2504 diploid samples (n = 5008) x 10^6 sites from fm_synth_fill with
26 populations (sigma = 0.05), device-resident u8, min_maf 0.01, max_missing 0.02, at 0 % and 1 % missing cells:
window 100 over every site, and an inversion-heatmap case (the first 20,000 sites, full upper triangle with D').
Prints JSON lines: the card; per workload M, pairs, pair-words (useful and as tiled), the stage times of fm_ld_info
(median of warmed calls), the whole call, the POPC of fm_k_ld_band from its SASS and the POPC rate per SM and clock
at the sampled clock; a parity line against the numpy restatement on a 20,000-site slice, with the restatement's
host time scaled linearly to the whole workload (labelled extrapolated)."""
import argparse
import ctypes as C
import json
import os
import re
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SMS = 148  # B200


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, pl, sm, smax = [x.strip() for x in q.split(",")]
    return dict(card=name, power_limit=pl, sm_clock_sampled=sm, sm_clock_max=smax)


def band_popc(so):
    """POPC instructions of each float fm_k_ld_band instantiation (all in the main loop, unrolled over 2 haplotype words)."""
    sass = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", so], capture_output=True, text=True).stdout
    out = {}
    for part in re.split(r"\n\s*Function : ", sass):
        name = part.split("\n", 1)[0].strip()
        if name.startswith("_ZN2fm12fm_k_ld_bandILb") and "ELb0EEE" in name:  # the float forms, not the bit forms
            out["called_plane" if "ILb1E" in name else "no_called_plane"] = len(re.findall(r"\bPOPC\b", part))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sites", type=int, default=1_000_000)
    ap.add_argument("--samples", type=int, default=2504)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--heatmap-sites", type=int, default=20_000)
    ap.add_argument("--slice", type=int, default=20_000)
    args = ap.parse_args()
    import torch

    from ferromic_b200 import _lib
    from ferromic_b200.api import _matrix_ld
    from tests import ld_reference as lr
    L = _lib.lib()
    V, S = args.sites, args.samples
    print(json.dumps(dict(kind="card", **card(), band_popc_in_sass=band_popc(_lib.SO_PATH))), flush=True)
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
        h = C.c_void_p()
        _lib.check(L.fm_matrix_create_device(d_data.data_ptr(), d_miss.data_ptr() if missing else None, V, S, 2, 1,
                                             pos.ctypes.data, C.byref(h)))
        m = type("M", (), {"handle": h, "V": V, "P": 2})
        hm_region = (int(pos[0]), int(pos[min(V, args.heatmap_sites) - 1]))
        hm_M = int(_matrix_ld(m, haps, 1, region=hm_region, **kw)["info"].n_sites)
        for case, window, region, dprime in (("window100", 100, None, False),
                                             ("heatmap", max(1, hm_M - 1), hm_region, True)):
            _matrix_ld(m, haps, window, region=region, dprime=dprime, **kw)  # warm-up
            runs = []
            for _ in range(args.repeats):
                t0 = time.perf_counter()
                r = _matrix_ld(m, haps, window, region=region, dprime=dprime, **kw)
                runs.append((r["info"], (time.perf_counter() - t0) * 1e3))
            clk = card()
            info = runs[0][0]
            n, M, hc = int(info.n_haplotypes), int(info.n_sites), int(info.called_plane)
            n_words, n_blk = (n + 31) // 32, (M + 63) // 64
            chunks = (n_words + 7) // 8
            tpr = (window + 63) // 64 + 1
            tiles_live = sum(min(tpr, n_blk - bi) for bi in range(n_blk))  # tiles past the last block only write NaN
            tiled_pair_words = tiles_live * 64 * 64 * chunks * 8
            popc = tiled_pair_words * (4 if hc else 1)

            def med(f):
                return float(np.median([f(i) for i, _ in runs]))
            band_ms = med(lambda i: i.band_ms)
            mhz = float(clk["sm_clock_sampled"].split()[0])
            print(json.dumps(dict(
                kind="timing", case=case, missing=missing, n=n, sites=V, M=M, window=window, dprime=dprime,
                called_plane=hc, pairs=int(info.pairs), useful_pair_words=int(info.pairs) * n_words,
                tiled_pair_words=tiled_pair_words, slabs=int(info.slabs), repeats=args.repeats,
                stats_ms=med(lambda i: i.stats_ms), planes_ms=med(lambda i: i.planes_ms), band_ms=band_ms,
                copy_ms=med(lambda i: i.copy_ms), call_ms=med(lambda i: i.total_ms),
                call_wall_ms=float(np.median([w for _, w in runs])),
                output_bytes=M * window * 4 * (2 if dprime else 1), band_popc=popc,
                band_popc_per_sm_clk=popc / (band_ms * 1e-3) / SMS / (mhz * 1e6),
                pairwise_popc_per_sm_clk_design=10, sm_clock_sampled=clk["sm_clock_sampled"])), flush=True)
        # parity and host time on a slice of the same matrix
        sl = min(args.slice, V)
        raw = d_data.view(V, S * 2)[:sl].cpu().numpy()
        called = np.ones_like(raw, dtype=bool)
        if missing:
            bits = np.unpackbits(d_miss.cpu().numpy().view(np.uint8), bitorder="little")[: sl * S * 2]
            called = bits.reshape(sl, S * 2) == 0
        got = _matrix_ld(m, haps, 100, region=(int(pos[0]), int(pos[sl - 1])), dprime=True, **kw)
        t0 = time.perf_counter()
        ref = lr.haplotype_ld(lr.rows_from_arrays(raw, called), sl, lr.offsets(haps, S, 2), 100, pos[:sl], chunk=4096,
                              **kw)
        host_s = time.perf_counter() - t0
        M = ref["M"]
        print(json.dumps(dict(
            kind="parity", missing=missing, slice_sites=sl, M=M, window=100,
            kept_equal=bool(np.array_equal(got["kept"], ref["kept"])),
            r2_bit_equal_cells=int((got["r2"].view(np.uint32) == ref["r2"].view(np.uint32)).sum()),
            dprime_bit_equal_cells=int((got["dprime"].view(np.uint32) == ref["dprime"].view(np.uint32)).sum()),
            cells=M * 100, restatement_host_s=host_s,
            restatement_host_s_extrapolated_to_sites=host_s * V / sl, extrapolated=True)), flush=True)
        L.fm_matrix_release(h)


if __name__ == "__main__":
    main()
