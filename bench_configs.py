"""bench_configs.py -- the other BASELINE.json configs inside the driver-run line of bench.py (VERDICT r1 items 2
and 9): config 1 as a batch of 64 regions in one launch, config 3 (Hudson FST + Dxy, 10M sites), config 4
(Weir & Cockerham, 26 populations) and one GPU's shard of config 5 (200k haplotypes), each with its time, its
UNPADDED algorithmic bytes and the fraction of the measured HBM peak; plus the `strong` block: config 3's 10M
sites split over the N ranks, ONE un-pipelined sharded Hudson call per step (sweep + fold + NVLink exchange).

Cohorts come from the library's counter-based generator (fm_synth_fill), so any slice can be re-evaluated on
the CPU: every config checks 10^3..10^4-site slices against the oracle (checker only) before it is timed."""
from __future__ import annotations

import ctypes as C
import os
import time

import numpy as np

POP_SIZES = [96, 61, 86, 93, 99, 103, 105, 94, 99, 99, 91, 103, 113, 107, 102, 104, 99, 99, 85, 64, 85, 96, 104,
             102, 107, 108]  # 26 subpopulations, 1000G-like, sum 2504


class Cohort:
    """u8 matrix (+ bitmap) filled on the device by fm_synth_fill, wrapped in an fm_matrix handle."""

    def __init__(self, L, _lib, device, V, S, seed, pop_of_sample, sigma, missing_rate, first_variant=0, pos=None):
        import torch
        self.L, self._lib, self.V, self.S = L, _lib, V, S
        self.seed, self.sigma, self.missing_rate, self.first = seed, sigma, missing_rate, first_variant
        self.pop = np.ascontiguousarray(pop_of_sample, dtype=np.uint16)
        total = V * S * 2
        self.d_data = torch.empty(max(total, 16), dtype=torch.uint8, device=device)
        self.d_miss = torch.empty((total + 63) // 64 + 2, dtype=torch.int64, device=device) if missing_rate > 0 else None
        _lib.check(L.fm_synth_fill(self.d_data.data_ptr(), self.d_miss.data_ptr() if self.d_miss is not None else None,
                                   V, S, 2, first_variant, seed, self.pop.ctypes.data, sigma, missing_rate))
        if pos is None:
            pos = np.cumsum(np.random.default_rng(seed).integers(1, 50, size=V, dtype=np.int64))
        self.pos = np.ascontiguousarray(pos, dtype=np.int64)
        self.m = C.c_void_p()
        _lib.check(L.fm_matrix_create_device(self.d_data.data_ptr(),
                                             self.d_miss.data_ptr() if self.d_miss is not None else None, V, S, 2, 1,
                                             self.pos.ctypes.data, C.byref(self.m)))

    def groups(self, hap_lists):
        idx = np.concatenate([np.asarray([h[0] for h in hs], dtype=np.uint64) for hs in hap_lists])
        side = np.concatenate([np.asarray([h[1] for h in hs], dtype=np.uint8) for hs in hap_lists])
        sizes = (C.c_size_t * len(hap_lists))(*[len(hs) for hs in hap_lists])
        out = (C.c_void_p * len(hap_lists))()
        self._lib.check(self.L.fm_groups_create(self.m, idx.ctypes.data, side.ctypes.data, sizes, len(hap_lists), out))
        return [C.c_void_p(h) for h in out]

    def slice_rows(self, lo, hi):
        from tests.synth import synth_rows
        return synth_rows(self.seed, self.first + lo, self.first + hi, self.S, 2, self.pop, self.sigma, self.missing_rate)

    def close(self):
        import torch
        self.L.fm_matrix_release(self.m)
        self.d_data = self.d_miss = None
        torch.cuda.empty_cache()


def halves(S):
    return ([(s, k) for s in range(S // 2) for k in (0, 1)], [(s, k) for s in range(S // 2, S) for k in (0, 1)])


def release(L, handles):
    for h in handles:
        L.fm_group_release(h)


def stats_ms(L, _lib):
    t = _lib.Timings()
    L.fm_timings_get(C.byref(t))
    return t.stats_ms


def entry(name, what, ms, alg_bytes, peak, geno, extra=None):
    gbps = alg_bytes / (ms * 1e-3) / 1e9 if ms > 0 else None
    e = {"config": name, "what": what, "ms": ms, "algorithmic_bytes": alg_bytes, "GBps": gbps,
         "frac": gbps / peak if gbps else None, "genotypes_per_s": geno / (ms * 1e-3) if ms > 0 else None}
    if extra:
        e.update(extra)
    return e


def hudson_window(L, _lib, g1, g2, win):
    f = [np.zeros(1) for _ in range(5)]
    sk = np.zeros(1, dtype=np.uint64)
    w = np.ascontiguousarray(win, dtype=np.int64)
    _lib.check(L.fm_hudson_window_sums(g1, g2, w.ctypes.data, 1, f[0].ctypes.data, f[1].ctypes.data, f[2].ctypes.data,
                                       sk.ctypes.data, f[3].ctypes.data, f[4].ctypes.data))
    return np.array([x[0] for x in f]), int(sk[0])


def check_hudson_slices(L, _lib, co, g1, g2, h1, h2, n_slices, width, seed):
    """Window sums of random site slices against the oracle on CPU-regenerated genotypes (ints exact, f64 1e-9)."""
    from oracle import pyoracle as orc
    rng = np.random.default_rng(seed)
    for _ in range(n_slices):
        lo = int(rng.integers(0, max(1, co.V - width)))
        hi = min(co.V, lo + width)
        g = co.slice_rows(lo, hi)
        _, d = orc.from_numpy(g, co.pos[lo:hi])
        s1, s2 = orc.build_summary(d, h1), orc.build_summary(d, h2)
        Ls = int(co.pos[hi - 1] - co.pos[lo] + 1)
        rc, ref, _ = orc.hudson_pair(orc.Pop(h1, None, co.S, Ls, summary=s1), orc.Pop(h2, None, co.S, Ls, summary=s2))
        got, sk = hudson_window(L, _lib, g1, g2, [int(co.pos[lo]), int(co.pos[hi - 1])])
        fst = got[0] / got[1]
        if rc != 0 or abs(fst - ref["fst"]) > 1e-9 * abs(ref["fst"]):
            raise RuntimeError("parity: Hudson FST of a slice differs from the oracle")
        if abs(got[2] / (Ls - sk) - ref["d_xy"]) > 1e-9 * abs(ref["d_xy"]):
            raise RuntimeError("parity: Dxy of a slice differs from the oracle")
        for grp, s in ((g1, s1), (g2, s2)):
            w = np.array([int(co.pos[lo]), int(co.pos[hi - 1])], dtype=np.int64)
            nv, seg, unc = (np.zeros(1, dtype=np.uint64) for _ in range(3))
            pis = np.zeros(1)
            _lib.check(L.fm_group_window_sums(grp, w.ctypes.data, 1, nv.ctypes.data, seg.ctypes.data, pis.ctypes.data,
                                              unc.ctypes.data))
            if int(nv[0]) != hi - lo or int(seg[0]) != int(s.seg) or int(unc[0]) != int((s.called < 2).sum()):
                raise RuntimeError("parity: integer window counts differ from the oracle")
    return n_slices * width


# ----------------------------------------------------------------------------------------------- config 1 x 64
def cfg1_batched(L, _lib, device, peak, scale, n_regions=64):
    from oracle import pyoracle as orc
    V, S = max(64, int(100_000 * scale)), 2504
    H = 2 * S
    haps = [(s, k) for s in range(S) for k in (0, 1)]
    cohorts = [Cohort(L, _lib, device, V, S, 102_504 + r, np.zeros(S, dtype=np.uint16), 0.0, 0.0) for r in range(2)]

    def make_groups():
        # 64 region matrices: generated two at a time would need 32 GB of u8; the planes are what the timed call
        # streams, so the regions cycle over two generated cohorts (distinct plane buffers, 4 GB in total > L2)
        return [cohorts[r % 2].groups([haps])[0] for r in range(n_regions)]

    groups = make_groups()
    arr = (C.c_void_p * n_regions)(*[g.value for g in groups])
    seg = np.zeros(n_regions, dtype=np.uint64)
    pis = np.zeros(n_regions)
    L.fm_timings_reset()
    _lib.check(L.fm_groups_summary_batch(arr, n_regions, seg.ctypes.data, pis.ctypes.data, None))
    # parity: the first two regions against the oracle over all their sites' counts (slice of 5,000 sites)
    for r in range(2):
        lo, hi = 0, min(V, 5000)
        g = cohorts[r].slice_rows(lo, hi)
        _, d = orc.from_numpy(g, cohorts[r].pos[lo:hi])
        ref = orc.build_summary(d, haps)
        w = np.array([int(cohorts[r].pos[lo]), int(cohorts[r].pos[hi - 1])], dtype=np.int64)
        nv, sg, un = (np.zeros(1, dtype=np.uint64) for _ in range(3))
        ps = np.zeros(1)
        _lib.check(L.fm_group_window_sums(groups[r], w.ctypes.data, 1, nv.ctypes.data, sg.ctypes.data, ps.ctypes.data,
                                          un.ctypes.data))
        if int(sg[0]) != int(ref.seg) or abs(ps[0] - ref.pi_sum) > 1e-9 * abs(ref.pi_sum):
            raise RuntimeError("parity: config 1 region summary differs from the oracle")
    if not (seg[0] == seg[2] and pis[0] == pis[2] and seg[1] == seg[3]):
        raise RuntimeError("parity: identical regions of the batch gave different summaries")
    release(L, groups)
    times = []
    for _ in range(3):
        groups = make_groups()
        arr = (C.c_void_p * n_regions)(*[g.value for g in groups])
        L.fm_timings_reset()
        t0 = time.perf_counter()
        _lib.check(L.fm_groups_summary_batch(arr, n_regions, seg.ctypes.data, pis.ctypes.data, None))
        wall = (time.perf_counter() - t0) * 1e3
        times.append((stats_ms(L, _lib), wall))
        release(L, groups)
    # the same regions one call at a time (the reference CLI's shape)
    groups = make_groups()
    t0 = time.perf_counter()
    for g in groups:
        s_, p_, u_ = C.c_uint64(), C.c_double(), C.c_uint64()
        _lib.check(L.fm_group_summary(g, None, None, C.byref(s_), C.byref(p_), C.byref(u_)))
    serial_ms = (time.perf_counter() - t0) * 1e3
    release(L, groups)
    for c in cohorts:
        c.close()
    dev_ms, wall_ms = min(times)
    alg = n_regions * V * H / 8.0  # no missing data: one allele bit per genotype
    return entry("configs[0] x %d regions" % n_regions,
                 "segregating sites + pi + theta inputs (dense summary) of %d regions of %d sites x %d haplotypes in ONE "
                 "launch (fm_groups_summary_batch -> fm_k_plane_pass_seq), no missing data" % (n_regions, V, H),
                 dev_ms, alg, peak, n_regions * V * H,
                 {"wall_ms": wall_ms, "one_call_per_region_wall_ms": serial_ms, "regions": n_regions,
                  "timing": "CUDA events around the pass + fold inside the library (fm_timings.stats_ms)"})


# ----------------------------------------------------------------------------------------------- config 3
def cfg3_hudson(L, _lib, device, peak, scale):
    V, S = max(8192, int(10_000_000 * scale)), 2504
    H = 2 * S
    pop = (np.arange(S) >= S // 2).astype(np.uint16)
    co = Cohort(L, _lib, device, V, S, 10_002_504, pop, 0.05, 0.01)
    h1, h2 = halves(S)
    Lr = int(co.pos[-1] - co.pos[0] + 1)
    times = []
    out = _lib.HudsonOutcome()
    n = C.c_size_t()
    for it in range(3):
        g1, g2 = co.groups([h1, h2])
        L.fm_timings_reset()
        t0 = time.perf_counter()
        _lib.check(L.fm_hudson_pair(g1, g2, Lr, Lr, _lib.FM_HUDSON_SUMMARIES, 0, 0, 0, len(h1), len(h2), C.byref(out),
                                    None, C.byref(n)))
        times.append((stats_ms(L, _lib), (time.perf_counter() - t0) * 1e3))
        if it < 2:
            release(L, (g1, g2))
    first = (out.fst, out.d_xy)
    t0 = time.perf_counter()
    _lib.check(L.fm_hudson_pair(g1, g2, Lr, Lr, _lib.FM_HUDSON_SUMMARIES, 0, 0, 0, len(h1), len(h2), C.byref(out), None,
                                C.byref(n)))
    cached_ms = (time.perf_counter() - t0) * 1e3
    if (out.fst, out.d_xy) != first:
        raise RuntimeError("parity: cached Hudson call differs from the fused first call")
    checked = check_hudson_slices(L, _lib, co, g1, g2, h1, h2, 2, min(V, 4000), 3)
    release(L, (g1, g2))
    co.close()
    dev_ms, wall_ms = min(times)
    alg = V * H * 2 / 8.0  # allele + called bit of both populations; outputs are per-region scalars
    return entry("configs[2]", "Hudson FST + Dxy + pi of two populations, %d sites x %d haplotypes, first call on fresh "
                 "groups: ONE fused sweep (counts of both groups cached + Hudson partials), 1 GPU" % (V, H),
                 dev_ms, alg, peak, V * H,
                 {"wall_ms": wall_ms, "cached_counts_call_wall_ms": cached_ms, "fst": out.fst, "d_xy": out.d_xy,
                  "parity_slice_sites": checked, "extra_bytes_written": V * 16 + (V // 32) * 88,
                  "timing": "CUDA events around pass + folds inside the library (fm_timings.stats_ms)"})


# ----------------------------------------------------------------------------------------------- config 4
def cfg4_wc(L, _lib, device, peak, scale):
    from oracle import pyoracle as orc
    V, S = max(8192, int(10_000_000 * scale)), 2504
    H = 2 * S
    left = np.full(S, 0xFFFF, dtype=np.uint16)
    s = 0
    for p, k in enumerate(POP_SIZES):
        left[s:s + k] = p
        s += k
    co = Cohort(L, _lib, device, V, S, 10_002_504, left, 0.08, 0.0)  # no missing data: dense == sparse semantics
    ph = C.c_void_p()
    L.fm_timings_reset()
    t0 = time.perf_counter()
    _lib.check(L.fm_partition_create(co.m, left.ctypes.data, left.ctypes.data, S, 26, C.byref(ph)))
    part_wall = (time.perf_counter() - t0) * 1e3
    tim = _lib.Timings()
    L.fm_timings_get(C.byref(tim))
    NP = 325
    w = np.array([int(co.pos[0]), int(co.pos[-1])], dtype=np.int64)

    def wc(win):
        win = np.ascontiguousarray(win, dtype=np.int64)
        nv, osz = np.zeros(1, dtype=np.uint64), np.zeros(1, dtype=np.uint64)
        oa, ob = np.zeros(1), np.zeros(1)
        pa, pb, pn = np.zeros(NP), np.zeros(NP), np.zeros(NP, dtype=np.uint64)
        _lib.check(L.fm_wc_window_sums(ph, win.ctypes.data, 1, nv.ctypes.data, oa.ctypes.data, ob.ctypes.data,
                                       osz.ctypes.data, pa.ctypes.data, pb.ctypes.data, pn.ctypes.data))
        return nv, oa, ob, osz, pa, pb, pn

    times = []
    for _ in range(3):
        L.fm_timings_reset()
        t0 = time.perf_counter()
        whole = wc(w)
        times.append((stats_ms(L, _lib), (time.perf_counter() - t0) * 1e3))
    rng = np.random.default_rng(4)
    lo = int(rng.integers(0, max(1, V - 1000)))
    hi = min(V, lo + 1000)
    g = co.slice_rows(lo, hi)
    vs, _d = orc.from_numpy(g, co.pos[lo:hi])
    region = (int(co.pos[lo]), int(co.pos[hi - 1]))
    ref = orc.wc_fst(vs, left, left, 26, region, want_pairs=False)
    got = wc(np.array(region))
    ok = int(got[0][0]) == ref["n_sites"] and int(got[3][0]) == ref["overall"]["sites"]
    ok = ok and abs(got[1][0] - ref["overall"]["sum_a"]) <= 1e-9 * abs(ref["overall"]["sum_a"])
    for k in range(NP):
        e = ref["pairs"][k]
        ok = ok and int(got[6][k]) == e["sites"] and abs(got[4][k] - e["sum_a"]) <= 1e-9 * abs(e["sum_a"]) + 1e-300 \
            and abs(got[5][k] - e["sum_b"]) <= 1e-9 * abs(e["sum_b"]) + 1e-300
    if not ok:
        raise RuntimeError("parity: W&C sums of a slice differ from the oracle")
    L.fm_partition_release(ph)
    co.close()
    dev_ms, wall_ms = min(times)
    alg = V * 27 * 8.0  # K4 reads the cached (alt, called) counts of 26 populations + the rest: 8 B per site and group
    pair_sites = V * NP
    return entry("configs[3]", "Weir & Cockerham: overall + 325 pairwise (a, b) sums over %d sites x 26 populations from "
                 "cached counts (K4 pairs + overall + fold); FP64-pipe bound, not HBM" % V, dev_ms, alg, peak, V * H,
                 {"wall_ms": wall_ms, "bound": "fp64", "pair_sites_per_s": pair_sites / (dev_ms * 1e-3),
                  "partition_create_wall_ms": part_wall, "partition_count_kernel_ms": tim.repack_ms,
                  "overall_fst": float(whole[1][0] / (whole[1][0] + whole[2][0])), "parity_slice_sites": hi - lo,
                  "timing": "CUDA events around K4 + fold inside the library (fm_timings.stats_ms)"})


# ----------------------------------------------------------------------------------------------- config 5 shard
def cfg5_shard(L, _lib, device, peak, scale):
    V, S = max(256, int(250_000 * scale)), 100_000
    H = 2 * S
    pop = (np.arange(S) >= S // 2).astype(np.uint16)
    co = Cohort(L, _lib, device, V, S, 2_100_000, pop, 0.05, 0.01)
    h1, h2 = halves(S)
    times = []
    for it in range(2):
        g1, g2 = co.groups([h1, h2])
        arr = (C.c_void_p * 2)(g1.value, g2.value)
        L.fm_timings_reset()
        t0 = time.perf_counter()
        _lib.check(L.fm_groups_summary_batch(arr, 2, None, None, None))
        times.append((stats_ms(L, _lib), (time.perf_counter() - t0) * 1e3))
        if it == 0:
            release(L, (g1, g2))
    edges = np.arange(int(co.pos[0]), int(co.pos[-1]) + 1, 100_000, dtype=np.int64)
    windows = np.ascontiguousarray(np.stack([edges, edges + 99_999], axis=1))
    nw = len(windows)
    f = [np.zeros(nw) for _ in range(5)]
    sk = np.zeros(nw, dtype=np.uint64)
    t0 = time.perf_counter()
    _lib.check(L.fm_hudson_window_sums(g1, g2, windows.ctypes.data, nw, f[0].ctypes.data, f[1].ctypes.data,
                                       f[2].ctypes.data, sk.ctypes.data, f[3].ctypes.data, f[4].ctypes.data))
    win_ms = (time.perf_counter() - t0) * 1e3
    checked = check_hudson_slices(L, _lib, co, g1, g2, h1, h2, 1, min(V, 150), 6)
    release(L, (g1, g2))
    co.close()
    dev_ms, wall_ms = min(times)
    alg = V * H * 2 / 8.0
    return entry("configs[4] shard (1 of 8 GPUs)", "dense summaries (counts, S, sum pi) of two 100,000-haplotype populations "
                 "over %d sites with 1 %% missing data (column-chunked plane pass), then %d windows of 100 kb of Hudson "
                 "component sums from the cached counts" % (V, nw), dev_ms, alg, peak, V * H,
                 {"wall_ms": wall_ms, "windows": nw, "window_sums_wall_ms": win_ms, "parity_slice_sites": checked,
                  "timing": "CUDA events around the passes + folds inside the library (fm_timings.stats_ms)"})


# ----------------------------------------------------------------------------------------------- strong scaling
def strong_cfg3(L, _lib, args, rank, world, device, dist, peak, scale):
    """Config 3's sites split over the ranks (site-range shards aligned to 8192); per step ONE sharded Hudson
    call on fresh groups: sweep of the shard + fold + NVLink exchange + outcome on every rank, nothing pipelined."""
    import torch
    V_total, S = max(8192 * world, int(10_000_000 * scale)), 2504
    H = 2 * S
    per = ((V_total + world - 1) // world + 8191) // 8192 * 8192
    lo, hi = min(V_total, rank * per), min(V_total, (rank + 1) * per)
    pos_all = np.cumsum(np.random.default_rng(10_002_504).integers(1, 50, size=V_total, dtype=np.int64))
    pop = (np.arange(S) >= S // 2).astype(np.uint16)
    co = Cohort(L, _lib, device, hi - lo, S, 10_002_504, pop, 0.05, 0.01, first_variant=lo, pos=pos_all[lo:hi])
    h1, h2 = halves(S)
    Lr = int(pos_all[-1] - pos_all[0] + 1)
    comm = None
    if world > 1:
        comm = C.c_void_p()
        _lib.check(L.fm_comm_create(rank, world, C.byref(comm)))
        hb = (C.c_uint8 * 64)()
        _lib.check(L.fm_comm_export(comm, hb))
        mine = torch.tensor(list(hb), dtype=torch.uint8, device=device)
        allh = torch.empty(world * 64, dtype=torch.uint8, device=device)
        dist.all_gather_into_tensor(allh, mine)
        handles = np.ascontiguousarray(allh.cpu().numpy())
        _lib.check(L.fm_comm_connect(comm, handles.ctypes.data))
        dist.barrier()
    out, sums = _lib.HudsonOutcome(), _lib.HudsonSums()
    steps, warm = max(3, min(args.steps, 10)), 2
    wall, dev = [], []
    for it in range(warm + steps):
        g1, g2 = co.groups([h1, h2])  # fresh groups: nothing cached (K1 is outside the timed step)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        L.fm_timings_reset()
        t0 = time.perf_counter()
        _lib.check(L.fm_hudson_pair_sharded(g1, g2, Lr, len(h1), len(h2), comm, C.byref(out), C.byref(sums)))
        dt = (time.perf_counter() - t0) * 1e3
        if it >= warm:
            wall.append(dt)
            dev.append(stats_ms(L, _lib))
        release(L, (g1, g2))
    # every rank must hold the same bits; and they must equal the rank-ordered sum of the ranks' local totals
    local_out, local = _lib.HudsonOutcome(), _lib.HudsonSums()
    g1, g2 = co.groups([h1, h2])
    _lib.check(L.fm_hudson_pair_sharded(g1, g2, Lr, len(h1), len(h2), None, C.byref(local_out), C.byref(local)))
    checked = check_hudson_slices(L, _lib, co, g1, g2, h1, h2, 1, min(co.V, 2000), 100 + rank) if co.V else 0
    release(L, (g1, g2))
    agree = True
    if world > 1:
        vec = torch.tensor([local.num, local.den, local.dxy, local.pi1, local.pi2, float(local.dxy_uncallable),
                            float(local.unc1), float(local.unc2)], dtype=torch.float64, device=device)
        allv = [torch.empty_like(vec) for _ in range(world)]
        dist.all_gather(allv, vec)
        tot = np.zeros(8)
        for r in range(world):
            tot = tot + allv[r].cpu().numpy()
        got = np.array([sums.num, sums.den, sums.dxy, sums.pi1, sums.pi2, float(sums.dxy_uncallable), float(sums.unc1),
                        float(sums.unc2)])
        agree = bool(np.array_equal(got, tot))
        mine = torch.tensor([out.fst, out.d_xy, out.pi_pop1, out.pi_pop2], dtype=torch.float64, device=device)
        allo = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allo, mine)
        agree = agree and all(bool(torch.equal(allo[0], o)) for o in allo)
        if not agree:
            raise RuntimeError(f"parity: sharded Hudson totals differ across ranks / from the rank-ordered sum (rank {rank})")
    t = torch.tensor([float(np.mean(wall)), float(np.mean(dev))], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.barrier()
        L.fm_comm_destroy(comm)
    co.close()
    wall_ms, dev_ms = float(t[0].item()), float(t[1].item())
    alg = V_total * H * 2 / 8.0
    return {"config": "configs[2] variant-sharded", "scaling": "strong", "sites_total": V_total, "haplotypes": H,
            "n_gpus": world, "sites_per_gpu": per, "steps": steps,
            "ms_per_step": wall_ms, "device_ms_per_step": dev_ms,
            "value": V_total * H / (wall_ms * 1e-3), "unit": "genotypes/s",
            "aggregate_GBps": alg / (wall_ms * 1e-3) / 1e9, "frac_of_n_x_peak": alg / (wall_ms * 1e-3) / 1e9 / (peak * world),
            "fst": out.fst, "d_xy": out.d_xy, "parity": {"ranks_agree_bitwise": agree, "oracle_slice_sites": checked},
            "what": "one fm_hudson_pair_sharded call per step on fresh groups: fused two-population sweep of the rank's "
                    "shard + per-super-batch fold + fused fold/NVLink mailbox exchange + one small D2H; un-pipelined; "
                    "wall clock (barrier + synchronize on both sides), max over ranks",
            "timing": "ms_per_step: host wall clock around the synchronous call; device_ms_per_step: CUDA events inside"}


def run(L, _lib, args, rank, world, local, device, dist, peak):
    scale = float(os.environ.get("FM_BENCH_CONFIG_SCALE", "1.0"))
    out = {}
    if world == 1:
        cfgs = []
        for fn in (cfg1_batched, cfg3_hudson, cfg4_wc, cfg5_shard):
            try:
                cfgs.append(fn(L, _lib, device, peak, scale))
            except Exception as e:
                cfgs.append({"config": fn.__name__, "error": f"{type(e).__name__}: {e}"})
            L.fm_trim_pool()
        out["configs"] = cfgs
    try:
        out["strong"] = strong_cfg3(L, _lib, args, rank, world, device, dist, peak, scale)
    except Exception as e:
        out["strong"] = {"error": f"{type(e).__name__}: {e}"}
    return out
