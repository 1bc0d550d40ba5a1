#!/usr/bin/env python
"""bench.py -- headline benchmark of the per-site estimator path (BASELINE.json metric:
site x haplotype genotypes / second, and % of HBM peak).

Workload (BASELINE.json configs[1]): per-site pi/theta tracks (per_site_diversity) for 1M
biallelic sites x 2,504 diploid samples (5,008 haplotypes) split into two inversion-orientation
haplotype groups, mask BED applied, missing-data bitmap present.  One "step" = one pass of the
hot path over the whole shard: for both groups, stream the group's bitplanes once, derive
alt/called counts, evaluate per-site pi and theta (NaN for masked / uncallable sites) and the
region partials (S, sum pi, uncallable sites).

  value : device-resident throughput (planes already in HBM), CUDA events on the launching stream
  e2e   : same metric through the C-ABI with HOST (pinned) buffers: H2D of the u8 matrix +
          bitmap, on-device repack into bitplanes, the stats pass, D2H of the tracks
  roofline / cpu_baseline : see DESIGN.md "Measurement"

python bench.py --gpus N --steps K --warmup W          (our arm; torchrun for N > 1)
python bench.py --impl reference ...                   (CPU arm: oracle port of the Rust path)
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "site_x_haplotype_genotypes_per_sec"
UNIT = "genotypes/s"
N_SITES = 1_000_000
N_SAMPLES = 2_504
MISSING_RATE = 0.01
N_MASK = 2_000
CPU_SAMPLE_SITES = 100_000


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ----------------------------------------------------------------------------- synthetic data
def make_positions(n, seed):
    rng = np.random.default_rng(seed)
    return np.cumsum(rng.integers(1, 50, size=n, dtype=np.int64))


def make_mask(positions, seed, n_mask=N_MASK):
    rng = np.random.default_rng(seed + 1)
    lo, hi = int(positions[0]), int(positions[-1])
    starts = rng.integers(lo, max(hi, lo + 1), size=n_mask, dtype=np.int64)
    lens = rng.integers(1_000, 5_000, size=n_mask, dtype=np.int64)
    return np.ascontiguousarray(np.stack([starts, starts + lens], axis=1).reshape(-1))


def make_groups(n_samples, seed):
    """Inversion orientation per haplotype ~ Bernoulli(0.3) -> haplotype groups 0 / 1."""
    rng = np.random.default_rng(seed + 2)
    orient = rng.random((n_samples, 2)) < 0.3
    g0 = [(s, side) for s in range(n_samples) for side in (0, 1) if not orient[s, side]]
    g1 = [(s, side) for s in range(n_samples) for side in (0, 1) if orient[s, side]]
    return g0, g1


def gen_device(n_sites, n_samples, seed, device, missing_rate=MISSING_RATE, inband=None):
    """u8 matrix [V, S, 2] + packed missing bitmap generated on the GPU (host never has to
    synthesise 5 GB with numpy).  Beta(0.8, 0.8) site frequencies, Bernoulli alleles."""
    import torch

    gen = torch.Generator(device=device)
    gen.manual_seed(seed)
    stride = n_samples * 2
    total = n_sites * stride
    data = torch.empty(total, dtype=torch.uint8, device=device)
    words = (total + 63) // 64
    bitmap = torch.zeros(words, dtype=torch.int64, device=device)
    weights = (torch.ones(64, dtype=torch.int64, device=device) << torch.arange(64, device=device))
    beta = torch.distributions.Beta(torch.tensor(0.8), torch.tensor(0.8))
    chunk = max(64, min(64 * 512, ((1 << 28) // max(n_samples * 2, 1)) // 64 * 64))  # bounds the temporaries
    for s0 in range(0, n_sites, chunk):
        s1 = min(n_sites, s0 + chunk)
        n = s1 - s0
        torch.manual_seed(seed * 1_000_003 + s0)
        f = beta.sample((n,)).to(device).clamp_(0.001, 0.999)
        a = (torch.rand((n, stride), generator=gen, device=device) < f[:, None])
        # whole genotypes are missing ("./." in a VCF): the dense per-allele bitmap then carries exactly the
        # sparse missingness calculate_per_site_diversity sees (SURVEY appendix item 2)
        miss = (torch.rand((n, n_samples), generator=gen, device=device) < missing_rate).repeat_interleave(2, dim=1)
        a &= ~miss
        data[s0 * stride:s1 * stride] = a.reshape(-1).to(torch.uint8)
        if inband is not None:  # the same cohort as an int8 array: missing cells are negative (0xFF)
            a8 = a.to(torch.uint8)
            a8[miss] = 255
            inband[s0 * stride:s1 * stride] = a8.reshape(-1)
        flat = miss.reshape(-1)
        e0 = s0 * stride  # multiple of 64 because chunk is
        pad = (-flat.numel()) % 64
        if pad:
            flat = torch.cat([flat, torch.zeros(pad, dtype=torch.bool, device=device)])
        w = (flat.reshape(-1, 64).to(torch.int64) * weights).sum(dim=1)
        bitmap[e0 // 64:e0 // 64 + w.numel()] = w
    return data, bitmap


def gen_host_sample(n_sites, n_samples, seed):
    """CPU-only generator for the reference arm / cpu baseline sample (numpy)."""
    rng = np.random.default_rng(seed)
    stride = n_samples * 2
    f = np.clip(rng.beta(0.8, 0.8, size=n_sites), 0.001, 0.999).astype(np.float32)
    data = np.empty((n_sites, stride), dtype=np.uint8)
    miss = np.empty((n_sites, stride), dtype=bool)
    step = 8192
    for s0 in range(0, n_sites, step):
        s1 = min(n_sites, s0 + step)
        r = rng.random((s1 - s0, stride), dtype=np.float32)
        m = np.repeat(rng.random((s1 - s0, n_samples), dtype=np.float32) < MISSING_RATE, 2, axis=1)
        data[s0:s1] = (r < f[s0:s1, None]) & ~m
        miss[s0:s1] = m
    return data, miss


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock and throttle reasons under load.  NVML (nvidia_ml_py) is polled every ~0.3 ms so that samples fall
    INSIDE the few-millisecond timed region; `nvidia-smi` (one query per 0.1 s) is the fallback."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NVML_REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"),
                    (0x4, "sw_power_cap"))

    def __init__(self, index):
        self.index, self.samples, self.times, self.reasons, self.max = index, [], [], set(), None
        self.source = "nvidia-smi"
        self._nvml = None
        self._stop = threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)

    def _init_nvml(self):
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        self.max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
        get_reasons(h)
        self._nvml = (pynvml, h, get_reasons)
        self.source = "nvml"

    def _run_nvml(self):
        pynvml, h, get_reasons = self._nvml
        while not self._stop.is_set():
            c = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
            r = int(get_reasons(h))
            self.samples.append(c)
            self.times.append(time.perf_counter())
            for bit, name in self.NVML_REASONS:
                if r & bit:
                    self.reasons.add(name)
            self._stop.wait(0.0003)

    def _run(self):
        try:
            if self._nvml is not None:
                self._run_nvml()
                return
        except Exception:
            self.source = "nvidia-smi"
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                p = [x.strip() for x in out.stdout.strip().split(",")]
                self.samples.append(float(p[0]))
                self.times.append(time.perf_counter())
                self.max = float(p[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                   p[2:6]):
                    if v.lower().startswith("active"):
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.1)

    def count_between(self, t0, t1):
        return sum(1 for t in list(self.times) if t0 <= t <= t1)

    def median_between(self, t0, t1):
        v = [c for c, t in zip(list(self.samples), list(self.times)) if t0 <= t <= t1]
        return statistics.median(v) if v else None

    def __enter__(self):
        try:
            self._init_nvml()  # before the timed region: the library takes tens of milliseconds to load
        except Exception:
            self._nvml = None
        self._t.start()
        t0 = time.perf_counter()
        while self._nvml is not None and not self.samples and time.perf_counter() - t0 < 1.0:
            time.sleep(0.0005)  # the sampler is running when the timed call starts
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max,
                "reasons": sorted(self.reasons), "samples": len(self.samples), "source": self.source}


# ----------------------------------------------------------------------------- CPU arm
def cpu_pass(data2d, miss2d, positions, groups, mask, threads):
    """One pass of the reference's CPU path over a block of sites, per group: the dense summary
    (rayon-parallel in the reference, stats.rs:1415-1460 -> threaded here) plus the serial
    per-site track loop (stats.rs:4693).  Returns seconds."""
    from oracle import pyoracle as orc

    V, stride = data2d.shape
    S = stride // 2
    bits = orc.pack_missing_bits(miss2d.reshape(-1))
    dense = orc.Dense(data2d.reshape(-1), bits, V, S, 2, 1)
    gt = data2d.reshape(V, S, 2).copy()
    gt[np.broadcast_to(miss2d.reshape(V, S, 2).any(axis=2, keepdims=True), gt.shape)] = 0xFF
    vs = orc.Variants(positions, gt)
    region = (int(positions[0]), int(positions[-1]))
    t0 = time.perf_counter()
    for haps in groups:
        orc.build_summary(dense, haps, threads=threads)
        orc.per_site_diversity(vs, haps, region, mask=mask.reshape(-1, 2))
    return time.perf_counter() - t0


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    n = args.cpu_sample_sites
    seed = N_SITES + N_SAMPLES
    pos = make_positions(n, seed)
    data, miss = gen_host_sample(n, args.samples, seed)
    groups = make_groups(args.samples, seed)
    mask = make_mask(pos, seed, max(1, N_MASK * n // N_SITES))
    for _ in range(args.warmup):
        cpu_pass(data[: n // 10], miss[: n // 10], pos[: n // 10], groups, mask, threads)
    times = [cpu_pass(data, miss, pos, groups, mask, threads) for _ in range(args.steps)]
    t = sum(times) / len(times)
    geno = n * args.samples * 2
    val = geno / t
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8 -> popcount u32 + f64", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{n} of {args.sites} sites x {args.samples * 2} haplotypes per step "
                                   "(oracle port of the Rust path; the Rust crate cannot be built here)"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def workload_config(args):
    return {"workload": "configs[1]: per-site pi/theta tracks, two inversion-orientation haplotype groups, "
                        "mask BED, missing bitmap",
            "sites_per_gpu": args.sites, "diploid_samples": args.samples, "haplotypes": args.samples * 2,
            "groups": 2, "mask_intervals": N_MASK, "missing_rate": MISSING_RATE,
            "l2_policy": "inputs larger than L2 (bitplanes ~1.3 GB per pass vs 126 MB L2)"}


# ----------------------------------------------------------------------------- our arm
def group_arrays(haps):
    return (np.asarray([h[0] for h in haps], dtype=np.uint64), np.asarray([h[1] for h in haps], dtype=np.uint8))


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, pi, theta, res, world):
    """--dump-outputs: what the timed call computed in its last step, for comparing two builds output for output.
    pi.npy / theta.npy: the per-site tracks of both groups ([2, sites] float64).  A track has no value (NaN) at a
    masked or uncallable site; the dump keeps every array finite so that two dumps compare element by element:
    pi_defined.npy / theta_defined.npy ([2, sites] float32) hold 1 where the track has a value and 0 where it is
    NaN, and the track holds 0 there.  Beyond DUMP_BYTES a fixed seeded sample of sites, whose indices go to
    site_index.npy.  region_totals.npy: per group [segregating sites, sum of pi, uncallable sites] ([2, 3] float64,
    exact below 2**53); with N > 1 also merged_region_totals.npy, the totals after the exchange between the ranks."""
    os.makedirs(out_dir, exist_ok=True)
    n_groups, V = pi.shape
    keep = (DUMP_BYTES - (1 << 20)) // (2 * n_groups * (8 + 4) + 8)  # tracks, flags, index per site; 1 MB for the rest
    if V > keep:
        idx = np.sort(np.random.default_rng(0).choice(V, keep, replace=False))
        pi, theta = pi[:, idx], theta[:, idx]
        np.save(os.path.join(out_dir, "site_index.npy"), idx.astype(np.float64))
    for name, track in (("pi", pi), ("theta", theta)):
        undefined = np.isnan(track)
        np.save(os.path.join(out_dir, name + ".npy"), np.where(undefined, 0.0, track))
        np.save(os.path.join(out_dir, name + "_defined.npy"), (~undefined).astype(np.float32))
    totals = {"region_totals": (res.last_seg, res.last_pi_sum, res.last_unc)}
    if world > 1:
        totals["merged_region_totals"] = (res.merged_seg, res.merged_pi_sum, res.merged_unc)
    for name, (seg, pi_sum, unc) in totals.items():
        arr = np.array([[seg[k], pi_sum[k], unc[k]] for k in range(n_groups)], dtype=np.float64)
        np.save(os.path.join(out_dir, name + ".npy"), arr)
    log(f"wrote the last timed step's outputs to {out_dir}")


def load_peaks():
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        peaks = {}
    peak = float(peaks.get("hbm_gbs", 6650.0))
    src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    return peak, src


def parity_of_run(L, _lib, groups, g_lists, pos, mask, d_data, d_bitmap, V, S, res, rank, world, dist, device):
    """SURVEY 8(d) "parity check per run": (1) the public call (same fused kernel as the timed steps) against the
    CPU oracle on a 10^4-site slice of THIS rank's shard: positions and NaN pattern exact, pi / theta <= 1e-9
    relative, alt / called counts and S bit-exact; (2) the timed loop's own last-step region totals against the
    public call; (3) N > 1: the totals that came out of the peer exchange against a rank-ordered sum of every
    rank's local totals gathered with torch.distributed (bit-equal).  Raises on any mismatch."""
    import torch
    from oracle import pyoracle as orc  # the checker, never the thing measured

    garr = (C.c_void_p * 2)(*[g.value for g in groups])
    raw_n = (C.c_size_t * 2)(*[len(h) for h in g_lists])
    out_pos = np.empty(V, dtype=np.int64)
    out_pi = np.empty((2, V), dtype=np.float64)
    out_th = np.empty((2, V), dtype=np.float64)
    n = C.c_size_t()
    _lib.check(L.fm_per_site_diversity_multi(garr, raw_n, 2, int(pos[0]), int(pos[-1]), mask.ctypes.data,
                                             mask.size // 2, None, 0, out_pos.ctypes.data, out_pi.ctypes.data,
                                             out_th.ctypes.data, V, C.byref(n)))
    assert n.value == V, "per-site call returned a wrong number of sites"
    ns = min(10_000, V)
    s0 = ((V // 3) // 64) * 64
    s0 = max(0, min(s0, V - ns))
    stride = S * 2
    rows = d_data[s0 * stride:(s0 + ns) * stride].cpu().numpy().reshape(ns, S, 2)
    e0 = s0 * stride
    w0, w1 = e0 // 64, ((s0 + ns) * stride + 63) // 64
    words = d_bitmap[w0:w1].cpu().numpy().view(np.uint64)
    bits = np.unpackbits(words.view(np.uint8), bitorder="little")[e0 - w0 * 64:e0 - w0 * 64 + ns * stride]
    miss = bits.reshape(ns, S, 2).astype(bool)
    gt = rows.copy()
    gt[miss] = 0xFF
    assert np.array_equal(miss[:, :, 0], miss[:, :, 1]), "generator must drop whole genotypes"
    spos = np.ascontiguousarray(pos[s0:s0 + ns])
    vs = orc.Variants(spos, gt)
    dense = orc.Dense(rows.reshape(-1), orc.pack_missing_bits(miss.reshape(-1)), ns, S, 2, 1)
    region = (int(spos[0]), int(spos[-1]))
    checked = 0
    for k, haps in enumerate(g_lists):
        rp, rpi, rth = orc.per_site_diversity(vs, haps, region, mask=mask.reshape(-1, 2))
        gp, gpi, gth = out_pos[s0:s0 + ns], out_pi[k, s0:s0 + ns], out_th[k, s0:s0 + ns]
        if not np.array_equal(gp, rp):
            raise RuntimeError("parity: per-site positions differ from the oracle")
        for got, ref, name in ((gpi, rpi, "pi"), (gth, rth, "theta")):
            if not np.array_equal(np.isnan(got), np.isnan(ref)):
                raise RuntimeError(f"parity: NaN pattern of {name} differs from the oracle (group {k})")
            ok = ~np.isnan(ref)
            if not np.all(np.abs(got[ok] - ref[ok]) <= 1e-9 * np.abs(ref[ok])):
                raise RuntimeError(f"parity: {name} differs from the oracle by more than 1e-9 relative (group {k})")
        checked += 2 * ns
        # integer side: counts of the slice window through the public window call vs the oracle's dense summary
        summ = orc.build_summary(dense, haps)
        w = np.array([region[0], region[1]], dtype=np.int64)
        nv, seg, unc = (np.zeros(1, dtype=np.uint64) for _ in range(3))
        pis = np.zeros(1)
        _lib.check(L.fm_group_window_sums(groups[k], w.ctypes.data, 1, nv.ctypes.data, seg.ctypes.data, pis.ctypes.data,
                                          unc.ctypes.data))
        if int(nv[0]) != ns or int(seg[0]) != int(summ.seg) or int(unc[0]) != int((summ.called < 2).sum()):
            raise RuntimeError(f"parity: window S / uncallable counts differ from the oracle (group {k})")
        if abs(pis[0] - summ.pi_sum) > 1e-9 * abs(summ.pi_sum):
            raise RuntimeError(f"parity: window sum of pi differs from the oracle (group {k})")
    # (2) the timed loop's last step against the public call over the whole shard
    local = []
    for k in range(2):
        seg, unc, pis = C.c_uint64(), C.c_uint64(), C.c_double()
        _lib.check(L.fm_group_summary(groups[k], None, None, C.byref(seg), C.byref(pis), C.byref(unc)))
        if res.last_seg[k] != seg.value or res.last_unc[k] != unc.value:
            raise RuntimeError(f"parity: timed step totals (S {res.last_seg[k]}, uncallable {res.last_unc[k]}) differ "
                               f"from the public call ({seg.value}, {unc.value}) for group {k}")
        if abs(res.last_pi_sum[k] - pis.value) > 1e-9 * abs(pis.value):
            raise RuntimeError(f"parity: timed step sum of pi differs from the public call for group {k}")
        local += [res.last_pi_sum[k], float(res.last_seg[k]), float(res.last_unc[k])]
    exchange = None
    if world > 1:  # (3) what the mailbox exchange delivered == rank-ordered sum of all ranks' local totals
        mine = torch.tensor(local, dtype=torch.float64, device=device)
        allv = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allv, mine)
        tot = np.zeros(6)
        for r in range(world):  # rank order, like fm_k_comm_exchange
            tot = tot + allv[r].cpu().numpy()
        for k in range(2):
            if (res.merged_pi_sum[k] != tot[3 * k] or float(res.merged_seg[k]) != tot[3 * k + 1] or
                    float(res.merged_unc[k]) != tot[3 * k + 2]):
                raise RuntimeError(f"parity: exchanged totals differ from the rank-ordered sum on rank {rank} "
                                   f"(group {k}: {res.merged_pi_sum[k]!r} vs {tot[3 * k]!r})")
        exchange = "merged totals bit-equal to the rank-ordered all_gather sum on every rank"
    return {"status": "ok", "oracle_slice_sites": ns, "values_checked": checked, "tolerance": "ints exact, f64 1e-9 rel",
            "timed_step_totals": "equal to the public call", "exchange": exchange}


def run_ours(args):
    # libraries (NCCL's version banner) may write to fd 1: keep the real stdout for the one JSON line
    json_fd = os.dup(1)
    os.dup2(2, 1)
    import torch
    import torch.distributed as dist

    import ferromic_b200 as fm  # noqa: F401  (fails loudly when the CUDA library is missing)
    from ferromic_b200 import _lib

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    L = _lib.lib()
    _lib.check(L.fm_set_device(local))

    V, S = args.sites, args.samples
    seed = N_SITES + N_SAMPLES + rank
    pos = make_positions(V, seed)
    mask = make_mask(pos, seed)
    g0, g1 = make_groups(S, N_SITES + N_SAMPLES)
    g_lists = (g0, g1)
    garrs = [group_arrays(h) for h in g_lists]
    t0 = time.perf_counter()
    d_data, d_bitmap = gen_device(V, S, seed, device)
    torch.cuda.synchronize()
    log(f"[rank {rank}] generated {V}x{S * 2} u8 matrix on device in {time.perf_counter() - t0:.1f}s")

    # ---------------- device-resident (value)
    m = C.c_void_p()
    _lib.check(L.fm_matrix_create_device(d_data.data_ptr(), d_bitmap.data_ptr(), V, S, 2, 1, pos.ctypes.data,
                                         C.byref(m)))
    groups = []
    for idx, side in garrs:
        h = C.c_void_p()
        _lib.check(L.fm_group_create(m, idx.ctypes.data, side.ctypes.data, len(idx), C.byref(h)))
        groups.append(h)
    garr = (C.c_void_p * 2)(*[g.value for g in groups])
    res = _lib.BenchResult()
    # N > 1: every step ends with the exchange of the groups' region totals (S, sum pi, uncallable
    # sites) -- a fused fold + P2P mailbox kernel over NVLink (csrc/fm_comm.cuh); torch.distributed
    # only carries the 64-byte mailbox handles at start-up and the barriers.
    comm = None
    if world == 1 and os.environ.get("FM_BENCH_SELF_COMM"):  # diagnostic: the exchange kernel alone
        comm = C.c_void_p()
        _lib.check(L.fm_comm_create(0, 1, C.byref(comm)))
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
    warm = max(args.warmup, 3)
    _lib.check(L.fm_bench_diversity(garr, 2, 1, mask.ctypes.data, mask.size // 2, warm, comm, C.byref(res), None,
                                    None))
    # the timed call copies its last step's tracks into these device buffers once its timed region has ended
    last_pi = last_th = None
    if args.dump_outputs and rank == 0:
        last_pi = torch.empty((2, V), dtype=torch.float64, device=device)
        last_th = torch.empty_like(last_pi)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    with ClockSampler(local) as clocks:
        wall0 = time.perf_counter()
        _lib.check(L.fm_bench_diversity(garr, 2, 1, mask.ctypes.data, mask.size // 2, args.steps, comm,
                                        C.byref(res), None if last_pi is None else last_pi.data_ptr(),
                                        None if last_th is None else last_th.data_ptr()))
        dev_ms = res.step_ms_avg * args.steps
        torch.cuda.synchronize()
        wall1 = time.perf_counter()
        wall_ms = (wall1 - wall0) * 1e3
        timed_samples = len(clocks.samples)
        in_region = clocks.count_between(wall0, wall1)
        in_region_mhz = clocks.median_between(wall0, wall1)
        if world > 1:
            dist.barrier()
        # the timed region is a few milliseconds: keep the same kernels running (untimed) until the
        # sampler has seen the clocks under this load a few times
        t_keep = time.perf_counter()
        while len(clocks.samples) < timed_samples + 8 and time.perf_counter() - t_keep < 4.0:
            _lib.check(L.fm_bench_diversity(garr, 2, 1, mask.ctypes.data, mask.size // 2, 200, None,
                                            C.byref(_lib.BenchResult()), None, None))
    if last_pi is not None:
        dump_outputs(args.dump_outputs, last_pi.cpu().numpy(), last_th.cpu().numpy(), res, world)
        del last_pi, last_th
    tmax = torch.tensor([dev_ms], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    dev_ms_max = float(tmax.item())
    geno_per_rank = V * S * 2
    value = world * geno_per_rank * args.steps / (dev_ms_max * 1e-3)

    # ---------------- roofline of the dominant kernel: UNPADDED algorithmic bytes (SURVEY 8d): 2 bits per
    # genotype of the analysed groups + 16 B of tracks per site and group; the 16-byte row padding of the
    # planes shows up in traffic / algorithmic, not in `achieved`
    peak, peak_src = load_peaks()
    launches_per_step = max(1, int(round(res.plane_launches / args.steps)))
    n_hap = len(g0) + len(g1)
    algorithmic = (V * n_hap * 2) / 8.0 + 2 * 16.0 * V
    padded = float(res.plane_bytes_per_step)
    achieved = algorithmic / launches_per_step / (res.plane_ms_avg * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "traffic_plane_pass.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            traffic = tj.get("dram_bytes_per_launch")
            if tj.get("launches_per_step") and tj["launches_per_step"] != launches_per_step:
                traffic = traffic * tj["launches_per_step"] / launches_per_step  # same bytes, other launch split
            traffic_src = "static: ncu --set full capture " + str(tj.get("capture", "profiles/traffic_plane_pass.json")) + \
                          " (not measured in this run)"
        except Exception:
            traffic = None
    kname = ("fm_k_plane_pass_seq (both groups' planes streamed by one persistent launch)" if launches_per_step == 1
             else "fm_k_plane_pass<1>")
    roofline = {"bound": "hbm", "kernel": kname, "launches_per_step": launches_per_step, "achieved": achieved,
                "peak": peak, "unit": "GB/s", "frac": achieved / peak, "frac_of_nominal_8TBs": achieved / 8000.0,
                "peak_source": peak_src, "traffic": traffic, "traffic_source": traffic_src,
                "traffic_over_algorithmic": (traffic / (algorithmic / launches_per_step)) if traffic else None,
                "bytes_per_launch": algorithmic / launches_per_step,
                "bytes_per_launch_def": "V*H*0.25 (allele + called bit of every analysed haplotype) + 2 groups * 16 B/site "
                                        "of pi/theta tracks; row padding excluded",
                "padded_bytes_per_launch": padded / launches_per_step, "ms_per_launch": res.plane_ms_avg,
                "per_group": None if launches_per_step == 1 else
                [{"haplotypes": len(h), "ms": res.group_ms_avg[i],
                  "GBps": res.group_bytes[i] / (res.group_ms_avg[i] * 1e-3) / 1e9} for i, h in enumerate((g0, g1))]}

    # ---------------- parity of this run (oracle = checker only)
    parity = None
    if not args.skip_parity:
        parity = parity_of_run(L, _lib, groups, g_lists, pos, mask, d_data, d_bitmap, V, S, res, rank, world, dist,
                               device)

    # ---------------- K1 + stats from the device-resident u8 matrix (secondary, like-for-like with the CPU arm's
    # input: the reference layout with its bitmap, already in HBM)
    from_u8 = None
    if not args.skip_from_u8:
        def one():
            hs = (C.c_void_p * 2)()
            idx = np.concatenate([a[0] for a in garrs])
            side = np.concatenate([a[1] for a in garrs])
            sizes = (C.c_size_t * 2)(len(g0), len(g1))
            _lib.check(L.fm_groups_create(m, idx.ctypes.data, side.ctypes.data, sizes, 2, hs))
            r = _lib.BenchResult()
            _lib.check(L.fm_bench_diversity(hs, 2, 1, mask.ctypes.data, mask.size // 2, 1, None, C.byref(r), None, None))
            for h in hs:
                L.fm_group_release(C.c_void_p(h))
        one()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        reps = 3
        for _ in range(reps):
            one()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / reps
        from_u8 = {"value": geno_per_rank / dt, "unit": UNIT, "ms_per_step": dt * 1e3,
                   "what": "fm_groups_create (K1 repack of both groups from the device-resident u8 matrix + bitmap) + one "
                           "fused per-site pass, wall clock, per rank"}

    for g in groups:
        L.fm_group_release(g)
    L.fm_matrix_release(m)
    if comm is not None:
        if world > 1:
            dist.barrier()  # nobody may still be writing into a mailbox that is about to be freed
        L.fm_comm_destroy(comm)

    # ---------------- end to end through the C ABI with HOST buffers
    e2e = None
    if not args.skip_e2e:
        stride = S * 2
        h_data = torch.empty(d_data.numel(), dtype=torch.uint8, pin_memory=True)
        h_bitmap = torch.empty(d_bitmap.numel(), dtype=torch.int64, pin_memory=True)
        h_data.copy_(d_data)
        h_bitmap.copy_(d_bitmap)
        torch.cuda.synchronize()
        del d_data, d_bitmap
        torch.cuda.empty_cache()
        rw = (stride + 31) // 32
        # the packed rows a parser would write directly (2 bits per genotype); produced here by the library's own
        # host packer, timed separately
        h_ab = torch.empty(V * rw, dtype=torch.int32, pin_memory=True)
        h_cb = torch.empty(V * rw, dtype=torch.int32, pin_memory=True)
        threads = os.cpu_count() or 1
        pack_ms = []
        for _ in range(2):
            t0 = time.perf_counter()
            _lib.check(L.fm_pack_rows(h_data.data_ptr(), h_bitmap.data_ptr(), 1, 0, V, V, stride, h_ab.data_ptr(),
                                      h_cb.data_ptr(), 0))
            pack_ms.append((time.perf_counter() - t0) * 1e3)
        # the same rows with a sparse missing list instead of the called plane (1.17 instead of 2 bits per genotype
        # at 1 % missing): what a parser emits when it notes the "./." calls as it reads them
        h_start = torch.empty(V + 1, dtype=torch.int64, pin_memory=True)
        need = C.c_size_t()
        cap = int(V * stride * MISSING_RATE * 1.5) + 1024
        h_cols = torch.empty(cap, dtype=torch.int16, pin_memory=True)
        h_ab2 = torch.empty(V * rw, dtype=torch.int32, pin_memory=True)
        pack_sparse_ms = []
        for _ in range(2):
            t0 = time.perf_counter()
            _lib.check(L.fm_pack_rows_sparse(h_data.data_ptr(), h_bitmap.data_ptr(), 1, 0, V, V, stride, h_ab2.data_ptr(),
                                             h_start.data_ptr(), h_cols.data_ptr(), cap, 2, 0, C.byref(need)))
            pack_sparse_ms.append((time.perf_counter() - t0) * 1e3)
        n_missing = int(need.value)
        # ... and the same list as one-byte gap codes (col_bytes = 1, include/ferromic_gpu.h): the headline input
        h_startg = torch.empty(V + 1, dtype=torch.int64, pin_memory=True)
        h_gaps = torch.empty(cap * 2, dtype=torch.uint8, pin_memory=True)
        _lib.check(L.fm_pack_rows_sparse(h_data.data_ptr(), h_bitmap.data_ptr(), 1, 0, V, V, stride, h_ab2.data_ptr(),
                                         h_startg.data_ptr(), h_gaps.data_ptr(), cap * 2, 1, 0, C.byref(need)))
        n_gap_bytes = int(need.value)
        out_pos = torch.empty(V, dtype=torch.int64, pin_memory=True).numpy()  # caller-owned result buffers are pinned
        out_pi = torch.empty((2, V), dtype=torch.float64, pin_memory=True).numpy()
        out_th = torch.empty((2, V), dtype=torch.float64, pin_memory=True).numpy()
        raw_n = (C.c_size_t * 2)(len(g0), len(g1))
        gidx2 = np.array([0, 1], dtype=np.uint64)

        def e2e_step(mode, phases, src=None):
            t = [time.perf_counter()]

            def lap(name):
                t.append(time.perf_counter())
                phases[name] = phases.get(name, 0.0) + (t[-1] - t[-2]) * 1e3

            ih = C.c_void_p()
            _lib.check(L.fm_ingest_begin(V, S, 2, 1, 1, pos.ctypes.data, 0, C.byref(ih)))
            for idx, side in garrs:
                _lib.check(L.fm_ingest_add_group(ih, idx.ctypes.data, side.ctypes.data, len(idx), None))
            streamed = mode == "packed_gaps_streamed"
            n = C.c_size_t()
            if streamed:  # the tracks are requested up front and stream out while the rows stream in
                _lib.check(L.fm_ingest_request_tracks(ih, gidx2.ctypes.data, raw_n, 2, int(pos[0]), int(pos[-1]),
                                                      mask.ctypes.data, mask.size // 2, None, 0, out_pos.ctypes.data,
                                                      out_pi.ctypes.data, out_th.ctypes.data, V, C.byref(n)))
            lap("begin+declare_groups")
            if mode in ("packed_gaps", "packed_gaps_streamed"):  # allele bits + gap-coded missing list
                _lib.check(L.fm_ingest_rows_packed_sparse(ih, h_ab2.data_ptr(), h_startg.data_ptr(), h_gaps.data_ptr(), 1, 0, V))
            elif mode == "packed_sparse":  # the same with u16 column indices
                _lib.check(L.fm_ingest_rows_packed_sparse(ih, h_ab2.data_ptr(), h_start.data_ptr(), h_cols.data_ptr(), 2, 0, V))
            elif mode == "packed":    # 2-bit rows over PCIe, compressed into both groups' planes chunk by chunk
                _lib.check(L.fm_ingest_rows_packed(ih, h_ab.data_ptr(), h_cb.data_ptr(), 0, V))
            elif mode == "u8_pack":   # u8 + bitmap in, the library packs on the host while the previous chunk uploads
                d, b = src or (h_data.data_ptr(), h_bitmap.data_ptr())
                _lib.check(L.fm_ingest_rows_pack(ih, d, b, 0, V, 0))
            else:                     # round-1 path: the u8 matrix itself crosses PCIe
                d, b = src or (h_data.data_ptr(), h_bitmap.data_ptr())
                _lib.check(L.fm_ingest_rows(ih, d, b, 0, V))
            lap("ingest_rows")
            mh = C.c_void_p()
            gh = (C.c_void_p * 2)()
            _lib.check(L.fm_ingest_finish(ih, C.byref(mh), gh, None))
            lap("finish")
            if not streamed:
                _lib.check(L.fm_per_site_diversity_multi(gh, raw_n, 2, int(pos[0]), int(pos[-1]), mask.ctypes.data,
                                                         mask.size // 2, None, 0, out_pos.ctypes.data, out_pi.ctypes.data,
                                                         out_th.ctypes.data, V, C.byref(n)))
            lap("per_site_diversity_multi")
            for g in gh:
                L.fm_group_release(C.c_void_p(g))
            L.fm_matrix_release(mh)
            lap("release")
            return n.value

        def timed(mode, k, src=None):
            e2e_step(mode, {}, src)  # warm-up
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            L.fm_timings_reset()
            phases = {}
            t0 = time.perf_counter()
            for _ in range(k):
                e2e_step(mode, phases, src)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            tim = _lib.Timings()
            L.fm_timings_get(C.byref(tim))
            te = torch.tensor([dt], dtype=torch.float64, device=device)
            if world > 1:
                dist.all_reduce(te, op=dist.ReduceOp.MAX)
            dt = float(te.item())
            return {"value": world * geno_per_rank * k / dt, "ms_per_step": dt / k * 1e3,
                    "breakdown_ms_per_step": {"h2d": tim.h2d_ms / k, "repack": tim.repack_ms / k, "pack_host": tim.pack_ms / k,
                                              "stats": tim.stats_ms / k, "reduce": tim.reduce_ms / k, "d2h": tim.d2h_ms / k},
                    "host_phase_ms_per_step": {k_: v_ / k for k_, v_ in phases.items()}}

        k = max(1, min(args.steps, args.e2e_steps))
        r_two = timed("packed_gaps", k)
        check_pi = out_pi.copy()
        check_th, check_pos = out_th.copy(), out_pos.copy()
        out_pi[:] = -1.0
        out_th[:] = -1.0
        out_pos[:] = -1
        r_sparse = timed("packed_gaps_streamed", k)
        same_streamed = bool(np.array_equal(out_pos, check_pos) and
                             np.array_equal(np.isnan(check_pi), np.isnan(out_pi)) and
                             np.array_equal(check_pi[~np.isnan(check_pi)], out_pi[~np.isnan(out_pi)]) and
                             np.array_equal(np.isnan(check_th), np.isnan(out_th)) and
                             np.array_equal(check_th[~np.isnan(check_th)], out_th[~np.isnan(out_th)]))
        if not same_streamed:
            raise RuntimeError("parity: the streamed tracks differ from fm_per_site_diversity_multi after finish")
        r_cols = timed("packed_sparse", k)
        same_cols = bool(np.array_equal(np.isnan(check_pi), np.isnan(out_pi)) and
                         np.array_equal(check_pi[~np.isnan(check_pi)], out_pi[~np.isnan(out_pi)]))
        r_packed = timed("packed", k)
        same0 = same_cols and bool(np.array_equal(np.isnan(check_pi), np.isnan(out_pi)) and
                                   np.array_equal(check_pi[~np.isnan(check_pi)], out_pi[~np.isnan(out_pi)]))
        r_u8pack = timed("u8_pack", k)
        same = same0 and bool(np.array_equal(np.isnan(check_pi), np.isnan(out_pi)) and
                              np.array_equal(check_pi[~np.isnan(check_pi)], out_pi[~np.isnan(out_pi)]))
        r_u8 = timed("u8", k) if not args.skip_u8 else None
        if r_u8 is not None:
            same = same and bool(np.array_equal(check_pi[~np.isnan(check_pi)], out_pi[~np.isnan(out_pi)]))
        if not same:
            raise RuntimeError("parity: the packed, pack-on-host and u8 ingests produced different per-site tracks")
        pageable = None
        if rank == 0 and world == 1 and not args.skip_pageable:
            p_data = np.array(h_data.numpy(), copy=True)   # what a Rust Vec<u8> / numpy array is: pageable
            p_bitmap = np.array(h_bitmap.numpy(), copy=True)
            src = (p_data.ctypes.data, p_bitmap.ctypes.data)
            pageable = {"u8_pack_ms_per_step": timed("u8_pack", 1, src)["ms_per_step"],
                        "u8_ms_per_step": None if args.skip_u8 else timed("u8", 1, src)["ms_per_step"]}
            del p_data, p_bitmap
        h2d_packed = int(2 * V * rw * 4 + V * 8 + mask.size * 8)
        h2d_cols = int(V * rw * 4 + (V + 1) * 8 + n_missing * 2 + V * 8 + mask.size * 8)
        h2d_sparse = int(V * rw * 4 + (V + 1) * 8 + n_gap_bytes + V * 8 + mask.size * 8)
        # two public flows give the same tracks: `streamed` (fm_ingest_request_tracks: results flow out while the rows flow
        # in) and `two_calls` (per-site call after finish).  The headline is the faster one of this run: alone on its
        # link a GPU gains from the duplex traffic, several GPUs behind one host root complex may not.
        head, flow = (r_sparse, "streamed") if r_sparse["value"] >= r_two["value"] else (r_two, "two_calls")
        e2e = {"value": head["value"], "unit": UNIT, "h2d_bytes_per_step": h2d_sparse,
               "d2h_bytes_per_step": int(2 * 2 * V * 8 + V * 8), "steps": k, "ms_per_step": head["ms_per_step"],
               "breakdown_ms_per_step": head["breakdown_ms_per_step"],
               "host_phase_ms_per_step": head["host_phase_ms_per_step"],
               "flow": flow,
               "api": "streamed: fm_ingest_begin / add_group x2 / fm_ingest_request_tracks / fm_ingest_rows_packed_sparse (allele "
                      "bit words + gap-coded missing list from pinned host memory; chunked H2D overlapped with "
                      "fm_k_expand_called, the compress pass K1p and the per-site pass of every chunk, whose pi / theta tracks "
                      "and positions the kernels store straight into the caller's page-locked arrays over PCIe while the next "
                      "chunks upload) / finish.  two_calls: the same ingest, finish, then ONE fm_per_site_diversity_multi call "
                      "(tracks stored by the kernel into the page-locked arrays).  Per rank; `flow` names the one in `value`",
               "streamed": {**r_sparse, "h2d_bytes_per_step": h2d_sparse},
               "input": "packed rows: one allele bit per genotype + the missing cells of every row as one-byte gap codes "
                        "(CSR, col_bytes = 1), as a parser emits them (include/ferromic_gpu.h); %d missing cells = %.2f %% of "
                        "the matrix in %d bytes" % (n_missing, 100.0 * n_missing / (V * stride), n_gap_bytes),
               "bits_per_genotype_over_pcie": 8.0 * h2d_sparse / (V * stride),
               "two_calls": {**r_two, "h2d_bytes_per_step": h2d_sparse},
               "packed_u16_columns": {**r_cols, "h2d_bytes_per_step": h2d_cols,
                                      "what": "the same ingest with the missing list as u16 column indices (col_bytes = 2)"},
               "packed_called_plane": {**r_packed, "h2d_bytes_per_step": h2d_packed,
                                       "what": "fm_ingest_rows_packed: allele bit + called bit per genotype (2 bits)"},
               "packer": {"ms": min(pack_ms), "sparse_ms": min(pack_sparse_ms), "cores": threads,
                          "u8_GBps": V * stride / (min(pack_ms) * 1e-3) / 1e9,
                          "what": "fm_pack_rows / fm_pack_rows_sparse over the pinned u8 matrix + bitmap (AVX-512 or AVX2, all "
                                  "host threads), outside the timed region of `value` above; inside it for "
                                  "from_u8_pack_on_host"},
               "from_u8_pack_on_host": {**r_u8pack, "h2d_bytes_per_step": h2d_packed,
                                        "what": "fm_ingest_rows_pack: the caller holds the reference's u8 matrix + bitmap "
                                                "(pinned); the library packs chunk i+1 on the host while chunk i uploads"},
               "from_u8_over_pcie": None if r_u8 is None else
               {**r_u8, "h2d_bytes_per_step": int(h_data.numel() + h_bitmap.numel() * 8 + V * 8),
                "what": "round-1 path: fm_ingest_rows, the u8 matrix + bitmap cross PCIe and are repacked on the device"},
               "pageable_host": pageable,
               "tracks_identical_across_ingests": same,
               "timing": "wall clock around synchronous C-ABI calls, cuda-synchronised on both sides, max over ranks"}

    # ---------------- CPU baseline (rank 0, N = 1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu:
        n = min(args.cpu_sample_sites, V)
        threads = os.cpu_count() or 1
        sd, sm = gen_host_sample(n, S, N_SITES + N_SAMPLES)
        spos = pos[:n]
        smask = make_mask(spos, N_SITES + N_SAMPLES, max(1, N_MASK * n // N_SITES))
        t = cpu_pass(sd, sm, spos, (g0, g1), smask, threads)
        cpu = {"value": n * S * 2 / t, "unit": UNIT, "cores": threads, "kind": "port", "seconds": t,
               "sample": f"{n} of {V} sites x {S * 2} haplotypes, both groups (oracle port: threaded dense summary "
                         "+ serial per-site track loop, as in the reference)"}

    extra = {}
    if not args.skip_configs:
        try:
            import bench_configs
            extra = bench_configs.run(L, _lib, args, rank, world, local, device, dist if world > 1 else None, peak)
        except Exception as e:  # the headline line must still be printed
            extra = {"configs_error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        cl = clocks.summary()
        cl["samples_in_timed_region"] = in_region
        cl["sm_mhz_in_timed_region"] = in_region_mhz
        cl["sampling"] = (f"{in_region} samples inside the {wall_ms:.1f} ms wall-clock window of the timed call "
                          f"({dev_ms:.1f} ms of device time), the rest during an untimed keep-alive loop of the same "
                          "kernels right after it")
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": warm, "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "u8 -> 1-bit planes, popcount u32 + f64",
                "data": "synthetic", "config": workload_config(args), "roofline": roofline, "cpu_baseline": cpu,
                "e2e": e2e, "gpu_launches": int(res.plane_launches + res.other_launches),
                "parity": parity, "value_from_resident_u8": from_u8,
                "clocks": cl, "wall_ms_per_step": wall_ms / args.steps,
                "exchange_ms_per_step": res.comm_ms_avg if comm is not None else None,
                "collective": None if world == 1 else "per step: fused fold + P2P mailbox exchange of region totals "
                                                      "(fm_k_comm_exchange over NVLink peer memory), inside the timed region",
                "timing": "CUDA events on the launching stream (cudaStreamPerThread), max over ranks"}
        line.update(extra)
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--sites", type=int, default=N_SITES)
    ap.add_argument("--samples", type=int, default=N_SAMPLES)
    ap.add_argument("--cpu-sample-sites", type=int, default=CPU_SAMPLE_SITES)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-pageable", action="store_true")
    ap.add_argument("--skip-u8", action="store_true", help="skip the round-1 u8-over-PCIe e2e variant")
    ap.add_argument("--skip-parity", action="store_true")
    ap.add_argument("--skip-from-u8", action="store_true")
    ap.add_argument("--skip-configs", action="store_true", help="skip configs 1/3/4/5 and the strong-scaling block")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the per-site tracks and region totals of the last timed step as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
