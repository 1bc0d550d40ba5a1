"""Weir & Cockerham (K4, csrc/fm_wc.cuh, run_wc in csrc/fm_gpu.cu) at every kernel geometry and population limit.

The host picks K4's shapes from the number of populations G, the allele slots A and the window lengths: the biallelic
producer / consumer pairs kernel with 1-9 chunks of 352 pair slots per segment over a persistent grid, the
multi-allelic kernel with 1, 2, 4 or 8 pairs per lane, the fold with one or two rounds of 16-segment chunks, and two
count producers (count-only groups or bitplanes + ensure_counts) depending on the row width.  This file restates those
host rules in Python, lists one case per class in a table whose coverage a CPU test asserts, and runs every case on
the GPU against the C oracle (oracle/ferromic_oracle.c, orc_wc_fst):

  * per-site overall state / a / b and per-pair a / b bit for bit (NaN exactly where the oracle has no pair data), and
    the per-group sample sizes against called counts taken directly from the genotype array;
  * window and region totals bit for bit against the association the DESIGN fixes: segments cut at multiples of 1024
    of the site index, each segment summed sequentially in site order, the window's segments folded in 16-segment
    chunks counted from its first segment, the chunk sums added in order;
  * the same totals against an exact sum (math.fsum) within gamma_{k-1} * sum |x|, which holds for any association.
"""
import ctypes as C
import math
import os
import subprocess
import sys
from typing import NamedTuple, Tuple

import numpy as np
import pytest

EPS = 2.0 ** -53
UNG = 0xFFFF
B200_SMS = 148  # the table's class predictions; the GPU tests re-check with the device's own SM count

# ------------------------------------------------------------------ host rules, restated
SEG = 1024                          # fm_wc.cuh:32 kWcSegSites
MULTI_MAX_PAIR_WARPS = 11           # fm_wc.cuh:33 kWcMaxPairWarps
MAX_KP = 8                          # fm_wc.cuh:34 kWcMaxKP
PC_SITES, PC_STAGES = 16, 4         # fm_wc.cuh:159-160 kWcPcSites, kWcPcStages
PC_PAIR_WARPS = 11                  # fm_wc.cuh:162 kWcPcPairWarps
FOLD_CHUNK, FOLD_MAX_WARPS = 16, 16  # fm_wc.cuh:674-675
STAGING_LIMIT = 200 * 1024          # fm_gpu.cu:3473-3476
SM_SMEM, BLOCK_RESERVED = 228 * 1024, 1024  # shared memory per SM of sm_100 and the per-block reservation


def segments(lo, hi):
    """fm_gpu.cu:3451-3456: a window [lo, hi) of site indices cut at multiples of SEG."""
    out, v = [], lo
    while v < hi:
        e = min(hi, (v // SEG + 1) * SEG)
        out.append((v, e))
        v = e
    return out


def n_pairs(G):
    return G * (G - 1) // 2 if G > 0 else 0  # fm_gpu.cu:3441


def pc_chunks(G):
    """fm_gpu.cu:3563: chunks of 352 pair slots per segment of the biallelic pairs kernel."""
    return (n_pairs(G) + PC_PAIR_WARPS * 32 - 1) // (PC_PAIR_WARPS * 32)


def pc_smem(G):
    """fm_wc.cuh:164-168 fm_wc_pc_smem: 4 stages of 16 sites x (G | 1) x (double4 + uint2), barriers, 16 bytes."""
    return PC_STAGES * PC_SITES * (G | 1) * (32 + 8) + 2 * PC_STAGES * 8 + 16


def pc_blocks_per_sm_bound(G):
    """Upper bound of the pairs kernel's CTAs per SM (fm_gpu.cu:3567-3571 asks the occupancy API): 384 threads and
    pc_smem(G) + the block reservation out of the SM's shared memory."""
    return min(2048 // ((PC_PAIR_WARPS + 1) * 32), SM_SMEM // (pc_smem(G) + BLOCK_RESERVED))


def multi_geometry(G, kp_pref=1):
    """fm_gpu.cu:3467-3469: (pair warps, pairs per lane needed) of the multi-allelic kernel; FM_WC_KP = kp_pref."""
    P = n_pairs(G)
    n_pw = max(1, min(MULTI_MAX_PAIR_WARPS, (P + 32 * kp_pref - 1) // (32 * kp_pref)))
    return n_pw, max(1, (P + n_pw * 32 - 1) // (n_pw * 32))


def kp_template(kp_need):
    """fm_gpu.cu:3551-3554: the fm_k_wc_multi<KP> instance launched."""
    return 1 if kp_need <= 1 else 2 if kp_need <= 2 else 4 if kp_need <= 4 else 8


def multi_smem(G, A):
    """fm_wc.cuh:462-465 fm_wc_multi_cta_smem: freq f64 [32][G][A] | cn u32 [32][G+1] | ca u32 [32][G+1][A] | info."""
    return 32 * G * A * 8 + 32 * (G + 1) * 4 + 32 * (G + 1) * A * 4 + 32 * 4 + 16


def wc_refusal(G, A):
    """fm_gpu.cu:3471-3477: why run_wc refuses G populations with A allele slots, or None."""
    if A > 2:
        if multi_geometry(G)[1] > MAX_KP:
            return "pairs per lane"
        if multi_smem(G, A) > STAGING_LIMIT:
            return "staging"
    elif n_pairs(G) and pc_smem(G) > STAGING_LIMIT:
        return "staging"
    return None


def multi_blocks(n_seg, sms):
    """fm_gpu.cu:3540: one CTA per segment, at most 8 per SM (each CTA then takes several segments)."""
    return max(1, min(n_seg, 8 * sms))


def fold_warps(max_seg):
    """fm_gpu.cu:3595-3597: warps of fm_k_wc_fold (one chunk each per round)."""
    return max(1, min(FOLD_MAX_WARPS, (max(max_seg, 1) + FOLD_CHUNK - 1) // FOLD_CHUNK))


def repack_warp_smem(stride, packed, bitmap):
    """fm_gpu.cu:1781-1791 repack_warp_smem (bitmap: a u8 matrix with a missing bitmap, not in-band)."""
    row_buf = 0 if packed else ((stride + 15) & ~15) + 32
    bit_buf = ((stride + 63) // 64 + 2) * 8 if (not packed and bitmap) else 0
    cnt_buf = 2 * ((stride + 31) // 32 + 1) * 4 + (((stride + 127) // 128) * 4 + 4) * 4
    return (row_buf + bit_buf + cnt_buf + 15) & ~15


def count_only(stride, packed, bitmap, A):
    """fm_gpu.cu:1792-1793, 1815: a partition group keeps only alt / called counts (the count pass writes them);
    otherwise it gets bitplanes and ensure_counts derives the counts."""
    return A == 2 and repack_warp_smem(stride, packed, bitmap) <= (100 * 1024 if packed else 24 * 1024)


def slots(max_allele):
    """Allele slots A = 2^n_bits with the smallest n_bits such that 2^n_bits > max_allele (fm_gpu.cu:1800-1801)."""
    b = 1
    while (1 << b) <= max_allele:
        b += 1
    return 1 << b


# ------------------------------------------------------------------ the case table
FORM_PACKED = {"u8": False, "u8-nobitmap": False, "inband": False, "stream": False, "packed-dense": True,
               "packed-sparse": True}
FORM_BITMAP = {"u8": True, "u8-nobitmap": False, "inband": False, "stream": True, "packed-dense": True,
               "packed-sparse": True}
ALL_FORMS = ("u8", "inband", "packed-dense", "packed-sparse", "stream")


class Case(NamedTuple):
    name: str
    max_allele: int
    sizes: Tuple[int, ...]       # samples per group (both sides in the group); 0 = an empty group
    V: object                    # sites, or a function of the SM count
    region: object               # (lo, hi) site indices, negative hi counts from V; or a function of V
    forms: Tuple[str, ...] = ("u8",)
    missing: float = 0.06
    special: bool = True         # samples whose sides sit in different groups + the edge rows
    seed: int = 1

    @property
    def G(self):
        return len(self.sizes)

    @property
    def A(self):
        return slots(self.max_allele)

    def n_sites(self, sms):
        return self.V(sms) if callable(self.V) else self.V

    def bounds(self, sms):
        V = self.n_sites(sms)
        lo, hi = self.region(V) if callable(self.region) else self.region
        return lo, (hi if hi > 0 else V + hi)

    @property
    def S(self):
        return (2 if self.special and self.G >= 2 else 0) + sum(self.sizes) + 3


def _pc_tasks_V(sms):
    """Segments of the G = 79 case: more than 3 x the host's grid of tasks (9 chunks per segment, 1 CTA per SM)."""
    grid = pc_blocks_per_sm_bound(79) * sms
    return (3 * grid // pc_chunks(79) + 2) * SEG + 300


def _multi_many_V(sms):
    return (8 * sms + 40) * SEG


MID = (200, -211)  # starts and ends mid-segment
TABLE = [
    # biallelic: fm_k_wc_overall + fm_k_wc_pairs_pc<1>
    Case("bi-G1", 1, (9,), 3300, MID, seed=11),
    Case("bi-G2-one-sample-groups", 1, (1, 1), 3300, MID, special=False, seed=12),
    Case("bi-G2-split-samples", 1, (4, 3), 3300, MID, seed=13),
    Case("bi-G27", 1, (2,) * 27, 3300, MID, seed=14),
    Case("bi-G28", 1, (2,) * 28, 3300, MID, seed=15),
    Case("bi-G40", 1, (2,) * 40, 3300, MID, seed=16),
    Case("bi-G79-tasks", 1, (2,) * 79, _pc_tasks_V, (37, -301), seed=17),
    Case("bi-producers", 1, (6, 5, 7, 0, 4), 3300, MID, forms=ALL_FORMS, seed=18),
    Case("bi-producers-nomiss", 1, (6, 5, 7, 4), 3300, MID, missing=0.0, special=False,
         forms=("u8-nobitmap", "u8", "inband", "packed-dense", "packed-sparse", "stream"), seed=19),
    Case("bi-wide-8165", 1, (4000, 4100, 40, 20), 300, (3, -5), forms=("u8", "packed-dense"), seed=20),
    Case("bi-large-n", 1, (15000, 15100, 3, 0), 200, (0, 200), forms=("packed-dense", "u8"), missing=0.01, seed=21),
    # multi-allelic: fm_k_wc_multi<KP>
    Case("multi-A4-G3", 3, (3, 4, 3), 3300, MID, forms=("u8", "inband", "stream"), seed=31),
    Case("multi-A4-G28", 2, (2,) * 28, 3300, MID, seed=32),
    Case("multi-A4-G40", 3, (2,) * 40, 3300, MID, seed=33),
    Case("multi-A4-G75", 3, (2,) * 75, 3300, MID, seed=34),
    Case("multi-A8-G63", 7, (2,) * 63, 3300, MID, seed=35),
    Case("multi-A16-G32", 15, (2,) * 32, 3300, MID, seed=36),
    Case("multi-A4-many-segments", 3, (3, 3, 4), _multi_many_V, (17, -100), seed=37),
    # the FM_WC_SITES_PER_STEP = 2 / FM_WC_KP = 4 process compares these two (see KNOB_CASES)
    Case("knob-bi-G5", 1, (4, 3, 5, 2, 3), 3700, (100, 3 * SEG + 511), seed=41),
    Case("knob-multi-A4-G30", 3, (2,) * 30, 2600, (5, 2 * SEG + 300), seed=42),
]
REFUSED = [  # (max_allele, G): the smallest G each limit refuses
    (1, 80), (3, 76), (7, 64), (15, 33),
]
KNOB_CASES = ("knob-bi-G5", "knob-multi-A4-G30")
KNOB_ENV = {"FM_WC_SITES_PER_STEP": "2", "FM_WC_KP": "4"}
BY_NAME = {c.name: c for c in TABLE}

# windows of one fm_wc_window_sums call, as site-index ranges [lo, hi) (V >= 340k); None = an empty window
WINDOW_CASE = Case("bi-windows", 1, (5, 6, 4, 5, 3), 340_000, (0, 340_000), seed=51)


def window_list(V):
    k = 37
    return [
        (5, 5 + 300_000 + 1000),            # > 256 segments: a second, partial fold round
        (3 * SEG, 19 * SEG),                # exactly 16 segments, aligned
        (2 * SEG + 100, 17 * SEG + 50),     # exactly 16 segments, both ends mid-segment
        (20 * SEG, 37 * SEG),               # exactly 17 segments
        (20 * SEG + 1, 37 * SEG + 1),       # 18 segments
        (k * SEG, (k + 1) * SEG),           # one aligned segment [1024k, 1024(k+1) - 1]
        (7, 8), (5 * SEG, 5 * SEG + 1), (6 * SEG - 1, 6 * SEG),  # one site
        None,                               # empty
        (1000, 50_000), (30_000, 80_000),   # overlapping
        (40 * SEG + 3, 42 * SEG + 37),      # last segment ends inside a 16-site stage
        (60 * SEG + 17, 60 * SEG + 530),    # one segment, both ends mid-stage
        (0, V),
    ]


def classes(case, sms=B200_SMS):
    """Kernel classes one table entry reaches."""
    G, A = case.G, case.A
    lo, hi = case.bounds(sms)
    segs = segments(lo, hi)
    out = set()
    if A == 2:
        if G == 1:
            out.add("bi-no-pairs-kernel")
        elif G > 1:
            ch = pc_chunks(G)
            out.add(f"bi-chunks-{ch}")
            if n_pairs(G) % (PC_PAIR_WARPS * 32) == PC_PAIR_WARPS * 32 - 1:
                out.add("bi-one-empty-slot")
            if wc_refusal(G + 1, 2):
                out.add("bi-largest-G")
            tasks = len(segs) * ch
            if tasks > 3 * pc_blocks_per_sm_bound(G) * sms:
                out.add("bi-tasks>3xgrid")
            if case.name in KNOB_CASES and (hi - lo) % SEG and segs[-1][1] - segs[-1][0] & 1:
                out.add("bi-SU2-odd-last-segment")
    else:
        n_pw, kp = multi_geometry(G)
        out.add(f"multi-A{A}-KP{kp_template(kp)}")
        if wc_refusal(G + 1, A):
            out.add(f"multi-A{A}-largest-G")
        if len(segs) > 8 * sms:
            out.add("multi-CTA-several-segments")
        if case.name in KNOB_CASES:
            kn_pw, kn_kp = multi_geometry(G, kp_pref=4)
            if (n_pw, kp) == (11, 2) and (kn_pw, kn_kp) == (4, 4):
                out.add("multi-KP4-with-4-pair-warps")
    if len(segs) >= 3 and lo % SEG and hi % SEG:
        out.add(f"A{A}-3-segments-mid-segment-region")
    for f in case.forms:
        stride = 2 * case.S
        co = count_only(stride, FORM_PACKED[f], FORM_BITMAP[f], A)
        out.add(f"form-{f}")
        out.add(f"A{A}-{'count-only' if co else 'bitplanes'}")
        if A == 2 and not co and count_only(2 * 8160, FORM_PACKED[f], FORM_BITMAP[f], A):
            out.add(f"wide-{f}-bitplanes")
        if A == 2 and co and case.S > 8160 and f.startswith("packed"):
            out.add("wide-packed-count-only")
    if 0 in case.sizes:
        out.add("empty-group")
    if case.sizes.count(1) >= 2 and not case.special:
        out.add("two-one-sample-groups")
    if G >= 2 and sorted(case.sizes)[-2] * 2 >= 30_000:
        out.add("large-n")
    if case.special and G >= 2:
        out.add("edge-rows")
    return out


def window_classes(V):
    out = set()
    for w in window_list(V):
        if w is None:
            out.add("win-empty")
            continue
        lo, hi = w
        segs = segments(lo, hi)
        n_ch = (len(segs) + FOLD_CHUNK - 1) // FOLD_CHUNK
        if n_ch > FOLD_MAX_WARPS:
            out.add("win-second-fold-round")
        if len(segs) in (16, 17):
            out.add(f"win-{len(segs)}-segments")
        if lo % SEG == 0 and hi == lo + SEG:
            out.add("win-aligned-segment")
        if hi - lo == 1:
            out.add("win-one-site")
        if (hi - segs[-1][0]) % PC_SITES:
            out.add("win-last-segment-mid-stage")
    ws = [w for w in window_list(V) if w is not None]
    if any(a[0] < b[0] < a[1] for a in ws for b in ws):
        out.add("win-overlapping")
    return out


REQUIRED = ({"bi-no-pairs-kernel", "bi-chunks-1", "bi-chunks-2", "bi-chunks-3", "bi-chunks-9", "bi-one-empty-slot",
             "bi-largest-G", "bi-tasks>3xgrid", "bi-SU2-odd-last-segment", "multi-CTA-several-segments",
             "multi-KP4-with-4-pair-warps", "A2-3-segments-mid-segment-region", "A4-3-segments-mid-segment-region",
             "A8-3-segments-mid-segment-region", "A16-3-segments-mid-segment-region", "A2-count-only",
             "A2-bitplanes", "A4-bitplanes", "A8-bitplanes", "A16-bitplanes", "wide-u8-bitplanes",
             "wide-packed-count-only", "empty-group", "two-one-sample-groups", "large-n", "edge-rows"} |
            {f"multi-A4-KP{k}" for k in (1, 2, 4, 8)} | {"multi-A8-KP8", "multi-A16-KP2"} |
            {f"multi-A{a}-largest-G" for a in (4, 8, 16)} |
            {f"form-{f}" for f in FORM_PACKED})
REQUIRED_WINDOWS = {"win-empty", "win-second-fold-round", "win-16-segments", "win-17-segments", "win-aligned-segment",
                    "win-one-site", "win-last-segment-mid-stage", "win-overlapping"}


def test_table_reaches_every_kernel_class():
    reached = set().union(*(classes(c) for c in TABLE))
    assert REQUIRED <= reached, f"classes no case reaches: {sorted(REQUIRED - reached)}"
    assert REQUIRED_WINDOWS <= window_classes(WINDOW_CASE.V), sorted(REQUIRED_WINDOWS - window_classes(WINDOW_CASE.V))
    assert "multi-CTA-several-segments" in classes(BY_NAME["multi-A4-many-segments"])
    for c in TABLE:
        assert wc_refusal(c.G, c.A) is None, c.name
        assert c.bounds(B200_SMS)[1] <= c.n_sites(B200_SMS)


def test_population_limits_are_exact():
    """The largest G each limit admits: 79 biallelic (staging), 75 at A = 4 (pairs per lane), 63 at A = 8 and 32 at
    A = 16 (staging) -- and the refused cases sit exactly one above them."""
    def largest(A):
        G = 2
        while wc_refusal(G + 1, A) is None:
            G += 1
        return G
    assert [largest(a) for a in (2, 4, 8, 16)] == [79, 75, 63, 32]
    assert [(m, largest(slots(m)) + 1) for m, _ in REFUSED] == REFUSED
    assert wc_refusal(80, 2) == "staging" and pc_smem(79) <= STAGING_LIMIT < pc_smem(80)
    assert wc_refusal(76, 4) == "pairs per lane" and multi_smem(76, 4) <= STAGING_LIMIT
    assert wc_refusal(64, 8) == "staging" and multi_geometry(64)[1] <= MAX_KP
    assert wc_refusal(33, 16) == "staging"
    # pair-chunk and KP boundaries: 351 / 352 pairs, 27 / 28 populations
    assert (pc_chunks(27), pc_chunks(28), pc_chunks(79)) == (1, 2, 9)
    assert [kp_template(multi_geometry(G)[1]) for G in (26, 27, 28, 38, 39, 53, 54, 75)] == [1, 1, 2, 2, 4, 4, 8, 8]
    # FM_WC_KP = 4 on 30 populations: 4 pair warps with 4 pairs per lane instead of 11 with 2; 5 populations stay at 1
    assert multi_geometry(30) == (11, 2) and multi_geometry(30, 4) == (4, 4) and multi_geometry(5, 4) == (1, 1)
    # count-only widths: 8160 diploid samples of u8 rows with a bitmap, 136496 of packed rows
    assert count_only(2 * 8160, False, True, 2) and not count_only(2 * 8161, False, True, 2)
    assert count_only(2 * 136496, True, True, 2) and not count_only(2 * 136497, True, True, 2)
    assert not count_only(2 * 10, False, True, 4)
    # the fold: 16 warps x 16 segments per round
    assert fold_warps(256) == 16 and fold_warps(17) == 2 and fold_warps(1) == 1


def test_segment_cuts():
    assert segments(0, 0) == [] and segments(5, 6) == [(5, 6)]
    assert segments(1000, 3000) == [(1000, 1024), (1024, 2048), (2048, 3000)]
    assert segments(SEG, 2 * SEG) == [(SEG, 2 * SEG)]


# ------------------------------------------------------------------ reference association
def seq_sum(x, axis=0):
    """0.0 + x[0] + x[1] + ... along axis 0, in order (np.add.accumulate is sequential; np.sum is pairwise)."""
    x = np.asarray(x, dtype=np.float64)
    if x.shape[0] == 0:
        return np.zeros(x.shape[1:])
    return np.add.accumulate(np.concatenate([np.zeros((1,) + x.shape[1:]), x]), axis=0)[-1]


def fold(parts):
    """fm_k_wc_fold: 16-segment chunks counted from the window's first segment, each 0.0 + s0 + s1 + ..., then
    0.0 + c0 + c1 + ...; parts [n_seg, ...]."""
    parts = np.asarray(parts, dtype=np.float64)
    chunks = [seq_sum(parts[c:c + FOLD_CHUNK]) for c in range(0, parts.shape[0], FOLD_CHUNK)]
    return seq_sum(np.array(chunks).reshape((len(chunks),) + parts.shape[1:]))


def test_reference_association_is_sequential():
    """seq_sum adds in order (a pairwise or reordered sum gives a different double on this input), and fold groups
    exactly 16 segments per chunk."""
    x = np.array([1.0, 2.0 ** 53, 1.0, -(2.0 ** 53), 1.0, 1.0])
    loop = 0.0
    for v in x:
        loop += v
    assert seq_sum(x) == loop == 2.0 and float(np.sum(x[[1, 3, 0, 2, 4, 5]])) != loop
    y = np.tile(x[:, None], (1, 3))
    assert np.array_equal(seq_sum(y), np.full(3, 2.0))
    parts = np.zeros(18)
    parts[0], parts[15], parts[16], parts[17] = 2.0 ** 53, 1.0, 1.0, 1.0
    # chunk 0 = 2^53 + 1 -> 2^53, chunk 1 = 1 + 1 = 2: 2^53 + 2; one sequential pass loses every 1
    assert fold(parts) == 2.0 ** 53 + 2 and seq_sum(parts) == 2.0 ** 53


def gamma(k):
    return (k * EPS) / (1.0 - k * EPS)


def test_kernel_rewrites_of_the_size_terms_are_exact():
    """fm_wc_pair_site replaces the reference's (d1^2 + d2^2) / (2 n_bar n_bar) by 2 d1^2 / (nsd n_bar) and keeps
    1 - c^2 for the a-denominator: equal bit for bit for every pair with n_i, n_j <= 2048, and 1 - c^2 never has the
    all-ones significand fm_recip_rn cannot round."""
    n1, n2 = np.meshgrid(np.arange(1, 2049, dtype=np.float64), np.arange(1, 2049, dtype=np.float64))
    n1, n2 = n1.ravel(), n2.ravel()
    nsd = n1 + n2
    n_bar = nsd / 2.0
    d1, d2 = n1 - n_bar, n2 - n_bar
    ref = (0.0 + d1 * d1 + d2 * d2) / (2.0 * n_bar * n_bar)
    ker = (2.0 * (d1 * d1)) / (nsd * n_bar)
    assert np.array_equal(ref.view(np.uint64), ker.view(np.uint64))
    aden = 1.0 - ker
    assert np.array_equal(aden, 1.0 - ref / 1.0)
    mant = aden.view(np.uint64) & np.uint64((1 << 52) - 1)
    assert not np.any(mant == np.uint64((1 << 52) - 1))


# ------------------------------------------------------------------ cohorts
def make_genotypes(case, sms):
    """int8 [V, S, 2] with both sides of a sample missing together, the membership (left, right) and the edge rows."""
    from tests.synth import make_cohort
    from tests.test_gpu_parity import make_multi_cohort
    V, G, S = case.n_sites(sms), case.G, case.S
    if case.max_allele == 1:
        g, pos, _ = make_cohort(V, S, n_pops=max(G, 1), sigma=0.08, missing_rate=case.missing, seed=case.seed)
    else:
        g, pos = make_multi_cohort(V, S, case.max_allele, case.missing, seed=case.seed)
    g[:, :, 1][g[:, :, 0] < 0] = -1
    g[:, :, 0][g[:, :, 1] < 0] = -1
    left = np.full(S, UNG, dtype=np.uint16)
    right = np.full(S, UNG, dtype=np.uint16)
    s = 0
    split = case.special and G >= 2
    if split:  # sample 0: sides in groups 0 and 1; sample 1: one side in group 1, the other in no group
        left[0], right[0], left[1] = 0, 1, 1
        s = 2
    members = []
    for grp, k in enumerate(case.sizes):
        members.append(np.arange(s, s + k))
        left[s:s + k] = grp
        right[s:s + k] = grp
        s += k
    ungrouped = np.arange(s, S)
    if split:
        lo, hi = case.bounds(sms)
        rows = edge_rows(g, case, members, ungrouped, lo, hi)
    else:
        rows = {}
    return g, pos, left, right, rows


def edge_rows(g, case, members, ungrouped, lo, hi):
    """Rows that hit distinct kernel branches, placed at the start of the region and in its last segment."""
    top = case.max_allele
    where = {}
    names = ["ungrouped-only", "one-group", "groups-monomorphic", "nsum2", "nsum3", "full-call"]
    for k, name in enumerate(names):
        for r in (lo + 1 + k, hi - 2 - 2 * k):
            row = np.full(g.shape[1:], -1, dtype=np.int8)
            if name == "ungrouped-only":     # overall state 2 with data, no pair data
                row[ungrouped, 0], row[ungrouped, 1] = 0, min(1, top)
            elif name == "one-group":        # fewer than two groups with data
                m = members[0] if len(members[0]) else members[1]
                row[m, 0], row[m, 1] = 0, top
            elif name == "groups-monomorphic":
                for grp, m in enumerate(members):
                    row[m] = grp % (top + 1)
                row[0] = (0, 1 % (top + 1))
                row[1] = (1 % (top + 1), 0)
                row[ungrouped] = 0
            elif name == "nsum2":            # n_0 = n_1 = 1: n_bar - 1 < 1e-9
                row[0] = (0, top)
            elif name == "nsum3":            # n_0 = 1, n_1 = 2: the smallest polymorphic pair
                row[0] = (0, top)
                row[1] = (top, 0)
            else:                            # every sample called: n_i + n_j reaches the table's last entry
                rng = np.random.default_rng(r)
                row = rng.integers(0, top + 1, size=row.shape).astype(np.int8)
            g[r] = row
            where[r] = name
    return where


def numpy_sizes(g, left, right, G):
    """Called haplotypes per group at every site, straight from the genotype array (0 where nothing is called)."""
    called = (g[:, :, 0] >= 0).astype(np.float64)
    M = np.zeros((g.shape[1], max(G, 1)))
    for side in (left, right):
        ok = side != UNG
        np.add.at(M, (np.nonzero(ok)[0], side[ok].astype(np.int64)), 1.0)
    return np.rint(called @ M).astype(np.int64)[:, :G]


# ------------------------------------------------------------------ device handles
def _L():
    from ferromic_b200 import _lib
    return _lib


class Partition:
    """One count producer's partition of a cohort (released with the matrix)."""

    def __init__(self, form, g, pos, left, right, G, max_allele):
        from ferromic_b200.api import _Matrix
        L = _L()
        miss = g < 0
        alle = np.where(miss, 0, g).astype(np.uint8)
        self.m, self.ph = None, C.c_void_p()
        if form == "stream":
            self.m = _Matrix.ingest(alle, miss, pos, [], partitions=[(left, right, G)], always_bitmap=True)
            self.ph = self.m.partitions[0]
            return
        if form == "inband":
            self.m = _Matrix.from_int8(g, pos, max_allele, ingest="u8")
        elif form == "u8-nobitmap":
            assert not miss.any()
            self.m = _Matrix(alle, None, pos, max_allele=max_allele, ingest="u8")
        else:
            self.m = _Matrix(alle, miss, pos, max_allele=max_allele, always_bitmap=True, ingest=form)
            assert self.m.ingest_mode == form
        L.check(L.lib().fm_partition_create(self.m.handle, left.ctypes.data, right.ctypes.data, len(left), G,
                                            C.byref(self.ph)))
        self.own = True

    def release(self):
        if getattr(self, "own", False) and self.ph:
            _L().lib().fm_partition_release(self.ph)
        self.ph = None
        self.m = None


def device_sites(ph, pos, lo, hi, G):
    L = _L()
    P, ns = n_pairs(G), hi - lo
    est = L.FstEstimateC()
    pairs = (L.FstEstimateC * max(P, 1))()
    present = np.zeros(max(P, 1), dtype=np.uint8)
    out = dict(pos=np.zeros(ns, dtype=np.int64), state=np.zeros(ns, dtype=np.int32), a=np.zeros(ns), b=np.zeros(ns),
               sizes=np.zeros((ns, max(G, 1)), dtype=np.uint32), pa=np.zeros((ns, max(P, 1))),
               pb=np.zeros((ns, max(P, 1))))
    n = C.c_size_t()
    L.check(L.lib().fm_wc_fst(ph, int(pos[lo]), int(pos[hi - 1]), C.byref(est), pairs, present.ctypes.data,
                              out["pos"].ctypes.data, out["state"].ctypes.data, out["a"].ctypes.data,
                              out["b"].ctypes.data, out["sizes"].ctypes.data,
                              out["pa"].ctypes.data if P else None, out["pb"].ctypes.data if P else None, ns,
                              C.byref(n)))
    assert n.value == ns
    return out


def device_region(ph, pos, lo, hi, G):
    """fm_wc_fst over [lo, hi) without per-site outputs: (overall, pairs, pair_present)."""
    L = _L()
    P = n_pairs(G)
    est = L.FstEstimateC()
    pairs = (L.FstEstimateC * max(P, 1))()
    present = np.zeros(max(P, 1), dtype=np.uint8)
    n = C.c_size_t()
    L.check(L.lib().fm_wc_fst(ph, int(pos[lo]), int(pos[hi - 1]), C.byref(est), pairs, present.ctypes.data,
                              None, None, None, None, None, None, None, 0, C.byref(n)))
    return est, [pairs[k] for k in range(P)], present[:P]


def window_sums(ph, pos, windows, G):
    """fm_wc_window_sums over site-index windows [lo, hi) (None = an empty window), one call."""
    L = _L()
    P, nw = n_pairs(G), len(windows)
    wp = np.zeros((nw, 2), dtype=np.int64)
    for i, w in enumerate(windows):
        wp[i] = (pos[10], pos[10] - 1) if w is None else (pos[w[0]], pos[w[1] - 1])
    o = dict(nvar=np.zeros(nw, dtype=np.uint64), a=np.zeros(nw), b=np.zeros(nw), n=np.zeros(nw, dtype=np.uint64),
             pa=np.zeros((nw, max(P, 1))), pb=np.zeros((nw, max(P, 1))), pn=np.zeros((nw, max(P, 1)), dtype=np.uint64))
    L.check(L.lib().fm_wc_window_sums(ph, wp.ctypes.data, nw, o["nvar"].ctypes.data, o["a"].ctypes.data,
                                      o["b"].ctypes.data, o["n"].ctypes.data, o["pa"].ctypes.data,
                                      o["pb"].ctypes.data, o["pn"].ctypes.data))
    return o


# ------------------------------------------------------------------ comparisons
def bits(x):
    """uint64 image of x with both zeros as +0 (the sign of a zero sum is not part of the estimator)."""
    return (np.asarray(x, dtype=np.float64) + 0.0).view(np.uint64)


def assert_bits(got, ref, what):
    nan = np.isnan(ref)
    assert np.array_equal(np.isnan(got), nan), (what, np.argwhere(np.isnan(got) != nan)[:5])
    bad = bits(got[~nan]) != bits(ref[~nan])
    assert not bad.any(), (what, int(bad.sum()), got[~nan][bad][:4], ref[~nan][bad][:4])


class Sums:
    """Per-segment totals of one window (in segment order) and the exact-sum bookkeeping of the same values."""

    def __init__(self, P):
        self.P = P
        self.seg_o, self.seg_on, self.seg_p, self.seg_pn = [], [], [], []
        self.fs_o, self.fs_p = [], []        # per-block fsums: [2] and [P][2]
        self.abs_o, self.abs_p = np.zeros(2), np.zeros((max(P, 1), 2))

    def add_block(self, lo, hi, b0, state, a, b, pstate, pa, pb):
        """Per-site values of sites [b0, b0 + len(a)) of the window [lo, hi); the block holds whole segments."""
        ov = state != 3
        xo = np.stack([np.where(ov, a, 0.0), np.where(ov, b, 0.0)], axis=1)
        if self.P:
            pv = (pstate >= 0) & (pstate <= 2)
            xp = np.stack([np.where(pv, pa, 0.0), np.where(pv, pb, 0.0)], axis=2)
        for s0, s1 in segments(max(lo, b0), min(hi, b0 + len(a))):
            i0, i1 = s0 - b0, s1 - b0
            self.seg_o.append(seq_sum(xo[i0:i1]))
            self.seg_on.append(int(ov[i0:i1].sum()))
            if self.P:
                self.seg_p.append(seq_sum(xp[i0:i1]))
                self.seg_pn.append(pv[i0:i1].sum(axis=0))
        self.fs_o.append([math.fsum(xo[:, k]) for k in (0, 1)])
        self.abs_o += np.abs(xo).sum(axis=0)
        if self.P:
            self.fs_p.append({p: [math.fsum(xp[:, p, k]) for k in (0, 1)] for p in fsum_columns(self.P)})
            self.abs_p += np.abs(xp).sum(axis=0)

    def totals(self):
        t = dict(o=fold(self.seg_o) if self.seg_o else np.zeros(2), on=sum(self.seg_on))
        if self.P:
            t["p"] = fold(self.seg_p) if self.seg_p else np.zeros((self.P, 2))
            t["pn"] = np.sum(self.seg_pn, axis=0) if self.seg_pn else np.zeros(self.P, dtype=np.int64)
        return t


def fsum_columns(P):
    """Pair columns checked against the exact sum: all of them up to 64, else 64 spread over the range (every column
    is checked bit for bit against the fold)."""
    return range(P) if P <= 64 else sorted(set(np.linspace(0, P - 1, 64).astype(int).tolist()))


def assert_exact_bound(dev, fsums, sum_abs, k):
    """|dev - exact| <= gamma_{k-1} sum|x|; the exact sum is an fsum of per-block fsums, itself within eps sum|x|."""
    ref = math.fsum(fsums)
    bound = (gamma(max(k - 1, 0)) + 2 * EPS) * sum_abs * (1 + 1e-6)
    assert abs(dev - ref) <= bound, (dev, ref, bound, k)


def fst_state(a, b):
    from oracle import pyoracle as orc
    return orc.STATE_NAMES.index(orc.fst_estimate_from_components(a, b)["state"])


def assert_estimate(e, a, b, n, sites_if_none):
    if n == 0:
        assert (e.state, e.sites) == (3, sites_if_none) and (e.sum_a, e.sum_b) == (0.0, 0.0)
        return
    st = fst_state(a, b)
    assert (e.state, e.sites) == (st, n) and bits(e.sum_a) == bits(a) and bits(e.sum_b) == bits(b)
    if st == 0:
        assert bits(e.value) == bits(a / (a + b))


def block_edges(lo, hi, P):
    """Blocks of whole segments (cut at multiples of a multiple of SEG) with at most ~100 MB of per-pair arrays
    alive (oracle and device a / b, the oracle's pair states)."""
    per = max(1, 100_000_000 // (max(P, 1) * 8 * 5 * SEG)) * SEG
    out, b = [], lo
    while b < hi:
        e = min(hi, (b // per + 1) * per)
        out.append((b, e))
        b = e
    return out


def compare_case(case, sms, keep_sites=False):
    """Every form of one case against the oracle, block by block; returns the reference sums and, with keep_sites,
    the per-site reference values of the region."""
    from oracle import pyoracle as orc
    G, P = case.G, n_pairs(case.G)
    g, pos, left, right, rows = make_genotypes(case, sms)
    lo, hi = case.bounds(sms)
    parts = [Partition(f, g, pos, left, right, G, case.max_allele) for f in case.forms]
    try:
        sums = Sums(P)
        kept = dict(state=[], a=[], b=[], pstate=[], pa=[], pb=[])
        hit = set()
        for b0, b1 in block_edges(lo, hi, P):
            vs, _ = orc.from_numpy(g[b0:b1], pos[b0:b1])
            ref = orc.wc_fst(vs, left, right, G, (int(pos[b0]), int(pos[b1 - 1])), want_pairs=P > 0)
            assert ref["n_sites"] == b1 - b0
            sizes = numpy_sizes(g[b0:b1], left, right, G)
            anyc = (g[b0:b1, :, 0] >= 0).any(axis=1)
            exp_sizes = np.where(anyc[:, None], sizes, 0)
            assert np.array_equal(ref["pop_sizes"].astype(np.int64), exp_sizes)
            pstate = ref.get("pair_state")
            if P:
                nan = ~((pstate >= 0) & (pstate <= 2))
                rpa = np.where(nan, np.nan, ref["pair_a"])
                rpb = np.where(nan, np.nan, ref["pair_b"])
            for part in parts:
                d = device_sites(part.ph, pos, b0, b1, G)
                assert np.array_equal(d["pos"], pos[b0:b1] + 1)
                assert np.array_equal(d["state"], ref["state"]), (case.name, part)
                assert_bits(d["a"], ref["a"], "site a")
                assert_bits(d["b"], ref["b"], "site b")
                assert np.array_equal(d["sizes"][:, :G].astype(np.int64), exp_sizes)
                if P:
                    assert_bits(d["pa"][:, :P], rpa, "pair a")
                    assert_bits(d["pb"][:, :P], rpb, "pair b")
            sums.add_block(lo, hi, b0, ref["state"], ref["a"], ref["b"], pstate,
                           ref.get("pair_a"), ref.get("pair_b"))
            if keep_sites:
                for k, v in (("state", ref["state"]), ("a", ref["a"]), ("b", ref["b"]), ("pstate", pstate),
                             ("pa", ref.get("pair_a")), ("pb", ref.get("pair_b"))):
                    kept[k].append(v)
            for r, name in rows.items():
                if b0 <= r < b1:
                    hit.add(name)
                    if name == "ungrouped-only":
                        assert ref["state"][r - b0] == 2 and (not P or (pstate[r - b0] == -1).all() or
                                                              (pstate[r - b0] == 3).all())
                    if name == "nsum2" and P:
                        assert pstate[r - b0, 0] == 2 and ref["pair_a"][r - b0, 0] == 0.0
        if rows:
            assert hit == set(rows.values()), hit
        t = sums.totals()
        for part in parts:
            w = window_sums(part.ph, pos, [(lo, hi)], G)
            assert int(w["nvar"][0]) == hi - lo and int(w["n"][0]) == t["on"]
            assert bits(w["a"][0]) == bits(t["o"][0]) and bits(w["b"][0]) == bits(t["o"][1]), case.name
            est, pest, present = device_region(part.ph, pos, lo, hi, G)
            assert_estimate(est, t["o"][0], t["o"][1], t["on"], hi - lo)
            assert_exact_bound(w["a"][0], [f[0] for f in sums.fs_o], sums.abs_o[0], t["on"])
            assert_exact_bound(w["b"][0], [f[1] for f in sums.fs_o], sums.abs_o[1], t["on"])
            if P:
                assert np.array_equal(w["pn"][0, :P].astype(np.int64), t["pn"])
                assert np.array_equal(bits(w["pa"][0, :P]), bits(t["p"][:, 0]))
                assert np.array_equal(bits(w["pb"][0, :P]), bits(t["p"][:, 1]))
                assert np.all(present == (t["on"] > 0))
                for k in range(P):
                    if t["on"] == 0:
                        continue
                    if t["pn"][k] == 0:
                        assert (pest[k].state, pest[k].sites) == (3, t["on"])
                    else:
                        assert_estimate(pest[k], t["p"][k, 0], t["p"][k, 1], int(t["pn"][k]), 0)
                for k in fsum_columns(P):
                    for j in (0, 1):
                        assert_exact_bound(w["pa" if j == 0 else "pb"][0, k], [f[k][j] for f in sums.fs_p],
                                           sums.abs_p[k, j], int(t["pn"][k]))
        if keep_sites:
            kept = {k: (np.concatenate(v) if v and v[0] is not None else None) for k, v in kept.items()}
        return g, pos, left, right, parts, kept
    except BaseException:
        for p in parts:
            p.release()
        raise


def release(parts):
    for p in parts:
        p.release()


def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# ------------------------------------------------------------------ GPU tests
@pytest.mark.gpu
@pytest.mark.parametrize("name", [c.name for c in TABLE if c.name != "multi-A4-many-segments"])
def test_case_against_oracle(name):
    """Per-site values of every count producer bit for bit against the oracle, region totals against the fixed
    association and the exact sum, region estimates through the state ladder."""
    case = BY_NAME[name]
    sms = sm_count()
    lo, hi = case.bounds(sms)
    if name == "bi-G79-tasks":
        assert len(segments(lo, hi)) * pc_chunks(79) > 3 * pc_blocks_per_sm_bound(79) * sms
    *_, parts, _ = compare_case(case, sms)
    release(parts)


def check_windows(case, windows, sms):
    G, P = case.G, n_pairs(case.G)
    g, pos, left, right, parts, ref = compare_case(case, sms, keep_sites=True)
    try:
        lo0, _ = case.bounds(sms)
        for part in parts:
            w = window_sums(part.ph, pos, windows, G)
            assert fold_warps(max(len(segments(*x)) for x in windows if x)) == FOLD_MAX_WARPS
            for i, win in enumerate(windows):
                if win is None:
                    assert (int(w["nvar"][i]), int(w["n"][i]), w["a"][i], w["b"][i]) == (0, 0, 0.0, 0.0)
                    if P:
                        assert not w["pn"][i, :P].any() and not w["pa"][i, :P].any()
                    continue
                s = Sums(P)
                a0, a1 = win[0] - lo0, win[1] - lo0
                s.add_block(win[0], win[1], win[0], ref["state"][a0:a1], ref["a"][a0:a1], ref["b"][a0:a1],
                            None if not P else ref["pstate"][a0:a1], None if not P else ref["pa"][a0:a1],
                            None if not P else ref["pb"][a0:a1])
                t = s.totals()
                assert int(w["nvar"][i]) == win[1] - win[0] and int(w["n"][i]) == t["on"], win
                assert bits(w["a"][i]) == bits(t["o"][0]) and bits(w["b"][i]) == bits(t["o"][1]), win
                assert_exact_bound(w["a"][i], s.fs_o[0][:1], s.abs_o[0], t["on"])
                if P:
                    assert np.array_equal(w["pn"][i, :P].astype(np.int64), t["pn"]), win
                    assert np.array_equal(bits(w["pa"][i, :P]), bits(t["p"][:, 0])), win
                    assert np.array_equal(bits(w["pb"][i, :P]), bits(t["p"][:, 1])), win
    finally:
        release(parts)


@pytest.mark.gpu
def test_windows_biallelic():
    """One fm_wc_window_sums call: a 300k-site window (second fold round), 16 / 17 / 18 segments, an aligned
    segment, one-site, empty, overlapping and mid-stage windows -- totals bit for bit against the fold."""
    check_windows(WINDOW_CASE, window_list(WINDOW_CASE.V), sm_count())


@pytest.mark.gpu
def test_windows_multi_allelic():
    """The same window kinds on a multi-allelic partition whose segments outnumber 8 CTAs per SM."""
    case = BY_NAME["multi-A4-many-segments"]
    sms = sm_count()
    lo, hi = case.bounds(sms)
    assert len(segments(lo, hi)) > 8 * sms and multi_blocks(len(segments(lo, hi)), sms) == 8 * sms
    wins = [w for w in window_list(WINDOW_CASE.V) if w is None or (w[0] >= lo and w[1] <= hi)] + [(lo, hi)]
    check_windows(case, wins, sms)


@pytest.mark.gpu
@pytest.mark.parametrize("max_allele,G", REFUSED)
def test_population_limit_refused_without_a_launch(max_allele, G):
    """One population above each limit: FM_ERR_UNSUPPORTED before any K4 kernel is launched."""
    L = _L()
    case = Case("refused", max_allele, (2,) * G, 300, (0, 300), seed=60 + G)
    g, pos, left, right, _ = make_genotypes(case, B200_SMS)
    part = Partition("u8", g, pos, left, right, G, max_allele)
    try:
        L.check(L.lib().fm_timings_reset())
        est = L.FstEstimateC()
        pairs = (L.FstEstimateC * n_pairs(G))()
        n = C.c_size_t()
        st = L.lib().fm_wc_fst(part.ph, int(pos[0]), int(pos[-1]), C.byref(est), pairs, None, None, None, None,
                               None, None, None, None, 0, C.byref(n))
        assert st == L.FM_ERR_UNSUPPORTED, L.lib().fm_last_error()
        t = L.Timings()
        L.check(L.lib().fm_timings_get(C.byref(t)))
        assert t.kernel_launches == 0
        # the admitted neighbour runs
        ok = Case("admitted", max_allele, (2,) * (G - 1), 300, (0, 300), seed=60 + G)
        g2, pos2, l2, r2, _ = make_genotypes(ok, B200_SMS)
        p2 = Partition("u8", g2, pos2, l2, r2, G - 1, max_allele)
        try:
            device_region(p2.ph, pos2, 0, 300, G - 1)
        finally:
            p2.release()
    finally:
        part.release()


def knob_outputs():
    """Per-site values and region totals of the KNOB_CASES in this process (its FM_WC_* settings)."""
    out = {}
    for name in KNOB_CASES:
        case = BY_NAME[name]
        g, pos, left, right, _ = make_genotypes(case, B200_SMS)
        lo, hi = case.bounds(B200_SMS)
        part = Partition("u8", g, pos, left, right, case.G, case.max_allele)
        try:
            d = device_sites(part.ph, pos, lo, hi, case.G)
            w = window_sums(part.ph, pos, [(lo, hi)], case.G)
        finally:
            part.release()
        for k, v in list(d.items()) + list(w.items()):
            out[f"{name}.{k}"] = v
    return out


@pytest.mark.gpu
def test_tuning_knobs_give_identical_bits(tmp_path):
    """FM_WC_SITES_PER_STEP = 2 (fm_k_wc_pairs_pc<2>, last segment of odd length) and FM_WC_KP = 4 (4 pair warps
    with 4 pairs per lane on 30 populations) in a separate process: every per-site value and total bit-identical
    to this process's defaults (which test_case_against_oracle ties to the oracle)."""
    assert not any(k in os.environ for k in KNOB_ENV)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dst = tmp_path / "knobs.npz"
    code = ("import sys, numpy as np; sys.path.insert(0, sys.argv[1]); "
            "import tests.test_gpu_wc_geometry as T; np.savez(sys.argv[2], **T.knob_outputs())")
    r = subprocess.run([sys.executable, "-c", code, root, str(dst)], env={**os.environ, **KNOB_ENV}, cwd=root,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    mine = knob_outputs()
    theirs = np.load(dst)
    assert set(theirs.files) == set(mine)
    for k, v in mine.items():
        u = theirs[k]
        if v.dtype == np.float64:
            nan = np.isnan(v)
            assert np.array_equal(nan, np.isnan(u)) and np.array_equal(v[~nan].view(np.uint64),
                                                                       u[~nan].view(np.uint64)), k
        else:
            assert np.array_equal(v, u), k
