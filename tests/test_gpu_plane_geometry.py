"""Every plane-pass geometry against an exact count reference.

The host picks the plane-pass kernel shape from the group widths of a launch (row pass LG 0-4 with 1-16 rounds of
sites per lane, the tail layout, the column-chunked pass with one or more chunks, inline or uploaded segment tables,
Hudson pair units).  This file restates those host rules in Python, lists one case per geometry class in a table
whose coverage a CPU test asserts, and runs every case on the GPU against a plain numpy reference:

  * counts: per-site alt and called of a haplotype list with the library's group semantics (duplicates count once,
    out-of-range samples are dropped, side 1 is dropped at ploidy 1), exact integers;
  * per-site pi / theta: recomputed with the kernels' order of operations from the same per-n tables alloc_group
    builds, so the device tracks must equal them bit for bit; the restatement itself is anchored to the exact values
    (fractions.Fraction for pi, 60-digit decimals for the harmonic numbers of theta);
  * region sums: the exact sum over the (n, a) histogram, with a bound of a few ulps per term.
"""
import ctypes as C
import decimal
import math
from fractions import Fraction

import numpy as np
import pytest

from oracle import pyoracle as orc

EPS = 2.0 ** -53

# ------------------------------------------------------------------ host geometry rules, restated
WARP_SMEM = 14 * 1024   # fm_kernels.cuh:22 kWarpSmemBytes
WARPS_PER_CTA = 16      # fm_kernels.cuh:21
MAX_STAGES = 6          # fm_kernels.cuh:23
STEP_TARGET = 7 * 1024  # fm_kernels.cuh:24 kStepBytesTarget
MAX_SEQ = 4             # fm_kernels.cuh:945 kMaxSeq
CHUNK_WARPS = 8         # fm_gpu.cu:744 (FM_CHUNK_WARPS default)
CHUNK_STEP = 14336      # fm_gpu.cu:745 (FM_CHUNK_STEP_BYTES default)


def repack_warp_smem(stride, packed, bitmap):
    """fm_gpu.cu:1652 repack_warp_smem: shared memory one warp of the staged K1 needs for a row."""
    row_buf = 0 if packed else ((stride + 15) & ~15) + 32
    bit_buf = ((stride + 63) // 64 + 2) * 8 if (not packed and bitmap) else 0
    cnt_buf = 2 * ((stride + 31) // 32 + 1) * 4 + (((stride + 127) // 128) * 4 + 4) * 4
    return (row_buf + bit_buf + cnt_buf + 15) & ~15


def row_fits(stride, packed, bitmap):
    """fm_gpu.cu:1663-1664 row_fits_smem (in-band u8 has no bitmap slice)."""
    return repack_warp_smem(stride, packed, bitmap) <= (100 * 1024 if packed else 24 * 1024)


def layout(n, fits):
    """fm_gpu.cu:1684-1699 alloc_group: (wq, tw) of a biallelic plane group of n haplotypes."""
    wq = max(1, (n + 127) // 128)
    tail_bits = n % 128
    tw = (tail_bits + 31) // 32
    if fits and n >= 128 and 0 < tail_bits <= 96 and (16 - 4 * tw) * 50 >= 16 * wq:
        return n // 128, tw
    return wq, 0


def row_lanes_log2(wq):
    """fm_gpu.cu:733 row_lanes_log2 (5 = column-chunked pass)."""
    lg = 0
    while (1 << lg) < min(wq, 8):
        lg += 1
    while lg < 5 and wq * 16 * (32 >> lg) * 2 > WARP_SMEM:
        lg += 1
    return lg


def rounds_of(wq, lg):
    """fm_gpu.cu:852-856 plan_rows: rounds of (32 >> lg) sites per pipeline step."""
    round_bytes = wq * 16 * (32 >> lg)
    r = 1
    while r * 2 <= (1 << lg) and round_bytes * r * 2 <= STEP_TARGET:
        r *= 2
    return r


def chunk_geom(wq):
    """fm_gpu.cu:743 make_geom: (warps, n_chunks, chunk words, words of the last chunk)."""
    row_bytes = wq * 16
    warps = CHUNK_WARPS if row_bytes * 2 > WARP_SMEM else WARPS_PER_CTA
    warp_smem = (WARPS_PER_CTA * WARP_SMEM // warps) & ~127
    cq, n_chunks = wq, 1
    if row_bytes * 2 > warp_smem:
        cq = max(1, CHUNK_STEP // 16)
        n_chunks = (wq + cq - 1) // cq
    return warps, n_chunks, cq, wq - (n_chunks - 1) * cq


# u8 + bitmap rows of 8160 diploid samples are the widest the staged K1 takes (repack_warp_smem <= 24 KB)
NARROW_S, NARROW_V = 8160, 8192 + 161
WIDE_S, WIDE_V = 114752, 97
NARROW_SIZES = (1, 2, 31, 33, 127, 128, 129, 200, 224, 225, 384, 480, 640, 1473, 1601, 3105, 3233, 3463, 4609, 4737,
                5008, 10000, 14336, 14337, 16320)
WIDE_SIZES = (129, 16320, 28673, 57344, 57345, 114688, 114689, 229376, 229504)
COHORTS = {  # name: (row stride, packed rows, bitmap)
    "narrow": (2 * NARROW_S, False, True),
    "wide-u8": (2 * WIDE_S, False, True),
    "wide-packed": (2 * WIDE_S, True, True),
}
MULTI_MIXES = ((1, 129, 16320), (2, 480, 3463, 5008, 10000))
BATCHES = ((31, 224, 1473, 14336), (1, 33, 640, 3105, 4609, 14337))
PAIRS = ((129, 16320), (2, 14337), (480, 3463))
WIDE_PAIR = (114689, 229504)

# one entry per case: (cohort, launch, group sizes); "one" = a single group's pass, "multi" / "batch" = one row
# launch over several groups, "pair" = the Hudson pair units of one row launch (or two chunked passes)
TABLE = ([("narrow", "one", (n,)) for n in NARROW_SIZES] +
         [("narrow", "multi", mix) for mix in MULTI_MIXES] +
         [("narrow", "batch", b) for b in BATCHES] +
         [("narrow", "pair", p) for p in PAIRS] +
         [(c, "one", (n,)) for c in ("wide-u8", "wide-packed") for n in WIDE_SIZES] +
         [("wide-u8", "pair", WIDE_PAIR), ("wide-packed", "pair", (129, 16320))])


def classes(entry):
    """Geometry classes one table entry reaches."""
    cohort, launch, sizes = entry
    stride, packed, bitmap = COHORTS[cohort]
    fits = row_fits(stride, packed, bitmap)
    lays = [layout(n, fits) for n in sizes]
    out = set()
    for n, (wq, tw) in zip(sizes, lays):
        out.add(f"tw{tw}")
        bits = n % 128
        if fits and n >= 128 and 0 < bits <= 96 and tw == 0:
            out.add(f"shrink-refused-tw{(bits + 31) // 32}")
    max_wq = max(wq for wq, _ in lays)
    lg = row_lanes_log2(max_wq)
    if lg == 5:
        for wq, _ in lays:
            warps, n_chunks, _, last = chunk_geom(wq)
            out.add(f"chunked-{warps}w-{n_chunks}c")
            if n_chunks > 1 and last == 1:
                out.add("last-chunk-1-word")
        return out
    out.add(f"LG{lg}")
    for wq, _ in lays:
        out.add(f"rounds{rounds_of(wq, lg)}")
        if wq == 1 and lg == 4:
            out.add("1-word-at-LG4")
    out.add("inline-table" if len(sizes) <= MAX_SEQ else "uploaded-table")
    if launch == "pair" and lays[0] != lays[1]:
        out.add("pair-mismatched")
        if any(tw for _, tw in lays) and lg == 4:
            out.add("pair-tail-with-LG4")
    return out


REQUIRED = ({f"LG{i}" for i in range(5)} | {f"rounds{r}" for r in (1, 2, 4, 8, 16)} | {f"tw{t}" for t in range(4)} |
            {f"shrink-refused-tw{t}" for t in (1, 2, 3)} | {"1-word-at-LG4", "inline-table", "uploaded-table",
             "pair-mismatched", "pair-tail-with-LG4", "chunked-16w-1c", "chunked-8w-1c", "chunked-8w-2c",
             "chunked-8w-3c", "last-chunk-1-word"})


def test_table_reaches_every_geometry_class():
    reached = set().union(*(classes(e) for e in TABLE))
    assert REQUIRED <= reached, f"classes no case reaches: {sorted(REQUIRED - reached)}"
    # both sides of each row-shrink boundary of the tail rule
    fits = row_fits(*COHORTS["narrow"])
    assert fits and not row_fits(2 * (NARROW_S + 1), False, True)
    for inside, outside in ((1473, 1601), (3105, 3233), (4609, 4737)):
        assert layout(inside, fits)[1] > 0 and layout(outside, fits)[1] == 0
        assert (inside % 128 + 31) // 32 == (outside % 128 + 31) // 32
    # the wide u8 rows are repacked by fm_k_repack: no tail layout; packed rows keep it
    assert layout(129, row_fits(*COHORTS["wide-u8"])) == (2, 0)
    assert layout(129, row_fits(*COHORTS["wide-packed"])) == (1, 1)


# ------------------------------------------------------------------ plain reference
_TAB = {}


def tables(n_max):
    """The per-n tables of alloc_group (fm_gpu.cu:1716-1727): 1/k, k/(k-1), 1/H_{k-1} with H summed forward."""
    if _TAB.get("n", -1) < n_max:
        tn = n_max + 1
        inv, scale, theta = np.zeros(tn), np.zeros(tn), np.zeros(tn)
        h = 0.0
        for k in range(1, tn):
            kd = float(k)
            inv[k] = 1.0 / kd
            scale[k] = kd / (kd - 1.0) if k > 1 else math.inf  # IEEE 1/0 on the host
            theta[k] = 1.0 / h if h > 0.0 else 0.0
            h += 1.0 / kd
        _TAB.update(n=n_max, inv=inv, scale=scale, theta=theta)
    return _TAB["inv"], _TAB["scale"], _TAB["theta"]


def member_cols(haps, S, P):
    """Sorted unique columns s * P + side of a haplotype list (DenseMembership::build semantics)."""
    cols = {int(s) * P + int(side) for s, side in haps if int(s) < S and (int(side) == 0 or P > 1)}
    return np.array(sorted(cols), dtype=np.int64)


def group_counts(data, called, col_lists, allele=None):
    """alt [V, G] and called [V, G] of every column list over u8 rows `data` [V, stride] with called mask `called`
    (None: every cell called).  alt counts cells with a non-zero allele, or == allele when given.  float32 products of
    0/1 matrices are exact below 2^24."""
    V, stride = data.shape
    M = np.zeros((stride, len(col_lists)), dtype=np.float32)
    for g, cols in enumerate(col_lists):
        M[cols, g] = 1.0
    alt = np.zeros((V, len(col_lists)), dtype=np.int64)
    cal = np.zeros((V, len(col_lists)), dtype=np.int64)
    step = max(1, (1 << 22) // max(stride, 1))
    for r0 in range(0, V, step):
        d = data[r0:r0 + step]
        a = (d != 0) if allele is None else (d == allele)
        if called is not None:
            ok = called[r0:r0 + step]
            a = a & ok
            cal[r0:r0 + step] = np.rint(ok.astype(np.float32) @ M)
        alt[r0:r0 + step] = np.rint(a.astype(np.float32) @ M)
    if called is None:
        cal[:] = np.array([len(c) for c in col_lists])
    return alt, cal


def site_pi(n, a):
    """Per-site pi in the kernels' order of operations (fm_div_site, fm_kernels.cuh:760-764); garbage where n < 2."""
    inv, scale, _ = tables(int(n.max(initial=1)))
    r = (n - a).astype(np.float64)
    af = a.astype(np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        return scale[n] * (1.0 - (r * r + af * af) * inv[n] * inv[n])


def ref_tracks(n, a, dropped):
    """calculate_per_site_diversity tracks: NaN where n < 2 or the site is masked / filtered."""
    _, _, theta = tables(int(n.max(initial=1)))
    bad = (n < 2) | dropped
    poly = (n >= 2) & (a > 0) & (a < n)
    pi = np.where(bad, np.nan, site_pi(n, a))
    th = np.where(bad, np.nan, np.where(poly, theta[n], 0.0))
    return pi, th


_CHECKED_PI, _CHECKED_N = set(), set()
_HARM = []


def exact_inv_harmonic(k):
    """1/H_{k-1} to 60 significant digits (far below one ulp of a double)."""
    ctx = decimal.Context(prec=60)
    while len(_HARM) <= k:
        _HARM.append(ctx.add(_HARM[-1], ctx.divide(1, len(_HARM))) if _HARM else decimal.Decimal(0))
    return ctx.divide(1, _HARM[k - 1])


def anchor(n, a):
    """The numpy restatement is within 16 eps of the exact pi and (n + 2) eps relative of the exact theta for every
    (n, a) pair that occurs -- so a restatement that drifts from the formula fails on its own."""
    ok = n >= 2
    pairs = set(zip(n[ok].tolist(), a[ok].tolist())) - _CHECKED_PI
    if pairs:
        pn = np.array([p[0] for p in pairs], dtype=np.int64)
        pa = np.array([p[1] for p in pairs], dtype=np.int64)
        got = site_pi(pn, pa)
        for k, al, g in zip(pn.tolist(), pa.tolist(), got.tolist()):
            exact = Fraction(2 * al * (k - al), k * (k - 1))
            assert abs(Fraction(g) - exact) <= Fraction(16) * Fraction(EPS), (k, al, g)
        _CHECKED_PI.update(pairs)
    _, _, theta = tables(int(n.max(initial=1)))
    for k in set(n[ok].tolist()) - _CHECKED_N:
        exact = exact_inv_harmonic(k)
        err = abs(decimal.Decimal(float(theta[k])) - exact)
        assert err <= decimal.Decimal((k + 2) * EPS) * exact, k
        _CHECKED_N.add(k)


def exact_pi_sum(n, a):
    """Exact sum of pi over sites with n >= 2 (pi = 2a(n-a) / (n(n-1))), as a Fraction."""
    ok = n >= 2
    nn, aa = n[ok].astype(np.int64), a[ok].astype(np.int64)
    keys, inv = np.unique(nn, return_inverse=True)
    num = np.zeros(len(keys), dtype=np.int64)
    np.add.at(num, inv, 2 * aa * (nn - aa))
    return sum((Fraction(int(s), int(k) * (int(k) - 1)) for s, k in zip(num, keys)), Fraction(0))


def assert_region_sum(dev, n, a):
    exact = exact_pi_sum(n, a)
    assert abs(Fraction(dev) - exact) <= Fraction(16 * EPS) * len(n) + Fraction(40 * EPS) * exact, (dev, float(exact))


def ref_scalars(n, a):
    return int(((n >= 2) & (a > 0) & (a < n)).sum()), int((n < 2).sum())


def random_haps(rng, S, P, n):
    """n distinct in-range haplotypes of an S x P cohort, shuffled, plus duplicates, out-of-range samples and (at
    ploidy 1) side-1 entries that the group must drop."""
    ids = rng.permutation(S * P)[:n]
    haps = [(int(c) // P, int(c) % P) for c in ids]
    extra = [haps[int(i)] for i in rng.integers(0, n, size=min(3, n))]
    extra += [(S + int(rng.integers(0, 40)), int(rng.integers(0, 2))), (S, 0)]
    if P == 1:
        extra += [(haps[0][0], 1), (int(rng.integers(0, S)), 1)]
    haps += extra
    order = rng.permutation(len(haps))
    return [haps[int(i)] for i in order]


def make_genotypes(V, S, seed, missing=0.02, P=2):
    """int8 [V, S, P] with per-cell missingness (-1), U-shaped site frequencies, some monomorphic and some
    all-missing sites; u8 data with alleles left under missing cells (the bitmap must win) and the missing mask."""
    rng = np.random.default_rng(seed)
    f = rng.beta(0.4, 0.4, size=V)
    f[rng.random(V) < 0.03] = 0.0
    f[rng.random(V) < 0.03] = 1.0
    g = (rng.random((V, S * P), dtype=np.float32) < f[:, None].astype(np.float32)).astype(np.int8)
    miss = rng.random((V, S * P), dtype=np.float32) < missing
    miss[rng.random(V) < 0.01] = True
    under = np.where(rng.random((V, S * P), dtype=np.float32) < 0.5, 1, 0).astype(np.uint8)
    data = np.where(miss, under, g).astype(np.uint8)
    g[miss] = -1
    pos = np.cumsum(rng.integers(1, 30, size=V, dtype=np.int64)) + 10
    return g.reshape(V, S, P), data.reshape(V, S, P), miss.reshape(V, S, P), pos


# ------------------------------------------------------------------ CPU self-tests of the reference
def test_numpy_counts_match_oracle_summary():
    """The numpy counts equal orc.build_summary of the C oracle: duplicates, out-of-range samples, ploidy 1,
    per-allele missingness and in-band missingness (the int8 form)."""
    rng = np.random.default_rng(7)
    for seed, (V, S, P, miss_rate) in enumerate([(67, 37, 2, 0.1), (70, 130, 2, 0.03), (33, 41, 1, 0.2),
                                                 (40, 64, 2, 0.0)]):
        g, data, miss, pos = make_genotypes(V, S, 100 + seed, missing=miss_rate, P=P)
        called = ~miss.reshape(V, -1)
        d = orc.Dense(data.reshape(-1), orc.pack_missing_bits(miss.reshape(-1)) if miss.any() else None, V, S, P, 1)
        lists = [random_haps(rng, S, P, n) for n in (1, 2, S // 2, S * P)]
        alt, cal = group_counts(data.reshape(V, -1), called if miss.any() else None,
                                [member_cols(h, S, P) for h in lists])
        # in-band form: the int8 cells alone carry the missingness
        g8 = g.reshape(V, -1)
        alt8, cal8 = group_counts((g8 == 1).astype(np.uint8), g8 >= 0, [member_cols(h, S, P) for h in lists])
        for i, haps in enumerate(lists):
            ref = orc.build_summary(d, haps)
            assert np.array_equal(alt[:, i], ref.alt) and np.array_equal(cal[:, i], ref.called)
            assert np.array_equal(alt8[:, i], ref.alt) and np.array_equal(cal8[:, i], ref.called)
            assert ref_scalars(cal[:, i], alt[:, i])[0] == ref.seg
            assert_region_sum(ref.pi_sum, cal[:, i], alt[:, i])


def test_reference_values_are_anchored():
    """site_pi / the theta table against the exact values at small and large n (incl. every pair up to n = 300)."""
    n = np.concatenate([np.repeat(np.arange(2, 301), np.arange(3, 302)), [229504, 229503, 57345, 16320, 2, 3]])
    a = np.concatenate([np.concatenate([np.arange(k + 1) for k in range(2, 301)]), [1, 114000, 57344, 8160, 1, 0]])
    anchor(n, a)
    # the pi restatement differs from the exact value, so the bound is doing work (not only 0 == 0)
    assert np.any(site_pi(n, a) != np.array([float(Fraction(2 * int(y) * (int(x) - int(y)), int(x) * (int(x) - 1)))
                                             for x, y in zip(n, a)]))


def test_table_predicts_the_layout_bytes():
    """group_bytes of fm_bench_diversity in mode 1 is V (16 wq + 4 tw + 4 + 16): the formula the GPU check uses."""
    fits = row_fits(*COHORTS["narrow"])
    assert layout(168, fits) == (1, 2) and layout(232, fits) == (2, 0)  # test_plane_bytes_per_step's groups
    assert layout(16320, fits) == (128, 0) and row_lanes_log2(128) == 4
    assert layout(3463, fits) == (27, 1) and rounds_of(27, 3) == 4
    assert chunk_geom(1793) == (8, 3, 896, 1) and chunk_geom(897) == (8, 2, 896, 1)
    assert chunk_geom(225) == (16, 1, 225, 225) and chunk_geom(449) == (8, 1, 449, 449)


# ------------------------------------------------------------------ GPU helpers
def _L():
    from ferromic_b200 import _lib
    return _lib


def fresh(m, haps):
    """A group that no other call has touched (the library caches counts per group)."""
    from ferromic_b200.api import _Group
    return _Group(m, haps)


def handles(groups):
    return (C.c_void_p * len(groups))(*[g.handle.value for g in groups])


class Ref:
    """Reference counts of one matrix's groups: haps -> (alt, called) arrays."""

    def __init__(self, data, called, S, P):
        self.data, self.called, self.S, self.P = data, called, S, P
        self.cache = {}

    def prime(self, lists):
        todo = [h for h in lists if tuple(h) not in self.cache]
        if todo:
            alt, cal = group_counts(self.data, self.called, [member_cols(h, self.S, self.P) for h in todo])
            for i, h in enumerate(todo):
                self.cache[tuple(h)] = (cal[:, i].copy(), alt[:, i].copy())
                anchor(cal[:, i], alt[:, i])

    def __call__(self, haps):
        self.prime([haps])
        return self.cache[tuple(haps)]


def check_summary(grp, ref, haps):
    """(1) fm_group_summary on a cold group: counts bit-exact, scalars exact / within the region-sum bound."""
    n, a = ref(haps)
    got = grp.summary(want_arrays=True)
    assert np.array_equal(got["called"], n) and np.array_equal(got["alt"], a), len(haps)
    assert (got["segregating_sites"], got["uncallable_lt2"]) == ref_scalars(n, a)
    assert_region_sum(got["pi_sum"], n, a)
    return got


def dropped_sites(pos, lo, hi, mask, filt):
    p = pos[lo:hi]
    d = np.isin(p, np.asarray(filt, dtype=np.int64))
    for s, e in mask or ():
        d |= (p >= s) & (p < e)
    return d


def per_site(grp, raw_n, pos, lo, hi, mask=None, filt=()):
    L = _L()
    cap = hi - lo
    out_p, pi, th = np.zeros(cap, dtype=np.int64), np.zeros(cap), np.zeros(cap)
    mk = None if mask is None else np.ascontiguousarray(mask, dtype=np.int64).reshape(-1)
    fl = np.ascontiguousarray(filt, dtype=np.int64)
    k = C.c_size_t()
    L.check(L.lib().fm_per_site_diversity(grp.handle, raw_n, int(pos[lo]), int(pos[hi - 1]),
                                          None if mk is None else mk.ctypes.data, 0 if mk is None else mk.size // 2,
                                          fl.ctypes.data if fl.size else None, fl.size, out_p.ctypes.data,
                                          pi.ctypes.data, th.ctypes.data, cap, C.byref(k)))
    return k.value, out_p, pi, th


def same_bits(x, y):
    """NaN at the same sites, every other value bit for bit."""
    nan = np.isnan(x)
    return np.array_equal(nan, np.isnan(y)) and np.array_equal(x[~nan].view(np.uint64), y[~nan].view(np.uint64))


def assert_tracks(pi, th, n, a, dropped):
    rpi, rth = ref_tracks(n, a, dropped)
    assert same_bits(pi, rpi) and same_bits(th, rth)


# regions by site index [lo, hi): v_lo % 32 in {0, 1, 31}, ends mid-batch, crossing the super-batch at site 8192
NARROW_REGIONS = ((0, NARROW_V), (1, 8193 + 7), (31, 4001), (8191, NARROW_V), (3201, 8210))


def region_mask(pos):
    V = len(pos)
    return [(int(pos[40]), int(pos[70])), (int(pos[V - 173]), int(pos[V - 153]) + 1),
            (int(pos[V * 3 // 5]), int(pos[V * 3 // 5]) + 1)]


def region_filt(pos):
    return [int(pos[i]) for i in (5, 33, 8191, 8192, len(pos) - 1) if i < len(pos)]


def check_tracks(grp, ref, haps, pos, regions, with_mask=True):
    """(3) fm_per_site_diversity on a group without cached counts (the plane pass writes the tracks)."""
    n, a = ref(haps)
    for lo, hi in regions:
        mask = region_mask(pos) if with_mask else None
        filt = region_filt(pos) if with_mask else ()
        k, p, pi, th = per_site(grp, len(haps), pos, lo, hi, mask, filt)
        assert k == hi - lo and np.array_equal(p, pos[lo:hi] + 1)
        assert_tracks(pi, th, n[lo:hi], a[lo:hi], dropped_sites(pos, lo, hi, mask, filt))


# ------------------------------------------------------------------ GPU: narrow cohort
@pytest.fixture(scope="module")
def narrow():
    g, data, miss, pos = make_genotypes(NARROW_V, NARROW_S, 20261020)
    rng = np.random.default_rng(11)
    lists = {n: random_haps(rng, NARROW_S, 2, n) for n in NARROW_SIZES}
    V = NARROW_V
    ref = Ref(data.reshape(V, -1), ~miss.reshape(V, -1), NARROW_S, 2)
    ref.prime(list(lists.values()))
    return dict(g=g, data=data, miss=miss, pos=pos, lists=lists, ref=ref)


@pytest.fixture(scope="module")
def narrow_u8(narrow):
    from ferromic_b200.api import _Matrix
    return _Matrix(narrow["data"], narrow["miss"], narrow["pos"], max_allele=1, always_bitmap=True, ingest="u8")


@pytest.mark.gpu
def test_narrow_summaries_tracks_and_layout(narrow, narrow_u8):
    """Every narrow size: cold summary, plane-pass tracks over every region class, and the layout the table
    predicts (fm_bench_diversity group_bytes, mode 1), bench tracks / totals in both modes."""
    L = _L()
    pos, ref, lists = narrow["pos"], narrow["ref"], narrow["lists"]
    fits = row_fits(*COHORTS["narrow"])
    for n in NARROW_SIZES:
        grp = fresh(narrow_u8, lists[n])
        check_tracks(grp, ref, lists[n], pos, NARROW_REGIONS)
        check_summary(grp, ref, lists[n])
    # (6) bench: every group in one row launch of mixed widths, per-group layout bytes, totals and tracks
    V = NARROW_V
    mask = region_mask(pos)
    mk = np.ascontiguousarray(mask, dtype=np.int64).reshape(-1)
    dropped = dropped_sites(pos, 0, V, mask, ())
    for part in (NARROW_SIZES[0:8], NARROW_SIZES[8:16], NARROW_SIZES[16:24], NARROW_SIZES[24:]):
        gs = [fresh(narrow_u8, lists[n]) for n in part]
        for mode in (0, 1):
            res = L.BenchResult()
            tp = np.zeros((len(gs), V)) if mode == 1 else None
            tt = np.zeros((len(gs), V)) if mode == 1 else None
            L.check(L.lib().fm_bench_diversity(handles(gs), len(gs), mode, mk.ctypes.data if mode else None,
                                               mk.size // 2 if mode else 0, 1, None, C.byref(res),
                                               None if tp is None else tp.ctypes.data,
                                               None if tt is None else tt.ctypes.data))
            for i, n_hap in enumerate(part):
                cnt, alt = ref(lists[n_hap])
                wq, tw = layout(n_hap, fits)
                assert res.group_bytes[i] == V * (16 * wq + 4 * tw + 4 + (16 if mode else 0)), n_hap
                assert (res.last_seg[i], res.last_unc[i]) == ref_scalars(cnt, alt)
                assert_region_sum(res.last_pi_sum[i], cnt, alt)
                if mode == 1:
                    assert_tracks(tp[i], tt[i], cnt, alt, dropped)


@pytest.mark.gpu
def test_narrow_batch_summaries(narrow, narrow_u8):
    """(2) fm_groups_summary_batch over <= 4 groups (inline table) and >= 5 (uploaded): scalars bit-equal to the
    single-group call, counts as the reference."""
    L = _L()
    ref, lists = narrow["ref"], narrow["lists"]
    for batch in BATCHES:
        single = {n: fresh(narrow_u8, lists[n]).summary() for n in batch}
        gs = [fresh(narrow_u8, lists[n]) for n in batch]
        k = len(gs)
        seg, unc, pis = np.zeros(k, dtype=np.uint64), np.zeros(k, dtype=np.uint64), np.zeros(k)
        L.check(L.lib().fm_groups_summary_batch(handles(gs), k, seg.ctypes.data, pis.ctypes.data, unc.ctypes.data))
        for i, n in enumerate(batch):
            s = single[n]
            assert (int(seg[i]), int(unc[i])) == (s["segregating_sites"], s["uncallable_lt2"])
            assert pis[i] == s["pi_sum"], n
            check_summary(gs[i], ref, lists[n])


@pytest.mark.gpu
def test_narrow_multi_group_tracks(narrow, narrow_u8):
    """(4) fm_per_site_diversity_multi with mixed widths in ONE launch (LG 4 with a 1-word group; five groups with an
    uploaded table): bit-equal to per-group calls and to the reference."""
    L = _L()
    pos, ref, lists = narrow["pos"], narrow["ref"], narrow["lists"]
    mask, filt = region_mask(pos), region_filt(pos)
    mk = np.ascontiguousarray(mask, dtype=np.int64).reshape(-1)
    fl = np.ascontiguousarray(filt, dtype=np.int64)
    for mix in MULTI_MIXES:
        for lo, hi in NARROW_REGIONS:
            gs = [fresh(narrow_u8, lists[n]) for n in mix]
            k, cap = len(gs), hi - lo
            raw = (C.c_size_t * k)(*[len(lists[n]) for n in mix])
            pi, th = np.zeros((k, cap)), np.zeros((k, cap))
            out_p = np.zeros(cap, dtype=np.int64)
            nout = C.c_size_t()
            L.check(L.lib().fm_timings_reset())
            L.check(L.lib().fm_per_site_diversity_multi(handles(gs), raw, k, int(pos[lo]), int(pos[hi - 1]),
                                                        mk.ctypes.data, mk.size // 2, fl.ctypes.data, fl.size,
                                                        out_p.ctypes.data, pi.ctypes.data, th.ctypes.data, cap,
                                                        C.byref(nout)))
            t = L.Timings()
            L.check(L.lib().fm_timings_get(C.byref(t)))
            assert t.stats_launches == 1, mix
            assert nout.value == cap and np.array_equal(out_p, pos[lo:hi] + 1)
            dropped = dropped_sites(pos, lo, hi, mask, filt)
            for i, n_hap in enumerate(mix):
                cnt, alt = ref(lists[n_hap])
                assert_tracks(pi[i], th[i], cnt[lo:hi], alt[lo:hi], dropped)
                _, _, spi, sth = per_site(fresh(narrow_u8, lists[n_hap]), len(lists[n_hap]), pos, lo, hi, mask, filt)
                assert same_bits(spi, pi[i]) and same_bits(sth, th[i])


def hudson_first(g1, g2, h1, h2, Lseq):
    L = _L()
    out = L.HudsonOutcome()
    ns = C.c_size_t()
    L.check(L.lib().fm_hudson_pair(g1.handle, g2.handle, Lseq, Lseq, L.FM_HUDSON_SUMMARIES, 0, 0, 0, len(h1), len(h2),
                                   C.byref(out), None, C.byref(ns)))
    return out


def check_pair(m, ref, h1, h2, pos):
    """(5) fm_hudson_pair as the first call on fresh groups (the fused pair pass) equals the cached-counts call bit
    for bit, caches the reference counts and agrees with the oracle's summaries path."""
    Lseq = int(pos[-1] - pos[0] + 1)
    g1, g2 = fresh(m, h1), fresh(m, h2)
    first = hudson_first(g1, g2, h1, h2, Lseq)
    again = hudson_first(g1, g2, h1, h2, Lseq)
    assert bytes(first) == bytes(again)
    n1, a1 = ref(h1)
    n2, a2 = ref(h2)
    check_summary(g1, ref, h1)
    check_summary(g2, ref, h2)
    S = ref.S
    s1 = orc.Summary(a1, n1, len(member_cols(h1, S, ref.P)), ref_scalars(n1, a1)[0], float(exact_pi_sum(n1, a1)))
    s2 = orc.Summary(a2, n2, len(member_cols(h2, S, ref.P)), ref_scalars(n2, a2)[0], float(exact_pi_sum(n2, a2)))
    rc, want, _ = orc.hudson_pair(orc.Pop(h1, None, S, Lseq, summary=s1), orc.Pop(h2, None, S, Lseq, summary=s2))
    for bit, key in enumerate(("fst", "d_xy", "pi_pop1", "pi_pop2", "pi_xy_avg")):
        has = bool(first.some >> bit & 1)
        assert has == (want[key] is not None), key
        if has:
            got = getattr(first, key)
            assert abs(got - want[key]) <= 1e-12 * max(abs(want[key]), 1.0), (key, got, want[key])


@pytest.mark.gpu
def test_narrow_hudson_pairs(narrow, narrow_u8):
    for p in PAIRS:
        check_pair(narrow_u8, narrow["ref"], narrow["lists"][p[0]], narrow["lists"][p[1]], narrow["pos"])


def window_set(pos):
    """Empty, before all, after all, one site, ends on positions, overlapping, descending order, everything,
    boundaries at sites 8191 / 8192."""
    p = [int(x) for x in pos]
    gap = next(i for i in range(len(p) - 1) if p[i + 1] > p[i] + 1)
    w = [(p[gap] + 1, p[gap + 1] - 1), (0, p[0] - 1), (p[-1] + 1, p[-1] + 1000), (p[77], p[77]), (p[3], p[2000]),
         (p[10], p[500]), (p[400], p[900]), (p[0] - 5, p[-1] + 5), (p[0], p[8191]), (p[8192], p[-1]),
         (p[8191], p[8192]), (p[8190], p[8193] - 1)]
    return np.array(w[::-1], dtype=np.int64)


def hudson_site_terms(n1, a1, n2, a2):
    """aggregate_hudson_components_from_summaries per site, restated (fm_hudson_contrib, variant < 0)."""
    n1, a1, n2, a2 = (x.astype(np.int64) for x in (n1, a1, n2, a2))
    skip = (n1 == 0) | (n2 == 0)
    with np.errstate(invalid="ignore", divide="ignore"):
        dxy = ((a1 * (n2 - a2) + (n1 - a1) * a2).astype(np.float64) / (n1 * n2).astype(np.float64))
        dxy = np.where(skip, 0.0, np.clip(dxy, 0.0, 1.0))
        both = ~skip & (n1 >= 2) & (n2 >= 2)
        p1 = np.where(both, 2.0 * a1.astype(np.float64) * (n1 - a1).astype(np.float64) / (n1 * (n1 - 1)).astype(
            np.float64), 0.0)
        p2 = np.where(both, 2.0 * a2.astype(np.float64) * (n2 - a2).astype(np.float64) / (n2 * (n2 - 1)).astype(
            np.float64), 0.0)
    fst_ok = both & (dxy > 1e-12)
    num = np.where(fst_ok, dxy - 0.5 * (p1 + p2), 0.0)
    den = np.where(fst_ok, dxy, 0.0)
    return num, den, dxy, p1, p2, skip


def assert_sum(dev, terms):
    terms = np.asarray(terms, dtype=np.float64)
    want = math.fsum(terms.tolist())
    assert abs(dev - want) <= 16 * EPS * len(terms) + 40 * EPS * float(np.abs(terms).sum()), (dev, want)


@pytest.mark.gpu
def test_narrow_window_sums(narrow, narrow_u8):
    """(7) fm_group_window_sums and fm_hudson_window_sums: every output of every window."""
    L = _L()
    pos, ref, lists = narrow["pos"], narrow["ref"], narrow["lists"]
    W = window_set(pos)
    nw = len(W)
    for h1, h2 in ((lists[129], lists[16320]), (lists[2], lists[14337]), (lists[480], lists[3463])):
        g1, g2 = fresh(narrow_u8, h1), fresh(narrow_u8, h2)
        nv, seg, unc = (np.zeros(nw, dtype=np.uint64) for _ in range(3))
        pis = np.zeros(nw)
        L.check(L.lib().fm_group_window_sums(g1.handle, W.ctypes.data, nw, nv.ctypes.data, seg.ctypes.data,
                                             pis.ctypes.data, unc.ctypes.data))
        f = [np.zeros(nw) for _ in range(5)]
        sk = np.zeros(nw, dtype=np.uint64)
        L.check(L.lib().fm_hudson_window_sums(g1.handle, g2.handle, W.ctypes.data, nw, f[0].ctypes.data,
                                              f[1].ctypes.data, f[2].ctypes.data, sk.ctypes.data, f[3].ctypes.data,
                                              f[4].ctypes.data))
        n1, a1 = ref(h1)
        n2, a2 = ref(h2)
        terms = hudson_site_terms(n1, a1, n2, a2)
        for w, (s, e) in enumerate(W):
            sel = (pos >= s) & (pos <= e)
            assert nv[w] == sel.sum()
            assert (int(seg[w]), int(unc[w])) == ref_scalars(n1[sel], a1[sel])
            assert_region_sum(pis[w], n1[sel], a1[sel])
            for k in range(5):
                assert_sum(f[k][w], terms[k][sel])
            assert sk[w] == int(terms[5][sel].sum())


def check_form(m, ref, lists, pos, sizes, regions):
    """(1) + (3) for one ingest form: tracks on a cold group, then its summary."""
    for n in sizes:
        grp = fresh(m, lists[n])
        if regions:
            check_tracks(grp, ref, lists[n], pos, regions)
        check_summary(grp, ref, lists[n])


FORM_REGIONS = ((1, 8193 + 7), (8191, NARROW_V))


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["in-band", "packed-dense", "packed-sparse-gap", "packed-sparse-u16", "no-missing",
                                  "staged-8159"])
def test_narrow_ingest_forms(narrow, form, monkeypatch):
    from ferromic_b200 import api
    from ferromic_b200.api import _Matrix
    pos, lists, data, miss = narrow["pos"], narrow["lists"], narrow["data"], narrow["miss"]
    ref = narrow["ref"]
    if form == "in-band":
        m = _Matrix.from_int8(narrow["g"], pos, 1, ingest="u8")
    elif form == "packed-dense":
        m = _Matrix(data, miss, pos, max_allele=1, always_bitmap=True, ingest="packed-dense")
    elif form.startswith("packed-sparse"):
        monkeypatch.setattr(api, "SPARSE_GAP_CODE", form.endswith("gap"))
        m = _Matrix(data, miss, pos, max_allele=1, always_bitmap=True, ingest="packed-sparse")
        assert m.ingest_mode == "packed-sparse"
    elif form == "no-missing":
        m = _Matrix(data, None, pos, max_allele=1, ingest="u8")
        ref = Ref(data.reshape(NARROW_V, -1), None, NARROW_S, 2)
    else:  # stride 16318 (not a multiple of 16): the staged rows of K1
        S = NARROW_S - 1
        m = _Matrix(data[:, :S], miss[:, :S], pos, max_allele=1, always_bitmap=True, ingest="u8")
        ref = Ref(data[:, :S].reshape(NARROW_V, -1), ~miss[:, :S].reshape(NARROW_V, -1), S, 2)
    check_form(m, ref, lists, pos, NARROW_SIZES, FORM_REGIONS if form != "no-missing" else NARROW_REGIONS)
    if form == "no-missing":
        for p in PAIRS[:1]:
            check_pair(m, ref, lists[p[0]], lists[p[1]], pos)


@pytest.mark.gpu
def test_narrow_ploidy_one(narrow):
    from ferromic_b200.api import _Matrix
    pos, data, miss = narrow["pos"], narrow["data"], narrow["miss"]
    m = _Matrix(np.ascontiguousarray(data[:, :, :1]), np.ascontiguousarray(miss[:, :, :1]), pos, max_allele=1,
                always_bitmap=True, ingest="u8")
    ref = Ref(data[:, :, 0].copy(), ~miss[:, :, 0], NARROW_S, 1)
    rng = np.random.default_rng(12)
    sizes = tuple(n for n in NARROW_SIZES if n <= NARROW_S)
    lists = {n: random_haps(rng, NARROW_S, 1, n) for n in sizes}
    ref.prime(list(lists.values()))
    check_form(m, ref, lists, pos, sizes, FORM_REGIONS)


@pytest.mark.gpu
def test_narrow_streaming_ingest(narrow):
    """u8 rows pushed in three calls with chunks of 1000 rows (not a multiple of 32), groups declared up front and
    tracks requested at ingest time."""
    from ferromic_b200.api import _Matrix
    pos, lists, ref = narrow["pos"], narrow["lists"], narrow["ref"]
    sizes = (1, 2, 33, 129, 1473, 3463, 5008, 14337, 16320)
    decl = [lists[n] for n in sizes]
    lo, hi = 8191, NARROW_V
    cap = hi - lo
    mask, filt = region_mask(pos), region_filt(pos)
    req = {"groups": list(range(len(decl))), "raw_n": [len(h) for h in decl], "region": (int(pos[lo]), int(pos[hi - 1])),
           "mask": np.array(mask, dtype=np.int64), "filtered": np.array(filt, dtype=np.int64),
           "pos": np.zeros(cap, dtype=np.int64), "pi": np.zeros((len(decl), cap)), "theta": np.zeros((len(decl), cap)),
           "capacity": cap}
    m = _Matrix.ingest(narrow["data"], narrow["miss"], pos, decl, chunk_rows=1000, calls=3, always_bitmap=True,
                       tracks=req)
    assert m.track_sites == cap and np.array_equal(req["pos"], pos[lo:hi] + 1)
    dropped = dropped_sites(pos, lo, hi, mask, filt)
    for i, haps in enumerate(decl):
        n, a = ref(haps)
        assert_tracks(req["pi"][i], req["theta"][i], n[lo:hi], a[lo:hi], dropped)
        check_summary(m.group(haps), ref, haps)


@pytest.mark.gpu
def test_synth_device_matrix():
    """A device-resident matrix from fm_synth_fill; the reference rebuilt by tests/synth.py::synth_rows."""
    import torch
    from tests.synth import synth_rows
    L = _L()
    V, S, seed = 2100, NARROW_S, 77
    total = V * S * 2
    d_data = torch.empty(total, dtype=torch.uint8, device="cuda:0")
    d_miss = torch.empty((total + 63) // 64, dtype=torch.int64, device="cuda:0")
    L.check(L.lib().fm_set_device(0))
    L.check(L.lib().fm_synth_fill(d_data.data_ptr(), d_miss.data_ptr(), V, S, 2, 0, seed, None, 0.05, 0.02))
    pos = np.cumsum(np.random.default_rng(seed).integers(1, 50, size=V, dtype=np.int64))
    h = C.c_void_p()
    L.check(L.lib().fm_matrix_create_device(d_data.data_ptr(), d_miss.data_ptr(), V, S, 2, 1, pos.ctypes.data,
                                            C.byref(h)))

    M = type("M", (), {"handle": h, "V": V})  # the matrix in the shape _Group expects
    g = synth_rows(seed, 0, V, S, missing_rate=0.02).reshape(V, -1)
    ref = Ref((g == 1).astype(np.uint8), g >= 0, S, 2)
    rng = np.random.default_rng(13)
    lists = {n: random_haps(rng, S, 2, n) for n in (2, 129, 640, 3463, 4609, 14336, 16320)}
    ref.prime(list(lists.values()))
    try:
        check_form(M, ref, lists, pos, tuple(lists), ((1, 2051), (31, V)))
    finally:
        import gc
        gc.collect()
        L.lib().fm_matrix_release(h)


# ------------------------------------------------------------------ GPU: wide cohort
@pytest.fixture(scope="module")
def wide():
    g, data, miss, pos = make_genotypes(WIDE_V, WIDE_S, 20261021, missing=0.01)
    rng = np.random.default_rng(21)
    lists = {n: random_haps(rng, WIDE_S, 2, n) for n in WIDE_SIZES}
    ref = Ref(data.reshape(WIDE_V, -1), ~miss.reshape(WIDE_V, -1), WIDE_S, 2)
    ref.prime(list(lists.values()))
    return dict(data=data, miss=miss, pos=pos, lists=lists, ref=ref)


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["u8", "packed-dense"])
def test_wide_rows(wide, form):
    """Chunked classes (16 warps, 8 warps, 2 and 3 chunks with a last chunk of one word), the narrow groups of a
    wide matrix (no tail layout on u8 rows repacked by fm_k_repack), a partial last batch, layout bytes and a
    chunked Hudson pair."""
    from ferromic_b200.api import _Matrix
    L = _L()
    pos, lists, ref = wide["pos"], wide["lists"], wide["ref"]
    m = _Matrix(wide["data"], wide["miss"], pos, max_allele=1, always_bitmap=True, ingest=form)
    fits = row_fits(*COHORTS["wide-u8" if form == "u8" else "wide-packed"])
    regions = ((0, WIDE_V), (1, WIDE_V), (31, 65))
    for n in WIDE_SIZES:
        grp = fresh(m, lists[n])
        check_tracks(grp, ref, lists[n], pos, regions, with_mask=False)
        check_summary(grp, ref, lists[n])
        res = L.BenchResult()
        gb = fresh(m, lists[n])
        L.check(L.lib().fm_bench_diversity(handles([gb]), 1, 1, None, 0, 1, None, C.byref(res), None, None))
        wq, tw = layout(n, fits)
        assert res.group_bytes[0] == WIDE_V * (16 * wq + 4 * tw + 4 + 16), n
        cnt, alt = ref(lists[n])
        assert (res.last_seg[0], res.last_unc[0]) == ref_scalars(cnt, alt)
    check_pair(m, ref, lists[WIDE_PAIR[0]], lists[WIDE_PAIR[1]], pos)
    check_pair(m, ref, lists[129], lists[16320], pos)


@pytest.mark.gpu
def test_wide_mixed_set(wide):
    """A set that mixes kinds -- a group too wide for the row pass, two fresh narrow groups and a narrow group whose
    summary is cached -- through fm_per_site_diversity_multi and fm_groups_summary_batch: the fresh narrow groups
    share one row launch (two stats launches in all) and every output equals the per-group calls bit for bit."""
    from ferromic_b200.api import _Matrix
    L = _L()
    pos, lists, ref = wide["pos"], wide["lists"], wide["ref"]
    m = _Matrix(wide["data"], wide["miss"], pos, max_allele=1, always_bitmap=True, ingest="u8")
    haps = [lists[114689], lists[129], lists[16320], random_haps(np.random.default_rng(22), WIDE_S, 2, 1000)]
    k = len(haps)

    def mixed_set():
        gs = [fresh(m, h) for h in haps]
        gs[-1].summary()
        return gs

    def stats_launches(call):
        L.check(L.lib().fm_timings_reset())
        L.check(call())
        t = L.Timings()
        L.check(L.lib().fm_timings_get(C.byref(t)))
        return t.stats_launches

    lo, hi = 1, WIDE_V
    cap = hi - lo
    mask, filt = [(int(pos[10]), int(pos[20]))], [int(pos[5]), int(pos[40])]
    mk = np.ascontiguousarray(mask, dtype=np.int64).reshape(-1)
    fl = np.ascontiguousarray(filt, dtype=np.int64)
    raw = (C.c_size_t * k)(*[len(h) for h in haps])
    pi, th, out_p, nout = np.zeros((k, cap)), np.zeros((k, cap)), np.zeros(cap, dtype=np.int64), C.c_size_t()
    gs = mixed_set()
    assert stats_launches(lambda: L.lib().fm_per_site_diversity_multi(
        handles(gs), raw, k, int(pos[lo]), int(pos[hi - 1]), mk.ctypes.data, mk.size // 2, fl.ctypes.data, fl.size,
        out_p.ctypes.data, pi.ctypes.data, th.ctypes.data, cap, C.byref(nout))) == 2
    assert nout.value == cap and np.array_equal(out_p, pos[lo:hi] + 1)
    dropped = dropped_sites(pos, lo, hi, mask, filt)
    for i, h in enumerate(haps):
        n, a = ref(h)
        assert_tracks(pi[i], th[i], n[lo:hi], a[lo:hi], dropped)
        _, _, spi, sth = per_site(fresh(m, h), len(h), pos, lo, hi, mask, filt)
        assert same_bits(spi, pi[i]) and same_bits(sth, th[i]), len(h)

    gs = mixed_set()
    seg, unc, pis = np.zeros(k, dtype=np.uint64), np.zeros(k, dtype=np.uint64), np.zeros(k)
    assert stats_launches(lambda: L.lib().fm_groups_summary_batch(handles(gs), k, seg.ctypes.data, pis.ctypes.data,
                                                                  unc.ctypes.data)) == 2
    for i, h in enumerate(haps):
        single = fresh(m, h).summary(want_arrays=True)
        got = gs[i].summary(want_arrays=True)
        assert (int(seg[i]), int(unc[i])) == (single["segregating_sites"], single["uncallable_lt2"]), len(h)
        assert pis[i] == single["pi_sum"] == got["pi_sum"], len(h)
        assert np.array_equal(got["alt"], single["alt"]) and np.array_equal(got["called"], single["called"]), len(h)
        check_summary(gs[i], ref, h)


# ------------------------------------------------------------------ GPU: multi-allelic counts
MULTI_V, MULTI_S = 300, 28673
MULTI_SIZES = (1, 31, 33, 127, 129, 1000, 16320, 57345)


@pytest.fixture(scope="module")
def multi_cohort():
    rng = np.random.default_rng(31)
    V, stride = MULTI_V, 2 * MULTI_S
    pos = np.cumsum(rng.integers(1, 30, size=V, dtype=np.int64)) + 5
    u = rng.random((V, stride), dtype=np.float32)
    miss = rng.random((V, stride), dtype=np.float32) < 0.02
    lists = {n: random_haps(rng, MULTI_S, 2, n) for n in MULTI_SIZES}
    return dict(pos=pos, u=u, miss=miss, lists=lists, rng=rng)


@pytest.mark.gpu
@pytest.mark.parametrize("bitmap", [True, False])
@pytest.mark.parametrize("max_allele", [2, 3, 15])
def test_multi_allelic_counts(multi_cohort, max_allele, bitmap):
    """fm_k_allele_counts at 1-57345 haplotypes (more than one 16-byte column: the no-bitmap padding mask), checked
    site by site through one-site windows of fm_group_window_sums (general dense forms), plus
    fm_group_segregating_sites and fm_group_pi(FM_PI_DENSE) against the oracle."""
    from ferromic_b200.api import _Matrix
    L = _L()
    V, S = MULTI_V, MULTI_S
    pos, lists = multi_cohort["pos"], multi_cohort["lists"]
    # skewed allele values: allele 0 common, the top value present
    data = np.minimum((multi_cohort["u"] ** 3 * (max_allele + 1)).astype(np.uint8), max_allele)
    data[::7, ::5] = max_allele
    data[::11] = 0  # monomorphic sites
    miss = multi_cohort["miss"] if bitmap else None
    m = _Matrix(data.reshape(V, S, 2), None if miss is None else miss.reshape(V, S, 2), pos, max_allele=max_allele,
                always_bitmap=bitmap, ingest="u8")
    d = orc.Dense(data.reshape(-1), None if miss is None else orc.pack_missing_bits(miss.reshape(-1)), V, S, 2,
                  max_allele)
    called = None if miss is None else ~miss
    cols = [member_cols(lists[n], S, 2) for n in MULTI_SIZES]
    per_allele = [group_counts(data, called, cols, allele=k) for k in range(max_allele + 1)]
    cnt = per_allele[0][1]
    W = np.stack([pos, pos], axis=1).astype(np.int64)
    Lseq = int(pos[-1] - pos[0] + 1)
    for gi, n_hap in enumerate(MULTI_SIZES):
        haps = lists[n_hap]
        grp = fresh(m, haps)
        nv, seg, unc = (np.zeros(V, dtype=np.uint64) for _ in range(3))
        pis = np.zeros(V)
        L.check(L.lib().fm_group_window_sums(grp.handle, W.ctypes.data, V, nv.ctypes.data, seg.ctypes.data,
                                             pis.ctypes.data, unc.ctypes.data))
        c = np.stack([pa[0][:, gi] for pa in per_allele], axis=1)
        n = cnt[:, gi]
        assert np.array_equal(c.sum(axis=1), n)
        distinct = (c > 0).sum(axis=1)
        nf = n.astype(np.float64)
        ssq = (c.astype(np.float64) ** 2).sum(axis=1)
        with np.errstate(invalid="ignore", divide="ignore"):
            want_pi = np.where(n >= 2, nf / (nf - 1.0) * (1.0 - ssq / (nf * nf)), 0.0)
        assert np.array_equal(seg, (distinct > 1).astype(np.uint64)), n_hap
        assert np.array_equal(unc, (n < 2).astype(np.uint64))
        assert np.array_equal(pis, want_pi), n_hap
        s = C.c_uint64()
        L.check(L.lib().fm_group_segregating_sites(grp.handle, C.byref(s)))
        pop = orc.Pop(haps, None, S, Lseq, dense=d)
        assert s.value == orc.count_segregating_sites_for_population(pop)
        assert s.value == (int((distinct > 1).sum()) if len(cols[gi]) > 1 else 0)
        got = grp.pi(Lseq, _L().FM_PI_DENSE)
        want = orc.pi_for_population(pop)
        assert (math.isnan(got) and math.isnan(want)) or abs(got - want) <= 1e-12 * abs(want), (n_hap, got, want)
