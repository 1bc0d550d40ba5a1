"""numpy restatement of haplotype LD (fm_haplotype_ld, include/ferromic_gpu.h; DESIGN.md §3 and §4 "Haplotype LD").
Haplotypes and site filters are those of tests/pca_reference.py.  The kept sites are packed into uint64 words of
haplotypes and counted with np.bitwise_count one diagonal d at a time, so 50k sites x window 1000 is quick; the
statistics follow the header's operation order in FP64 and are rounded to float32 once."""
import numpy as np

from tests.pca_reference import offsets, rows_from_arrays, site_stats  # noqa: F401  (re-exported for the tests)

NAN32 = np.float32(np.nan)  # 0x7fc00000


def pack_sites(get_rows, kept, off, chunk=16384):
    """(alt words, called words) uint64 [M, ceil(n / 64)]: bit h of word h // 64 is haplotype off[h]."""
    n, M = len(off), len(kept)
    W = max(1, (n + 63) // 64)
    A = np.zeros((M, W), np.uint64)
    Cw = np.zeros((M, W), np.uint64)
    for j in range(0, M, chunk):
        rows = kept[j:j + chunk]
        x, c = get_rows(int(rows[0]), int(rows[-1]) + 1)
        x, c = x[rows - rows[0]][:, off], c[rows - rows[0]][:, off]
        for dst, bits in ((A, c & (x == 1)), (Cw, c)):
            pad = np.zeros((len(rows), W * 64), bool)
            pad[:, :n] = bits
            dst[j:j + len(rows)] = np.packbits(pad, axis=1, bitorder="little").view(np.uint64)
    return A, Cw


def stats(c, a, b, ab, fp64=False):
    """(r2, D') float32 (FP64 when fp64) from int64 counts; NaN where c == 0 or a site is monomorphic among the jointly
    called."""
    c, a, b, ab = (np.asarray(v, np.int64) for v in (c, a, b, ab))
    ok = (c > 0) & (a > 0) & (a < c) & (b > 0) & (b < c)
    r2 = np.full(c.shape, np.nan)
    dp = np.full(c.shape, np.nan)
    c, a, b, ab = c[ok], a[ok], b[ok], ab[ok]
    dn = c * ab - a * b
    x = dn.astype(np.float64)
    r2[ok] = (x * x) / ((a * (c - a)).astype(np.float64) * (b * (c - b)).astype(np.float64))
    den = np.where(dn > 0, np.minimum(a * (c - b), (c - a) * b), np.minimum(a * b, (c - a) * (c - b)))
    dp[ok] = np.where(dn == 0, 0.0, x / den.astype(np.float64))
    return (r2, dp) if fp64 else (r2.astype(np.float32), dp.astype(np.float32))


def haplotype_ld(get_rows, n_variants, off, window, positions, max_distance=None, min_maf=0.0, max_missing=0.0,
                 site_range=None, chunk=16384):
    """dict(kept, n, M, pairs, r2 [M, window], dprime [M, window], counts) for the matrix rows given by get_rows;
    positions are the matrix rows' positions.  counts[d] = (c, a, b, ab) of the pairs (i, i + d), i < M - d."""
    off = np.asarray(off, dtype=np.int64)
    n = len(off)
    v_lo, v_hi = (0, n_variants) if site_range is None else site_range
    kept, called, alt = site_stats(get_rows, v_lo, v_hi, off, min_maf, max_missing, chunk)
    M = len(kept)
    r2 = np.full((M, window), NAN32, np.float32)
    dp = np.full((M, window), NAN32, np.float32)
    out = dict(kept=kept, n=n, M=M, pairs=0, r2=r2, dprime=dp, counts={})
    if M < 2:
        return out
    A, Cw = pack_sites(get_rows, kept, off, chunk)
    kpos = np.asarray(positions, np.int64)[kept]
    popc = lambda x: np.bitwise_count(x).sum(axis=1, dtype=np.int64)  # noqa: E731
    for d in range(1, min(window, M - 1) + 1):
        ai, aj, ci, cj = A[:M - d], A[d:], Cw[:M - d], Cw[d:]
        counts = (popc(ci & cj), popc(ai & cj), popc(ci & aj), popc(ai & aj))
        out["counts"][d] = counts
        pair = np.ones(M - d, bool) if max_distance is None else (kpos[d:] - kpos[:M - d] <= max_distance)
        out["pairs"] += int(pair.sum())
        rr, dd = stats(*counts)
        r2[:M - d, d - 1] = np.where(pair, rr, NAN32)
        dp[:M - d, d - 1] = np.where(pair, dd, NAN32)
    return out
