"""numpy restatement of haplotype LD pruning (fm_haplotype_ld_prune, include/ferromic_gpu.h; DESIGN.md §3 and §4 "LD
pruning").  Kept sites, pairs and counts are those of tests/ld_reference.py: the kept sites are packed into uint64
words and counted one diagonal d at a time; each diagonal's FP64 r^2 (ld_reference.stats, fp64=True) decides its
linked pairs, which go straight into forward bit rows (bit d - 1 of row i, ceil(w / 32) uint32 words a row), so no
FP64 M x window array is ever held.  The greedy scan walks those rows."""
import numpy as np

from tests import ld_reference as lr
from tests.pca_reference import site_stats


def subset_rows(get_rows, site_list):
    """get_rows in which the matrix rows outside `site_list` are monomorphic and fully called, so the site filter
    never keeps them and every other row is unchanged: the restatement of a site list for ld_reference.haplotype_ld,
    this module and pca_reference.haplotype_pca (whose test matrix is keyed by matrix row)."""
    listed = np.asarray(site_list, np.int64)

    def rows(a, b):
        x, c = get_rows(a, b)
        out = ~np.isin(np.arange(a, b), listed)
        x, c = x.copy(), c.copy()
        x[out], c[out] = 0, True
        return x, c
    return rows


def linked_bits(get_rows, n_variants, off, window, positions, r2_threshold, max_distance=None, min_maf=0.0,
                max_missing=0.0, site_range=None, chunk=16384):
    """dict(kept, M, w, pairs, linked_pairs, bits uint32 [M, max(1, ceil(w / 32))]) with w = min(window, M - 1)."""
    off = np.asarray(off, np.int64)
    v_lo, v_hi = (0, n_variants) if site_range is None else site_range
    kept = site_stats(get_rows, v_lo, v_hi, off, min_maf, max_missing, chunk)[0]
    M = len(kept)
    w = max(0, min(window, M - 1))
    bits = np.zeros((M, max(1, (w + 31) // 32)), np.uint32)
    out = dict(kept=kept, M=M, w=w, pairs=0, linked_pairs=0, bits=bits)
    if M < 2:
        return out
    A, Cw = lr.pack_sites(get_rows, kept, off, chunk)
    kpos = np.asarray(positions, np.int64)[kept]
    popc = lambda x: np.bitwise_count(x).sum(axis=1, dtype=np.int64)  # noqa: E731
    for d in range(1, w + 1):
        ai, aj, ci, cj = A[:M - d], A[d:], Cw[:M - d], Cw[d:]
        r2 = lr.stats(popc(ci & cj), popc(ai & cj), popc(ci & aj), popc(ai & aj), fp64=True)[0]
        pair = np.ones(M - d, bool) if max_distance is None else (kpos[d:] - kpos[:M - d] <= max_distance)
        linked = pair & (r2 > r2_threshold)  # NaN compares false
        out["pairs"] += int(pair.sum())
        out["linked_pairs"] += int(linked.sum())
        bits[:M - d, (d - 1) >> 5] |= linked.astype(np.uint32) << np.uint32((d - 1) & 31)
    return out


def greedy(bits, M):
    """Retained flags [M]: site j is retained unless a retained i < j has bit j - i - 1 set in row i."""
    retained = np.zeros(M, bool)
    blocked = 0  # bit j: site j is linked to an earlier retained site
    for j in range(M):
        if (blocked >> j) & 1:
            continue
        retained[j] = True
        blocked |= int.from_bytes(bits[j].tobytes(), "little") << (j + 1)
    return retained


def ld_prune(get_rows, n_variants, off, window, positions, r2_threshold, max_distance=None, min_maf=0.0,
             max_missing=0.0, site_range=None, chunk=16384):
    """dict(kept, M, pairs, linked_pairs, retained (matrix rows), bits) of fm_haplotype_ld_prune."""
    out = linked_bits(get_rows, n_variants, off, window, positions, r2_threshold, max_distance, min_maf, max_missing,
                      site_range, chunk)
    out["retained"] = out["kept"][greedy(out["bits"], out["M"])]
    return out
