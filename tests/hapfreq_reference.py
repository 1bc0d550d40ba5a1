"""numpy restatement of haplotype frequencies (fm_haplotype_frequencies, include/ferromic_gpu.h; DESIGN.md §3 and §4
"Haplotype frequencies").  Kept sites are those of tests/pca_reference.py::site_stats (as tests/ld_reference.py takes
them), limited to a site list by intersection; windows follow the header's three modes; a haplotype with a missing cell
in a window is dropped from it; keys are grouped with np.unique(axis=0).  The statistics are the header's single FP64
divisions of exact integers, so they equal the device's bit for bit."""
import numpy as np

from tests.pca_reference import offsets, rows_from_arrays, site_stats  # noqa: F401  (re-exported for the tests)

NAN = float("nan")


def count_windows(M, size, step=None):
    """(first, sites) of the count windows: [w step, w step + size) for every w that fits in M kept sites."""
    step = step or size
    return [(f, size) for f in range(0, M - size + 1, step)] if M >= size else []


def position_windows(kept_positions, windows):
    """(first, sites) of 0-based inclusive (start, end) position windows over the kept sites' (ascending) positions."""
    out = []
    for s, e in windows:
        a = int(np.searchsorted(kept_positions, s, "left"))
        b = max(a, int(np.searchsorted(kept_positions, e, "right")))
        out.append((a, b - a))
    return out


def statistics(sizes):
    """(N, K, (c1, c2, c3), s2, h1, h12, h123, h2_h1, diversity) of a window's class sizes, in the header's order."""
    c = sorted((int(x) for x in sizes), reverse=True)
    N, K = sum(c), len(c)
    c1, c2, c3 = (c + [0, 0, 0])[:3]
    s2 = sum(x * x for x in c)
    nn = float(N * N)
    if N == 0:
        return N, K, (c1, c2, c3), s2, NAN, NAN, NAN, NAN, NAN
    h1 = float(s2) / nn
    h12 = float(s2 + 2 * c1 * c2) / nn
    h123 = float(s2 + 2 * (c1 * c2 + c1 * c3 + c2 * c3)) / nn
    h2_h1 = float(s2 - c1 * c1) / float(s2)
    div = float(N * N - s2) / float(N * (N - 1)) if N > 1 else NAN
    return N, K, (c1, c2, c3), s2, h1, h12, h123, h2_h1, div


def class_sizes(keys):
    """Class sizes (descending) of the rows of a bool [N, s] key matrix."""
    N, s = keys.shape
    if N == 0:
        return np.zeros(0, np.int64)
    if s == 0:
        return np.array([N], np.int64)
    _, cnt = np.unique(np.packbits(keys, axis=1), axis=0, return_counts=True)
    return np.sort(cnt)[::-1].astype(np.int64)


def haplotype_frequencies(raw, called, off, min_maf=0.0, max_missing=0.0, site_range=None, sites=None, size=None,
                          step=None, windows=None, positions=None):
    """raw / called [V, cells]; off the haplotype offsets.  windows are position pairs (with `positions`, the matrix
    rows' positions); size / step count windows; neither: one window.  Returns dict(kept, n, M, windows [(first,
    sites)], n_used, distinct, top [k, 3], sum_sq, h1, h12, h123, h2_h1, diversity (arrays over the windows), counts
    (list of descending class-size arrays))."""
    off = np.asarray(off, dtype=np.int64)
    V = raw.shape[0]
    v_lo, v_hi = (0, V) if site_range is None else site_range
    kept = site_stats(rows_from_arrays(raw, called), v_lo, v_hi, off, min_maf, max_missing)[0]
    if sites is not None:
        kept = kept[np.isin(kept, np.asarray(sites, np.int64))]
    M = len(kept)
    if size is not None:
        wins = count_windows(M, size, step)
    elif windows is not None:
        wins = position_windows(np.asarray(positions, np.int64)[kept], windows)
    else:
        wins = [(0, M)]
    X = (raw[kept][:, off] == 1) & called[kept][:, off]  # [M, n] key bits
    Cm = called[kept][:, off]
    out = dict(kept=kept, n=len(off), M=M, windows=wins, counts=[])
    cols = {k: [] for k in ("n_used", "distinct", "top", "sum_sq", "h1", "h12", "h123", "h2_h1", "diversity")}
    for f, s in wins:
        used = Cm[f:f + s].all(axis=0)
        sizes = class_sizes(X[f:f + s].T[used])
        N, K, top, s2, h1, h12, h123, h21, div = statistics(sizes)
        for k, v in zip(cols, (N, K, top, s2, h1, h12, h123, h21, div)):
            cols[k].append(v)
        out["counts"].append(sizes)
    for k, v in cols.items():
        dt = np.float64 if k in ("h1", "h12", "h123", "h2_h1", "diversity") else np.int64
        out[k] = np.asarray(v, dt).reshape(len(wins), 3) if k == "top" else np.asarray(v, dt)
    return out
