"""numpy restatement of haplotype PCA (fm_haplotype_pca, include/ferromic_gpu.h; DESIGN.md §3 and §4 "Haplotype
PCA").  Site counts, filters and standardization follow the definition literally; the products run over site
chunks, so 10^6 sites need no dense Z; orth is numpy.linalg.qr and the eigenproblem numpy.linalg.eigh."""
import numpy as np

from tests.synth import _mix


def offsets(haplotypes, n_samples, ploidy):
    """fm_group_create semantics: sample * ploidy + side, sorted and de-duplicated; out-of-range samples and side 1
    at ploidy 1 dropped."""
    return np.asarray(sorted({s * ploidy + h for s, h in haplotypes if s < n_samples and (h == 0 or ploidy > 1)}),
                      dtype=np.int64)


def rows_from_arrays(raw, called):
    """get_rows for in-memory [V, cells] arrays of raw allele values and called flags."""
    return lambda a, b: (raw[a:b], called[a:b])


def rademacher(seed, rows, l):
    """G[v, c] = +1 when bit 63 of fm_mix(seed, v, c) is clear, else -1; v = matrix rows."""
    h = _mix(seed, np.asarray(rows, dtype=np.uint64)[:, None], np.arange(l, dtype=np.uint64)[None, :])
    return np.where((h >> np.uint64(63)) == 0, 1.0, -1.0)


def site_stats(get_rows, v_lo, v_hi, off, min_maf, max_missing, chunk=16384):
    """(kept matrix rows, called, alt) of the kept sites of [v_lo, v_hi)."""
    n = len(off)
    kept, cal, alt = [], [], []
    for a in range(v_lo, v_hi, chunk):
        b = min(v_hi, a + chunk)
        x, c = get_rows(a, b)
        x, c = x[:, off], c[:, off]
        called = c.sum(axis=1)
        alt_v = (c & (x == 1)).sum(axis=1)
        other = (c & (x != 0) & (x != 1)).sum(axis=1)
        minor = np.minimum(alt_v, called - alt_v)
        keep = ((other == 0) & (alt_v > 0) & (alt_v < called) &
                ((n - called).astype(np.float64) <= max_missing * float(n)) &
                (minor.astype(np.float64) >= min_maf * called.astype(np.float64)))
        kept.append(np.arange(a, b)[keep])
        cal.append(called[keep])
        alt.append(alt_v[keep])
    cat = lambda xs: np.concatenate(xs) if xs else np.zeros(0, np.int64)  # noqa: E731
    return cat(kept).astype(np.int64), cat(cal).astype(np.int64), cat(alt).astype(np.int64)


def haplotype_pca(get_rows, n_variants, off, k, oversampling=10, power_iterations=4, min_maf=0.0, max_missing=0.0,
                  seed=0, site_range=None, loadings=False, chunk=16384, dense=False):
    """Returns dict(kept, n, M, l, T, scores, singular_values, explained_variance_ratio, loadings[, Z])."""
    off = np.asarray(off, dtype=np.int64)
    n = len(off)
    v_lo, v_hi = (0, n_variants) if site_range is None else site_range
    kept, called, alt = site_stats(get_rows, v_lo, v_hi, off, min_maf, max_missing, chunk)
    M = len(kept)
    T = int(called.sum())
    l = min(k + oversampling, n, M)
    p = alt.astype(np.float64) / called.astype(np.float64)
    s = 1.0 / np.sqrt(p * (1.0 - p))
    u1, u0 = s * (1.0 - p), s * (0.0 - p)

    # Z restricted to kept sites, chunk by chunk (n x m blocks)
    blocks = []
    for j in range(0, M, chunk):
        rows = kept[j:j + chunk]
        blocks.append((j, rows))

    every_cell = None

    def z_block(j, rows):
        nonlocal every_cell
        x, c = get_rows(int(rows[0]), int(rows[-1]) + 1)
        if every_cell is None:
            every_cell = len(off) == x.shape[1] and np.array_equal(off, np.arange(x.shape[1]))
        if len(rows) != rows[-1] - rows[0] + 1:
            x, c = x[rows - rows[0]], c[rows - rows[0]]
        if not every_cell:
            x, c = x[:, off], c[:, off]
        sl = slice(j, j + len(rows))
        z = np.where(x == 1, u1[sl][:, None], u0[sl][:, None])
        z *= c
        return z.T  # n x m

    def z_times(R):  # Z R, R is M x l
        Y = np.zeros((n, R.shape[1]))
        for j, rows in blocks:
            Y += z_block(j, rows) @ R[j:j + len(rows)]
        return Y

    def zt_times(Q):  # Z^T Q
        W = np.zeros((M, Q.shape[1]))
        for j, rows in blocks:
            W[j:j + len(rows)] = z_block(j, rows).T @ Q
        return W

    Y = np.zeros((n, l))
    for j, rows in blocks:
        Y += z_block(j, rows) @ rademacher(seed, rows, l)
    Q = np.linalg.qr(Y)[0]
    for _ in range(power_iterations):
        Q = np.linalg.qr(z_times(zt_times(Q)))[0]
    W = zt_times(Q)
    lam, E = np.linalg.eigh(W.T @ W)
    lam, E = lam[::-1], E[:, ::-1]
    sig = np.sqrt(np.maximum(lam[:k], 0.0))
    scores = (Q @ E[:, :k]) * sig
    flip = np.where(scores[np.argmax(np.abs(scores), axis=0), np.arange(k)] < 0, -1.0, 1.0)
    scores *= flip
    out = dict(kept=kept, n=n, M=M, l=l, T=T, scores=scores, singular_values=sig,
               explained_variance_ratio=sig * sig / T, loadings=None)
    if loadings:
        out["loadings"] = (W @ E[:, :k]) / sig * flip
    if dense:
        out["Z"] = np.concatenate([z_block(j, rows) for j, rows in blocks], axis=1) if blocks else np.zeros((n, 0))
    return out


def cohort(seed, n_pops, per_pop, V, ploidy=2, missing=0.0, spread=0.35):
    """Structured test cohort: (alleles u8 [V, S, ploidy], missing bool [V, S, ploidy], positions, pop_of_sample).
    Each population draws its allele frequency around a shared one, so the top n_pops - 1 components are
    population axes."""
    rng = np.random.default_rng(seed)
    S = n_pops * per_pop
    base = rng.uniform(0.1, 0.9, size=V)
    f = np.clip(base[:, None] + rng.uniform(-spread, spread, size=(V, n_pops)), 0.02, 0.98)
    pop = np.repeat(np.arange(n_pops), per_pop)
    a = (rng.random((V, S, ploidy)) < f[:, pop][:, :, None]).astype(np.uint8)
    miss = rng.random((V, S, ploidy)) < missing
    a[miss] = 0
    pos = np.cumsum(rng.integers(1, 20, size=V)).astype(np.int64)
    return a, miss, pos, pop
