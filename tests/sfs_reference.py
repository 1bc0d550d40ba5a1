"""numpy restatement of the site frequency spectra (fm_site_frequency_spectrum / fm_joint_site_frequency_spectrum,
include/ferromic_gpu.h; DESIGN.md §3 and §4 "Site frequency spectra").  Per-site counts and the classification follow
the definition literally.  Weights come two ways: exactly, as Fractions of binomial coefficients, and in FP64 by the
definition's rule (Loader's saddle-point form at the support's mode, then the exact ratio walked outward one bin at a
time).  Spectra are summed in row order (np.add.at is unbuffered and runs in index order)."""
import math
from fractions import Fraction

import numpy as np

# stirlerr(n) = log(n!) - log(sqrt(2 pi)) - (n + 1/2) log(n) + n for n = 1 .. 15 (to 25 digits)
_SFERR = [0.0, 8.1061466795327258219670264e-2, 4.1340695955409294093822081e-2, 2.7677925684998339148789293e-2,
          2.0790672103765093111522772e-2, 1.6644691189821192163194865e-2, 1.3876128823070747998745727e-2,
          1.1896709945891770095055724e-2, 1.0411265261972096497478567e-2, 9.2554621827127329177286366e-3,
          8.3305634333628712564693187e-3, 7.5736754879518407949720242e-3, 6.9428401072095298656641527e-3,
          6.4089941880042070684396311e-3, 5.9513701127588477356244160e-3, 5.5547335519628013710386900e-3]
_S0, _S1, _S2, _S3, _S4 = 1.0 / 12, 1.0 / 360, 1.0 / 1260, 1.0 / 1680, 1.0 / 1188
_LN_2PI = 1.837877066409345483560659472811


def stirlerr(n):
    if n <= 15:
        return _SFERR[int(n)]
    nn = float(n) * float(n)
    n = float(n)
    if n > 500:
        return (_S0 - _S1 / nn) / n
    if n > 80:
        return (_S0 - (_S1 - _S2 / nn) / nn) / n
    if n > 35:
        return (_S0 - (_S1 - (_S2 - _S3 / nn) / nn) / nn) / n
    return (_S0 - (_S1 - (_S2 - (_S3 - _S4 / nn) / nn) / nn) / nn) / n


def bd0(x, np_):
    if abs(x - np_) < 0.1 * (x + np_):
        v = (x - np_) / (x + np_)
        s = (x - np_) * v
        ej = 2.0 * x * v
        v = v * v
        for j in range(1, 1000):
            ej *= v
            s1 = s + ej / (2 * j + 1)
            if s1 == s:
                return s1
            s = s1
    return x * math.log(x / np_) + np_ - x


def dbinom_raw(x, n, p, q):
    if p == 0.0:
        return 1.0 if x == 0 else 0.0
    if q == 0.0:
        return 1.0 if x == n else 0.0
    if x == 0:
        if n == 0:
            return 1.0
        return math.exp(-bd0(n, n * q) - n * p if p < 0.1 else n * math.log(q))
    if x == n:
        return math.exp(-bd0(n, n * p) - n * q if q < 0.1 else n * math.log(p))
    lc = stirlerr(n) - stirlerr(x) - stirlerr(n - x) - bd0(x, n * p) - bd0(n - x, n * q)
    lf = _LN_2PI + math.log(x) + math.log1p(-x / n)
    return math.exp(lc - 0.5 * lf)


def support(N, a, m):
    return max(0, m - (N - a)), min(a, m)


def mode(N, a, m):
    lo, hi = support(N, a, m)
    return min(max((m + 1) * (a + 1) // (N + 2), lo), hi)


def mode_weight(N, a, m):
    """h(mode; N, a, m) by Loader's form (R's dhyper): dbinom_raw(j, a) dbinom_raw(m - j, N - a) / dbinom_raw(m, N)
    at p = m / N.  A one-bin support has weight exactly 1."""
    lo, hi = support(N, a, m)
    if lo == hi:
        return 1.0
    j = mode(N, a, m)
    p = m / N
    q = (N - m) / N
    return dbinom_raw(j, a, p, q) * dbinom_raw(m - j, N - a, p, q) / dbinom_raw(m, N, p, q)


def weights_fp64(N, a, m):
    """(lo, FP64 weights of bins lo .. hi): the mode's value, then h(j + 1) = h(j) * r_up(j) upward and
    h(j - 1) = h(j) * r_down(j) downward, each ratio one division of two exact integer products."""
    lo, hi = support(N, a, m)
    md = mode(N, a, m)
    w = np.zeros(hi - lo + 1)
    h0 = mode_weight(N, a, m)
    w[md - lo] = h0
    h = h0
    for j in range(md, hi):
        h *= float((a - j) * (m - j)) / float((j + 1) * (N - a - m + j + 1))
        w[j + 1 - lo] = h
    h = h0
    for j in range(md, lo, -1):
        h *= float(j * (N - a - m + j)) / float((a - j + 1) * (m - j + 1))
        w[j - 1 - lo] = h
    return lo, w


def weights_exact(N, a, m):
    """(lo, [Fraction]) of C(a, j) C(N - a, m - j) / C(N, m) over the support."""
    lo, hi = support(N, a, m)
    den = math.comb(N, m)
    return lo, [Fraction(math.comb(a, j) * math.comb(N - a, m - j), den) for j in range(lo, hi + 1)]


def site_counts(raw, called, off):
    """(called, alt, other) per row over the cells `off` of [V, cells] arrays of raw values and called flags."""
    x, c = raw[:, off], called[:, off]
    return (c.sum(axis=1).astype(np.int64), (c & (x == 1)).sum(axis=1).astype(np.int64),
            (c & (x != 0) & (x != 1)).sum(axis=1).astype(np.int64))


def candidate_rows(V, site_range=None, sites=None):
    """Matrix rows of the region (site_range = (v_lo, v_hi), None: every row) that are in the site list."""
    v_lo, v_hi = (0, V) if site_range is None else site_range
    rows = np.arange(v_lo, v_hi)
    if sites is not None:
        rows = rows[np.isin(rows, np.asarray(sites, np.int64))]
    return rows


class _Weights:
    """Memoized FP64 (or exact) weights per (N, a, m)."""

    def __init__(self, exact=False):
        self.exact = exact
        self.cache = {}

    def __call__(self, N, a, m):
        key = (int(N), int(a), int(m))
        if key not in self.cache:
            if self.exact:
                lo, w = weights_exact(*key)
                self.cache[key] = (lo, np.array([float(f) for f in w]))
            else:
                self.cache[key] = weights_fp64(*key)
        return self.cache[key]


def classify(called, alt, other, m):
    """(contributing mask, projected_out mask, non_biallelic mask) of candidate rows, in the definition's order."""
    nb = other > 0
    po = ~nb & (called < m)
    return ~nb & ~po, po, nb


def sfs(raw, called, off, m, site_range=None, sites=None, windows=None, exact=False):
    """1-D spectrum: dict(spectrum [n_windows, m + 1] (one window without `windows`), window_sites, n_sites,
    projected_out, non_biallelic, candidates).  windows: matrix-row ranges [lo, hi) of the candidate rows."""
    V = raw.shape[0]
    rows = candidate_rows(V, site_range, sites)
    cal, alt, oth = site_counts(raw[rows], called[rows], off)
    contrib, po, nb = classify(cal, alt, oth, m)
    wf = _Weights(exact)
    ranges = [(0, V)] if windows is None else windows
    out = np.zeros((len(ranges), m + 1))
    wsites = np.zeros(len(ranges), np.int64)
    for k, (lo, hi) in enumerate(ranges):
        sel = np.nonzero(contrib & (rows >= lo) & (rows < hi))[0]
        wsites[k] = len(sel)
        idx, val = [], []
        for i in sel:  # row order
            j0, w = wf(cal[i], alt[i], m)
            idx.append(np.arange(j0, j0 + len(w)))
            val.append(w)
        if idx:
            np.add.at(out[k], np.concatenate(idx), np.concatenate(val))
    return dict(spectrum=out, window_sites=wsites, n_sites=int(contrib.sum()), projected_out=int(po.sum()),
                non_biallelic=int(nb.sum()), candidates=len(rows))


def joint_sfs(raw, called, off1, off2, m1, m2, site_range=None, sites=None, exact=False):
    """Joint spectrum [m1 + 1, m2 + 1] and the counts; entries h1(j1) * h2(j2) summed in row order."""
    V = raw.shape[0]
    rows = candidate_rows(V, site_range, sites)
    c1, a1, o1 = site_counts(raw[rows], called[rows], off1)
    c2, a2, o2 = site_counts(raw[rows], called[rows], off2)
    nb = (o1 > 0) | (o2 > 0)
    po = ~nb & ((c1 < m1) | (c2 < m2))
    contrib = ~nb & ~po
    wf = _Weights(exact)
    out = np.zeros((m1 + 1) * (m2 + 1))
    idx, val = [], []
    for i in np.nonzero(contrib)[0]:
        l1, w1 = wf(c1[i], a1[i], m1)
        l2, w2 = wf(c2[i], a2[i], m2)
        j1 = np.arange(l1, l1 + len(w1))[:, None]
        j2 = np.arange(l2, l2 + len(w2))[None, :]
        idx.append((j1 * (m2 + 1) + j2).ravel())
        val.append((w1[:, None] * w2[None, :]).ravel())
    if idx:
        np.add.at(out, np.concatenate(idx), np.concatenate(val))
    return dict(spectrum=out.reshape(m1 + 1, m2 + 1), n_sites=int(contrib.sum()), projected_out=int(po.sum()),
                non_biallelic=int(nb.sum()), candidates=len(rows))


def fold(xi, m1, m2=0):
    """The fold rule with c(j) = (m1 - j1, m2 - j2), M = m1 + m2; a 1-D spectrum is m2 = 0."""
    x = np.asarray(xi, np.float64).reshape(m1 + 1, m2 + 1)
    out = np.zeros_like(x)
    M = m1 + m2
    for j1 in range(m1 + 1):
        for j2 in range(m2 + 1):
            c1, c2 = m1 - j1, m2 - j2
            s = 2 * (j1 + j2)
            if s < M or (s == M and (j1, j2) != (c1, c2) and 2 * j1 < m1):
                out[j1, j2] = x[j1, j2] + x[c1, c2]
            elif s == M and (j1, j2) == (c1, c2):
                out[j1, j2] = x[j1, j2]
    return out if m2 else out[:, 0]


def stats(xi, m):
    """(S, theta_pi, theta_W, Tajima's D) of an unfolded spectrum in the header's operation order."""
    xi = np.asarray(xi, np.float64)
    S = 0.0
    num = 0.0
    for j in range(1, m):
        S += xi[j]
        num += float(j * (m - j)) * xi[j]
    a1 = a2 = 0.0
    for i in range(1, m):
        a1 += 1.0 / i
        a2 += 1.0 / float(i * i)
    with np.errstate(divide="ignore", invalid="ignore"):
        tp = np.float64(num) / np.float64(m * (m - 1) // 2)
        tw = np.float64(S) / np.float64(a1)
    if m < 4:
        return S, float(tp), float(tw), float("nan")
    fm = float(m)
    b1 = (fm + 1.0) / (3.0 * (fm - 1.0))
    b2 = 2.0 * (fm * fm + fm + 3.0) / (9.0 * fm * (fm - 1.0))
    c1 = b1 - 1.0 / a1
    c2 = b2 - (fm + 2.0) / (a1 * fm) + a2 / (a1 * a1)
    e1 = c1 / a1
    e2 = c2 / (a1 * a1 + a2)
    rad = e1 * S + e2 * S * (S - 1.0)
    if not (rad > 0.0 and math.isfinite(rad)):
        return S, float(tp), float(tw), float("nan")
    return S, float(tp), float(tw), float((tp - tw) / math.sqrt(rad))
