"""GPU site frequency spectra (fm_site_frequency_spectrum / fm_joint_site_frequency_spectrum) against the numpy
restatement of tests/sfs_reference.py: spectra within 1e-9 |ref| + 1e-290 (exactly equal when every contributing row
has N == m), counts exactly.  Every resident matrix form, ploidy 1 and 2, haplotype lists, projections, windows, a
region and a site list, folding, the joint pass and its tile edges, a 10^5-site x 5008-haplotype case, device weights
against exact rationals, repeated calls and threads, the size query and the argument errors, and the tie to the
existing per-window estimators."""
import ctypes as C
import math
import threading
from fractions import Fraction

import numpy as np
import pytest

from tests import pca_reference as pr
from tests import sfs_reference as sr
from tests.test_gpu_pca import _matrix

pytestmark = pytest.mark.gpu


def _all_haps(S, P):
    return [(s, h) for s in range(S) for h in range(P)]


def _cohort(seed, S, V, ploidy=2, missing=0.0):
    """(alleles u8 [V, S, ploidy], missing bool, positions): U-shaped allele frequencies, monomorphic rows included."""
    rng = np.random.default_rng(seed)
    f = rng.beta(0.3, 0.3, V)
    f[::19] = 0.0
    a = (rng.random((V, S, ploidy)) < f[:, None, None]).astype(np.uint8)
    miss = rng.random((V, S, ploidy)) < missing
    a[miss] = 0
    return a, miss, np.cumsum(rng.integers(1, 20, size=V)).astype(np.int64)


def _rows(pos, windows):
    return [(int(np.searchsorted(pos, s, "left")), max(int(np.searchsorted(pos, e, "right")),
                                                       int(np.searchsorted(pos, s, "left")))) for s, e in windows]


def _close(got, ref):
    assert got.shape == ref.shape
    assert np.all(np.abs(got - ref) <= 1e-9 * np.abs(ref) + 1e-290), np.max(np.abs(got - ref))


def _same(x, y):
    x, y = np.asarray(x, np.float64), np.asarray(y, np.float64)
    return np.array_equal(np.isnan(x), np.isnan(y)) and np.allclose(x[~np.isnan(x)], y[~np.isnan(y)], rtol=1e-9,
                                                                       atol=1e-300)


def _run(m, a, miss, pos, haps, proj=None, region=None, windows=None, sites=None, folded=False):
    from ferromic_b200.api import _matrix_sfs
    got = _matrix_sfs(m, haps, proj, region, windows, folded, sites)
    V, S, P = a.shape
    raw, called = a.reshape(V, -1), ~miss.reshape(V, -1)
    off = pr.offsets(haps, S, P)
    mm = len(off) if proj is None else proj
    site_range = None if region is None else _rows(pos, [region])[0]
    ref = sr.sfs(raw, called, off, mm, site_range, sites, None if windows is None else _rows(pos, windows))
    info = got["info"]
    assert got["offsets"].tolist() == off.tolist()
    assert int(info.projection) == mm and int(info.n_haplotypes) == len(off)
    assert (int(info.n_sites), int(info.projected_out), int(info.non_biallelic), int(info.candidates)) == (
        ref["n_sites"], ref["projected_out"], ref["non_biallelic"], ref["candidates"])
    assert got["window_sites"].tolist() == ref["window_sites"].tolist()
    xi = ref["spectrum"]
    st = np.array([sr.stats(x, mm) for x in xi])
    assert np.array_equal(got["segregating"], st[:, 0]) or _same(got["segregating"], st[:, 0])
    for k, key in enumerate(("segregating", "theta_pi", "theta_w", "tajimas_d")):
        assert _same(got[key], st[:, k]), key
    _close(got["spectrum"], np.array([sr.fold(x, mm) for x in xi]) if folded else xi)
    return got, ref


@pytest.mark.parametrize("form", ["u8", "inband", "nomiss", "packed-dense", "packed-sparse", "lut"])
def test_matrix_forms(form):
    a, miss, pos = _cohort(11, 80, 1500, missing=0.0 if form == "nomiss" else 0.01)
    if form == "lut":  # values above 15 go through the rank LUT; the counts must see the raw values
        a[::7, :3, 0] = 254
        a[5::11] *= 17
    m = _matrix(form, a, miss, pos)
    haps = _all_haps(80, 2)
    for proj in (None, 150):
        got, ref = _run(m, a, miss, pos, haps, proj, (int(pos[20]), int(pos[1400])))
        assert ref["n_sites"] > 150
        if form == "lut":
            assert ref["non_biallelic"] > 100
        if form == "nomiss" and proj is None:
            assert np.array_equal(got["spectrum"], ref["spectrum"])  # every N == m: integer counts


@pytest.mark.parametrize("ploidy", [1, 2])
def test_ploidy_and_haplotype_lists(ploidy):
    a, miss, pos = _cohort(12 + ploidy, 100, 700, ploidy=ploidy, missing=0.02)
    for form in ("u8", "packed-dense", "inband"):
        _run(_matrix(form, a, miss, pos), a, miss, pos, _all_haps(100, 2), 60)
    m = _matrix("u8", a, miss, pos)
    for haps in ([(s, h) for s in (5, 9, 17, 40, 41, 77, 90) for h in (1, 0)],
                 [(s, h) for s in range(0, 100, 2) for h in (0, 1)] * 2 + [(3, 1)],
                 [(s, h) for s in range(60, 130) for h in (0, 1)]):
        n = len(pr.offsets(haps, 100, ploidy))
        _run(m, a, miss, pos, haps, max(1, n - 3))


def test_projections_and_folding():
    a, miss, pos = _cohort(14, 40, 900, missing=0.02)
    a[::50, 7, 1] = 2  # a third allele: non_biallelic
    m = _matrix("u8", a, miss, pos)
    haps = _all_haps(40, 2)
    for proj in (1, 2, 3, 4, 20, 79, 80):
        for folded in (False, True):
            got, ref = _run(m, a, miss, pos, haps, proj, folded=folded)
            assert ref["non_biallelic"] == 18
    a0, miss0, pos0 = _cohort(15, 40, 900)
    m0 = _matrix("u8", a0, miss0, pos0)
    got, ref = _run(m0, a0, miss0, pos0, haps)
    assert np.array_equal(got["spectrum"], ref["spectrum"])


def test_windows_region_and_site_list():
    from ferromic_b200.api import _matrix_sfs
    a, miss, pos = _cohort(16, 30, 3000, missing=0.01)
    m = _matrix("u8", a, miss, pos)
    haps = _all_haps(30, 2)
    p0, p1 = int(pos[0]), int(pos[-1])
    windows = [(p0, p0 + 500), (p0 + 200, p0 + 900), (p1 + 10, p1 + 100), (-50, -1), (p0 + 7, p0 + 6),
               (int(pos[100]), int(pos[100])), (p0 - 100, p1 + 100), (int(pos[2000]), int(pos[2999]))]
    for folded in (False, True):
        got, ref = _run(m, a, miss, pos, haps, 55, windows=windows, folded=folded)
        assert got["window_sites"][2] == got["window_sites"][3] == got["window_sites"][4] == 0
    edges = np.linspace(p0, p1 + 1, 1001).astype(np.int64)
    many = [(int(edges[i]), int(edges[i + 1]) - 1) for i in range(1000)]
    got, ref = _run(m, a, miss, pos, haps, 58, windows=many)
    assert got["spectrum"].shape == (1000, 59) and int(got["window_sites"].sum()) == ref["n_sites"]
    sites = np.sort(np.random.default_rng(3).choice(3000, 700, replace=False))
    _run(m, a, miss, pos, haps, 50, region=(int(pos[300]), int(pos[2500])), sites=sites)
    _run(m, a, miss, pos, haps, 50, windows=windows, sites=sites)
    got = _matrix_sfs(m, haps, 50, sites=[])
    assert int(got["info"].candidates) == 0 and not got["spectrum"].any()
    with pytest.raises(ValueError, match="exclusive"):
        _matrix_sfs(m, haps, 50, region=(p0, p1), windows=windows)


def _joint(m, a, miss, haps1, haps2, proj=None, region=None, sites=None, folded=False, pos=None):
    from ferromic_b200.api import _matrix_joint_sfs
    got = _matrix_joint_sfs(m, haps1, haps2, proj, region, folded, sites)
    V, S, P = a.shape
    raw, called = a.reshape(V, -1), ~miss.reshape(V, -1)
    o1, o2 = pr.offsets(haps1, S, P), pr.offsets(haps2, S, P)
    m1, m2 = (len(o1), len(o2)) if proj is None else proj
    site_range = None if region is None else _rows(pos, [region])[0]
    ref = sr.joint_sfs(raw, called, o1, o2, m1, m2, site_range, sites)
    info = got["info"]
    assert (int(info.projection1), int(info.projection2)) == (m1, m2)
    assert (int(info.n_sites), int(info.projected_out), int(info.non_biallelic), int(info.candidates)) == (
        ref["n_sites"], ref["projected_out"], ref["non_biallelic"], ref["candidates"])
    _close(got["spectrum"], sr.fold(ref["spectrum"], m1, m2) if folded else ref["spectrum"])
    return got, ref


def test_joint_sets():
    a, miss, pos = _cohort(17, 60, 1200, missing=0.02)
    a[::40, 3, 0] = 3
    m = _matrix("u8", a, miss, pos)
    left = [(s, h) for s in range(30) for h in (0, 1)]
    right = [(s, h) for s in range(30, 60) for h in (0, 1)]
    overlap = [(s, h) for s in range(20, 45) for h in (0, 1)]
    small = [(s, 0) for s in range(50, 60)] + [(99, 0)]
    for h1, h2, proj in ((left, right, (55, 56)), (left, overlap, (58, 47)), (small, left, (9, 50)),
                         (right, right, None), (left, right, None)):
        for folded in (False, True):
            _joint(m, a, miss, h1, h2, proj, folded=folded)
    got, ref = _joint(m, a, miss, left, right, (50, 52), region=(int(pos[100]), int(pos[900])), pos=pos,
                      sites=np.arange(0, 1200, 3))
    assert ref["non_biallelic"] > 0
    pk = _matrix("packed-sparse", *_cohort(18, 60, 600, missing=0.01))
    a2, miss2, _ = _cohort(18, 60, 600, missing=0.01)
    _joint(pk, a2, miss2, left, right, (57, 58))


@pytest.mark.parametrize("m1,m2", [(14, 15), (15, 16), (16, 31), (31, 32), (32, 14), (47, 1), (1, 48)])
def test_joint_tile_edges(m1, m2):
    """(m1 + 1, m2 + 1) around multiples of the 16 x 16 tile."""
    a, miss, pos = _cohort(19, 50, 500, missing=0.03)
    m = _matrix("u8", a, miss, pos)
    h1 = [(s, h) for s in range(25) for h in (0, 1)]
    h2 = [(s, h) for s in range(25, 50) for h in (0, 1)]
    _joint(m, a, miss, h1, h2, (m1, m2))


def test_large_cohort():
    """10^5 sites x 5008 haplotypes (2504 diploid samples) at 1 % missing, projected to 4930 and to 20."""
    V, S = 100_000, 2504
    rng = np.random.default_rng(20)
    f = rng.beta(0.2, 0.2, V)
    a = np.empty((V, S, 2), np.uint8)
    miss = np.empty((V, S, 2), bool)
    for i in range(0, V, 10_000):  # in slices to bound host memory
        a[i:i + 10_000] = rng.random((min(10_000, V - i), S, 2)) < f[i:i + 10_000, None, None]
        miss[i:i + 10_000] = rng.random((min(10_000, V - i), S, 2)) < 0.01
    a[miss] = 0
    pos = np.arange(V, dtype=np.int64) * 10
    m = _matrix("u8", a, miss, pos)
    haps = _all_haps(S, 2)
    for proj in (4930, 20):
        got, ref = _run(m, a, miss, pos, haps, proj)
        assert ref["n_sites"] > 0.9 * V


def test_device_weights_are_exact():
    """One row per (N, a) with N <= 12, every m <= N, one window per row: each window's spectrum is that row's
    weights, within 1e-12 of the exact rational and exactly zero outside the support."""
    from ferromic_b200.api import _matrix_sfs
    n = 12
    rows = [(N, k) for N in range(1, n + 1) for k in range(N + 1)]
    a = np.zeros((len(rows), n, 1), np.uint8)
    miss = np.zeros_like(a, bool)
    for v, (N, k) in enumerate(rows):
        a[v, :k, 0] = 1
        miss[v, N:, 0] = True
    pos = np.arange(len(rows), dtype=np.int64) * 2
    m = _matrix("u8", a, miss, pos)
    windows = [(int(p), int(p)) for p in pos]
    for proj in range(1, n + 1):
        got = _matrix_sfs(m, _all_haps(n, 1), proj, windows=windows)
        for v, (N, k) in enumerate(rows):
            xi = got["spectrum"][v]
            if N < proj:
                assert not xi.any()
                continue
            lo, w = sr.weights_exact(N, k, proj)
            assert not xi[:lo].any() and not xi[lo + len(w):].any()
            for x, f in zip(xi[lo:lo + len(w)], w):
                assert abs(Fraction(float(x)) - f) <= Fraction(1, 10 ** 12) * f


def test_repeated_calls_and_threads_bit_identical():
    from ferromic_b200.api import _matrix_joint_sfs, _matrix_sfs
    a, miss, pos = _cohort(21, 60, 20_000, missing=0.02)
    m = _matrix("u8", a, miss, pos)
    haps = _all_haps(60, 2)
    h1, h2 = haps[:60], haps[60:]
    first = _matrix_sfs(m, haps, 110)
    jfirst = _matrix_joint_sfs(m, h1, h2, (55, 54))
    out, errs = [None] * 4, []

    def work(i):
        try:
            out[i] = (_matrix_sfs(m, haps, 110), _matrix_joint_sfs(m, h1, h2, (55, 54)))
        except Exception as e:  # pragma: no cover - reported below
            errs.append(e)
    ts = [threading.Thread(target=work, args=(i,)) for i in range(4)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errs
    for r, j in out + [(_matrix_sfs(m, haps, 110), _matrix_joint_sfs(m, h1, h2, (55, 54)))]:
        assert np.array_equal(r["spectrum"].view(np.uint64), first["spectrum"].view(np.uint64))
        assert np.array_equal(r["tajimas_d"].view(np.uint64), first["tajimas_d"].view(np.uint64))
        assert np.array_equal(j["spectrum"].view(np.uint64), jfirst["spectrum"].view(np.uint64))


def test_size_query_and_errors():
    import ferromic_b200 as fm
    from ferromic_b200 import _lib
    from ferromic_b200.api import _Matrix, _matrix_joint_sfs, _matrix_sfs
    a, miss, pos = _cohort(22, 20, 300, missing=0.01)
    m = _matrix("u8", a, miss, pos)
    haps = _all_haps(20, 2)
    idx = np.asarray([h[0] for h in haps], np.uint64)
    side = np.asarray([h[1] for h in haps], np.uint8)
    L = _lib.lib()

    def call(prm, spec=None, cap=0, windows=None, hs=(idx, side)):
        info = _lib.SfsInfo()
        p = lambda x: None if x is None else x.ctypes.data  # noqa: E731
        nw = 0 if windows is None else len(windows)
        st = L.fm_site_frequency_spectrum(m.handle, p(hs[0]), p(hs[1]), len(hs[0]), C.byref(prm), p(windows), nw,
                                          None, p(spec), cap, None, None, None, None, None, C.byref(info))
        return st, info, L.fm_last_error().decode()
    st, info, msg = call(_lib.SfsParams(30, 0, 0, 0, 0))
    assert st == _lib.FM_ERR_INVALID_ARG and "capacity too small" in msg
    assert info.n_haplotypes == 40 and info.projection == 30
    w = np.array([[0, 100], [50, 400]], np.int64)
    st, info, msg = call(_lib.SfsParams(0, 0, 0, 0, 0), np.zeros(81), 81, w)
    assert st == _lib.FM_ERR_INVALID_ARG and "capacity too small" in msg and info.projection == 40
    spec = np.zeros(82)
    st, info, msg = call(_lib.SfsParams(0, 0, 0, 0, 0), spec, 82, w)
    assert st == _lib.FM_OK and info.n_sites > 0
    for prm, what in ((_lib.SfsParams(41, 0, 0, 0, 0), "projection"), (_lib.SfsParams(0, 0, 1, 0, 100), "exclusive")):
        st, _, msg = call(prm, spec, 82, w if what == "exclusive" else None)
        assert st == _lib.FM_ERR_INVALID_ARG and what in msg, msg
    st, _, msg = call(_lib.SfsParams(0, 0, 0, 0, 0), spec, 82, hs=(np.array([99], np.uint64), np.array([0], np.uint8)))
    assert st == _lib.FM_ERR_INVALID_ARG and "empty" in msg
    info = _lib.SfsInfo()
    assert L.fm_site_frequency_spectrum(m.handle, None, None, 0, None, None, 0, None, None, 0, None, None, None, None,
                                        None, C.byref(info)) == _lib.FM_ERR_INVALID_ARG
    for sites, what in (([5, 3, 9], "ascending"), ([3, 3, 9], "ascending"), ([3, 300], "beyond")):
        with pytest.raises(ValueError, match=what):
            _matrix_sfs(m, haps, sites=sites)
        with pytest.raises(ValueError, match=what):
            _matrix_joint_sfs(m, haps[:10], haps[10:], sites=sites)
    with pytest.raises(ValueError, match="projection"):
        _matrix_joint_sfs(m, haps[:10], haps[10:], (11, 5))
    jinfo = _lib.JointSfsInfo()
    jprm = _lib.JointSfsParams(5, 6, 0, 0, 0, 0)
    st = L.fm_joint_site_frequency_spectrum(m.handle, idx.ctypes.data, side.ctypes.data, 10, idx.ctypes.data,
                                            side.ctypes.data, 20, C.byref(jprm), None, 0, C.byref(jinfo))
    assert st == _lib.FM_ERR_INVALID_ARG and b"capacity too small" in L.fm_last_error()
    assert (jinfo.n_haplotypes1, jinfo.n_haplotypes2, jinfo.projection1, jinfo.projection2) == (10, 20, 5, 6)
    a3 = np.zeros((50, 10, 3), np.uint8)
    with pytest.raises(NotImplementedError, match="ploidy"):
        _matrix_sfs(_Matrix(a3, None, np.arange(50), ingest="u8"), [(0, 0), (1, 0)])
    with pytest.raises(NotImplementedError, match="streamed"):
        _matrix_sfs(_Matrix.ingest(a, miss, pos, [haps]), haps)
    unsorted = _matrix("u8", a, miss, pos[::-1].copy())
    with pytest.raises(NotImplementedError, match="sorted"):
        _matrix_sfs(unsorted, haps, windows=[(0, 10)])
    with pytest.raises(NotImplementedError, match="sorted"):
        _matrix_joint_sfs(unsorted, haps[:10], haps[10:], region=(0, 10))
    big = _matrix("nomiss", np.zeros((4, 20000, 2), np.uint8), None, np.arange(4))
    with pytest.raises(NotImplementedError, match="2\\^28"):
        _matrix_joint_sfs(big, _all_haps(20000, 2)[:20000], _all_haps(20000, 2)[20000:])
    _run(m, a, miss, pos, haps, 33)  # the library is still usable
    res = fm.site_frequency_spectrum([(1, [[0, 1], [1, 1]]), (2, [[1, 0], [0, 0]])])
    assert res.projection == 4 and res.n_sites == 2 and res.spectrum.tolist() == [0.0, 1.0, 0.0, 1.0, 0.0]
    js = fm.joint_site_frequency_spectrum([(1, [[0, 1], [1, 1]]), (2, [[1, 0], [0, 0]])], [(0, 0), (0, 1)],
                                          [(1, 0), (1, 1)])
    assert js.projection == (2, 2) and js.spectrum.tolist() == [[0, 0, 0], [1, 0, 1], [0, 0, 0]]


def test_tie_to_existing_estimators():
    """Without missing data at m = n: S equals fm_group_window_sums' segregating sites exactly, theta_pi its pi_sum
    within 1e-12 and theta_W equals watterson_theta(S, n, 1) within 1e-12."""
    import ferromic_b200 as fm
    from ferromic_b200 import _lib
    from ferromic_b200.api import _matrix_sfs
    a, miss, pos = _cohort(23, 50, 5000)
    m = _matrix("u8", a, miss, pos)
    haps = _all_haps(50, 2)
    p0, p1 = int(pos[0]), int(pos[-1])
    windows = np.array([(s, s + 3999) for s in range(p0, p1 + 1, 4000)], np.int64)
    nw = len(windows)
    got = _matrix_sfs(m, haps, windows=windows)
    nv = np.zeros(nw, np.uint64)
    seg = np.zeros(nw, np.uint64)
    unc = np.zeros(nw, np.uint64)
    pis = np.zeros(nw)
    g = m.group(haps)
    _lib.check(_lib.lib().fm_group_window_sums(g.handle, windows.ctypes.data, nw, nv.ctypes.data, seg.ctypes.data,
                                               pis.ctypes.data, unc.ctypes.data))
    assert got["segregating"].tolist() == seg.astype(np.float64).tolist()
    np.testing.assert_allclose(got["theta_pi"], pis, rtol=1e-12, atol=0)
    for w in range(nw):
        expect = fm.watterson_theta(int(seg[w]), 100, 1)
        assert got["theta_w"][w] == pytest.approx(expect, rel=1e-12)
        assert math.isnan(got["tajimas_d"][w]) or seg[w] > 0
