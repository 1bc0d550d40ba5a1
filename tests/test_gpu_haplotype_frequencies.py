"""GPU haplotype frequencies (fm_haplotype_frequencies / haplotype_frequencies) against the numpy restatement of
tests/hapfreq_reference.py: kept sites, windows, N, K, the top three, sum c^2 and every class size exact, the FP64
statistics bit-identical.  Every resident matrix form, ploidy 1 and 2, haplotype lists, cohort sizes around a warp,
window sizes around a key word with starts off word boundaries, the three window modes, a region and a pruned site
list, excluded haplotypes, a constructed hash collision, a cohort wider than shared memory, the size query and the
errors, repeated calls and threads, and the tie to per-site pi.  The 8 GiB key limit needs a matrix of 8 GiB of
packed bits or 64 GiB of u8 cells and is not exercised here."""
import ctypes as C
import threading

import numpy as np
import pytest

from tests import hapfreq_reference as hr
from tests import pca_reference as pr
from tests.test_gpu_pca import _matrix

pytestmark = pytest.mark.gpu


def _all_haps(S, P):
    return [(s, h) for s in range(S) for h in range(P)]


def _cohort(seed, S, V, ploidy=2, missing=0.0, founders=12, mutation=0.004):
    """(alleles u8 [V, S, ploidy], missing bool, positions): every haplotype copies one of a few founders per block of
    40 sites (founder 0 at high frequency) with a small per-cell mutation rate, so windows hold shared haplotypes."""
    rng = np.random.default_rng(seed)
    n = S * ploidy
    fnd = rng.random((founders, V)) < rng.uniform(0.1, 0.6, V)
    a = np.empty((V, n), np.uint8)
    p = np.full(founders, 0.4 / (founders - 1))
    p[0] = 0.6
    for b in range(0, V, 40):
        pick = rng.choice(founders, size=n, p=p)
        a[b:b + 40] = fnd[pick, b:b + 40].T
    a ^= (rng.random((V, n)) < mutation).astype(np.uint8)
    a = a.reshape(V, S, ploidy)
    miss = rng.random((V, S, ploidy)) < missing
    a[miss] = 0
    return a, miss, np.cumsum(rng.integers(1, 20, size=V)).astype(np.int64)


def _rows(pos, region):
    return int(np.searchsorted(pos, region[0], "left")), int(np.searchsorted(pos, region[1], "right"))


def _bits_equal(x, y):
    x, y = np.asarray(x, np.float64), np.asarray(y, np.float64)
    return x.shape == y.shape and np.array_equal(x.view(np.uint64), y.view(np.uint64))


def _run(m, a, miss, pos, haps, size=None, step=None, windows=None, region=None, min_maf=0.0, max_missing=0.0,
         sites=None, counts=True):
    from ferromic_b200.api import _matrix_hapfreq
    got = _matrix_hapfreq(m, haps, size, step, windows, region, min_maf, max_missing, sites, counts)
    V, S, P = a.shape
    raw, called = a.reshape(V, -1), ~miss.reshape(V, -1)
    off = pr.offsets(haps, S, P)
    ref = hr.haplotype_frequencies(raw, called, off, min_maf, max_missing, None if region is None else _rows(pos, region),
                                   sites, size, step, windows, pos)
    info = got["info"]
    assert got["offsets"].tolist() == off.tolist()
    assert got["kept"].tolist() == ref["kept"].tolist()
    assert (int(info.n_haplotypes), int(info.n_sites), int(info.n_windows)) == (len(off), ref["M"], len(ref["windows"]))
    assert got["window_first"].tolist() == [f for f, _ in ref["windows"]]
    assert got["window_sites"].tolist() == [s for _, s in ref["windows"]]
    for k in ("n_used", "distinct", "sum_sq"):
        assert got[k].astype(np.int64).tolist() == ref[k].tolist(), k
    assert got["top_counts"].astype(np.int64).tolist() == ref["top"].tolist()
    for k in ("h1", "h12", "h123", "h2_h1", "diversity"):
        assert _bits_equal(got[k], ref[k]), k
    if counts:
        co = got["count_offsets"]
        assert co.tolist() == np.concatenate([[0], np.cumsum([len(c) for c in ref["counts"]])]).astype(int).tolist()
        for w, c in enumerate(ref["counts"]):
            assert got["counts"][co[w]:co[w + 1]].tolist() == c.tolist()
    return got, ref


@pytest.mark.parametrize("form", ["u8", "inband", "nomiss", "packed-dense", "packed-sparse", "lut"])
def test_matrix_forms(form):
    a, miss, pos = _cohort(11, 60, 1500, missing=0.0 if form == "nomiss" else 0.002)
    if form == "lut":  # values above 15 go through the rank LUT; keys and filters must see the raw values
        a[::7, :3, 0] = 254
        a[5::11] *= 17
    m = _matrix(form, a, miss, pos)
    haps = _all_haps(60, 2)
    for kw in (dict(), dict(size=65, step=30), dict(size=200, max_missing=0.02)):
        got, ref = _run(m, a, miss, pos, haps, **kw)
        assert ref["M"] > 500
    if form != "nomiss":
        assert min(ref["n_used"]) < 120  # haplotypes with a missing cell are left out


@pytest.mark.parametrize("ploidy", [1, 2])
def test_ploidy_and_haplotype_lists(ploidy):
    a, miss, pos = _cohort(12 + ploidy, 90, 900, ploidy=ploidy, missing=0.003)
    for form in ("u8", "packed-dense", "inband"):
        _run(_matrix(form, a, miss, pos), a, miss, pos, _all_haps(90, 2), size=100, step=40, max_missing=0.05)
    m = _matrix("u8", a, miss, pos)
    for haps in ([(s, h) for s in (5, 9, 17, 40, 41, 77, 89) for h in (1, 0)],
                 [(s, h) for s in range(0, 90, 2) for h in (0, 1)] * 2 + [(3, 1)],
                 [(s, h) for s in range(60, 130) for h in (0, 1)]):
        _run(m, a, miss, pos, haps, size=64, max_missing=0.05)


@pytest.mark.parametrize("n", [1, 31, 32, 33, 3000])
def test_cohort_sizes(n):
    a, miss, pos = _cohort(20 + n, n, 700, ploidy=1, founders=6)
    if n == 1:  # one haplotype keeps no site under the filters: no sites, one window of N = 1
        got, ref = _run(_matrix("u8", a, miss, pos), a, miss, pos, _all_haps(1, 1))
        assert ref["M"] == 0 and got["distinct"].tolist() == [1]
        return
    for form in ("u8", "packed-dense"):
        m = _matrix(form, a, miss, pos)
        _run(m, a, miss, pos, _all_haps(n, 1))
        _run(m, a, miss, pos, _all_haps(n, 1), size=65, step=17)


def test_window_edges():
    """Window sizes 1, 63, 64, 65 and over 1000 kept sites, steps below, above and equal to the size, starts off word
    boundaries, and position windows holding 0, 1 or many kept sites."""
    a, miss, pos = _cohort(30, 40, 2600)
    m = _matrix("u8", a, miss, pos)
    haps = _all_haps(40, 2)
    for size, step in ((1, None), (1, 3), (63, 5), (63, 100), (64, None), (64, 7), (65, 1), (65, 129), (1100, 333),
                       (1100, None)):
        got, ref = _run(m, a, miss, pos, haps, size=size, step=step)
        assert len(ref["windows"]) >= 1
    got, _ = _run(m, a, miss, pos, haps, size=5000)  # nothing fits: no window
    assert int(got["info"].n_windows) == 0 and got["h1"].size == 0
    p0, p1 = int(pos[0]), int(pos[-1])
    windows = [(p0 + 3 + 17 * i, p0 + 3 + 17 * i + 900 + 31 * i) for i in range(40)]
    windows += [(int(pos[100]), int(pos[100])), (int(pos[100]) + 1, int(pos[101]) - 1), (p0, p1)]
    got, ref = _run(m, a, miss, pos, haps, windows=windows)
    assert got["window_sites"][-2] == 0 and got["distinct"][-2] == 1 and got["h1"][-2] == 1.0


def test_position_windows_region_and_site_list():
    from ferromic_b200.api import _matrix_hapfreq, _matrix_ld_prune
    a, miss, pos = _cohort(31, 50, 3000, missing=0.002)
    m = _matrix("u8", a, miss, pos)
    haps = _all_haps(50, 2)
    p0, p1 = int(pos[0]), int(pos[-1])
    windows = [(p0, p0 + 500), (p0 + 200, p0 + 900), (p1 + 10, p1 + 100), (-50, -1), (p0 + 7, p0 + 6),
               (p0 - 100, p1 + 100), (int(pos[2000]), int(pos[2999]))]
    got, ref = _run(m, a, miss, pos, haps, windows=windows, max_missing=0.03)
    assert got["window_sites"][2] == got["window_sites"][3] == got["window_sites"][4] == 0
    region = (int(pos[300]), int(pos[2500]))
    _run(m, a, miss, pos, haps, size=80, step=60, region=region, max_missing=0.03)
    _run(m, a, miss, pos, haps, region=region, min_maf=0.05)
    pruned = _matrix_ld_prune(m, haps, 0.2, 50)["retained"]
    assert 0 < len(pruned) < 3000
    _run(m, a, miss, pos, haps, size=70, sites=pruned)
    _run(m, a, miss, pos, haps, windows=windows, sites=pruned)
    got = _matrix_hapfreq(m, haps, sites=[])
    assert int(got["info"].n_sites) == 0 and got["distinct"].tolist() == [1] and got["n_used"].tolist() == [100]


def test_hash_collision_is_split_exactly():
    """Keys A and B hash alike (B adds delta = mul^-1 to word 0 and subtracts delta * mul = 1 from word 1) but
    differ: one hash run, split into exact classes, and info.collisions counts it.  Site 0 of the matrix is an extra
    kept site, so the window starts one bit into a word (the funnel shift)."""
    from ferromic_b200.api import _matrix_hapfreq
    mul = 0x9E3779B97F4A7C15
    mask = (1 << 64) - 1
    delta = pow(mul, -1, 1 << 64)
    x0 = 0x0123456789ABCDEF
    words_a, words_b = (x0, 1), ((x0 + delta) & mask, 0)

    def horner(ws):
        h = 0
        for w in ws:
            h = (h * mul + w) & mask
        return h
    assert horner(words_a) == horner(words_b) and words_a != words_b

    def bits(ws):
        return [(ws[0] >> t) & 1 for t in range(64)] + [ws[1] & 1]
    keys = {"A": bits(words_a), "B": bits(words_b), "zero": [0] * 65, "one": [1] * 65}
    mult = {"A": 40, "B": 30, "zero": 2, "one": 1}  # the run of A and B spans three warps of the count kernel
    cols = [keys[k] for k in ("A", "B", "zero", "one") for _ in range(mult[k])]
    n = len(cols)
    key_rows = np.array(cols, np.uint8).T  # [65, n]
    lead = np.array([k == "one" for k in ("A", "B", "zero", "one") for _ in range(mult[k])], np.uint8)[None, :]
    a = np.concatenate([lead, key_rows])[:, :, None]
    miss = np.zeros_like(a, bool)
    pos = np.arange(66, dtype=np.int64) * 10
    for form in ("u8", "packed-dense"):
        m = _matrix(form, a, miss, pos)
        haps = _all_haps(n, 1)
        got, ref = _run(m, a, miss, pos, haps, windows=[(10, 650)])
        assert got["window_first"].tolist() == [1] and got["window_sites"].tolist() == [65]
        assert got["counts"].tolist() == [40, 30, 2, 1] and got["distinct"].tolist() == [4]
        assert int(got["info"].collisions) == 1
        full = _matrix_hapfreq(m, haps)  # the whole 66-site window: no run holds two keys
        assert int(full["info"].collisions) == 0 and full["distinct"].tolist() == [4]


def test_cohort_wider_than_shared_memory():
    """70,000 haplotypes: no per-haplotype state fits one CTA's shared memory."""
    a, miss, pos = _cohort(40, 35_000, 300, founders=20, mutation=0.001)
    m = _matrix("u8", a, miss, pos)
    haps = _all_haps(35_000, 2)
    got, ref = _run(m, a, miss, pos, haps, size=100, step=50)
    got, ref = _run(m, a, miss, pos, haps)
    assert ref["n"] == 70_000 and int(ref["top"][0][0]) > 500


def test_size_query_and_errors():
    import ferromic_b200 as fm
    from ferromic_b200 import _lib
    from ferromic_b200.api import _Matrix, _matrix_hapfreq
    a, miss, pos = _cohort(50, 20, 400, missing=0.002)
    m = _matrix("u8", a, miss, pos)
    haps = _all_haps(20, 2)
    idx = np.asarray([h[0] for h in haps], np.uint64)
    side = np.asarray([h[1] for h in haps], np.uint8)
    L = _lib.lib()

    def call(prm, out, windows=None, kept=None, cap=0, hs=(idx, side)):
        info = _lib.HapfreqInfo()
        p = lambda x: None if x is None else x.ctypes.data  # noqa: E731
        nw = 0 if windows is None else len(windows)
        st = L.fm_haplotype_frequencies(m.handle, p(hs[0]), p(hs[1]), len(hs[0]), C.byref(prm), p(windows), nw, None,
                                        p(kept), cap, C.byref(out), C.byref(info))
        return st, info, L.fm_last_error().decode()
    prm = _lib.HapfreqParams(50, 10, 0.0, 0.0)
    st, info, msg = call(prm, _lib.HapfreqOut())
    assert st == _lib.FM_ERR_INVALID_ARG and "capacity too small" in msg
    M = int(info.n_sites)
    assert info.n_haplotypes == 40 and M > 100 and info.n_windows == (M - 50) // 10 + 1
    kept = np.zeros(M, np.uint64)
    st, info, msg = call(prm, _lib.HapfreqOut(int(info.n_windows)), kept=kept, cap=M - 1)
    assert st == _lib.FM_ERR_INVALID_ARG and "site capacity" in msg
    nw = int(info.n_windows)
    h1 = np.zeros(nw)
    coff = np.zeros(nw + 1, np.uint64)
    out = _lib.HapfreqOut(nw, None, None, None, None, None, None, h1.ctypes.data, None, None, None, None,
                          coff.ctypes.data, None, 0)
    st, info, msg = call(prm, out, kept=kept, cap=M)
    assert st == _lib.FM_ERR_INVALID_ARG and "counts capacity" in msg and info.classes == coff[-1] > 0
    counts = np.zeros(int(info.classes), np.uint32)
    out.counts, out.counts_capacity = counts.ctypes.data, counts.size
    st, info, msg = call(prm, out, kept=kept, cap=M)
    assert st == _lib.FM_OK and np.all(h1 > 0) and counts.sum() > 0
    w = np.array([[0, 100], [50, 400]], np.int64)
    for p, what, win in ((_lib.HapfreqParams(5, 0, 0.0, 0.0), "exclusive", w),
                         (_lib.HapfreqParams(0, 0, 0.0, 0.0, 1, 0, 100), "exclusive", w),
                         (_lib.HapfreqParams(0, 3, 0.0, 0.0), "step", None),
                         (_lib.HapfreqParams(0, 0, 0.6, 0.0), "min_maf", None),
                         (_lib.HapfreqParams(0, 0, 0.0, 1.0), "max_missing", None)):
        st, _, msg = call(p, _lib.HapfreqOut(4), win)
        assert st == _lib.FM_ERR_INVALID_ARG and what in msg, msg
    st, _, msg = call(_lib.HapfreqParams(), _lib.HapfreqOut(4), hs=(np.array([99], np.uint64), np.array([0], np.uint8)))
    assert st == _lib.FM_ERR_INVALID_ARG and "empty" in msg
    info = _lib.HapfreqInfo()
    assert L.fm_haplotype_frequencies(m.handle, None, None, 0, None, None, 0, None, None, 0, None,
                                      C.byref(info)) == _lib.FM_ERR_INVALID_ARG
    for sites, what in (([5, 3, 9], "ascending"), ([3, 3, 9], "ascending"), ([3, 400], "beyond")):
        with pytest.raises(ValueError, match=what):
            _matrix_hapfreq(m, haps, sites=sites)
    with pytest.raises(ValueError, match="exclusive"):
        _matrix_hapfreq(m, haps, size=4, windows=[(0, 10)])
    with pytest.raises(ValueError, match="step needs size"):
        _matrix_hapfreq(m, haps, step=4)
    a3 = np.zeros((50, 10, 3), np.uint8)
    with pytest.raises(NotImplementedError, match="ploidy"):
        _matrix_hapfreq(_Matrix(a3, None, np.arange(50), ingest="u8"), [(0, 0), (1, 0)])
    with pytest.raises(NotImplementedError, match="streamed"):
        _matrix_hapfreq(_Matrix.ingest(a, miss, pos, [haps]), haps)
    unsorted = _matrix("u8", a, miss, pos[::-1].copy())
    with pytest.raises(NotImplementedError, match="sorted"):
        _matrix_hapfreq(unsorted, haps, windows=[(0, 10)])
    with pytest.raises(NotImplementedError, match="sorted"):
        _matrix_hapfreq(unsorted, haps, region=(0, 10))
    _run(m, a, miss, pos, haps, size=33)  # the library is still usable
    res = fm.haplotype_frequencies([(1, [[0, 1], [1, 1]]), (2, [[1, 0], [0, 0]])], counts=True)
    assert (res.n_used, res.distinct, res.sum_sq) == (4, 2, 10) and res.counts.tolist() == [3, 1]
    assert res.h1 == 10 / 16 and res.h12 == 1.0 and res.diversity == 0.5 and res.start == 1 and res.end == 2
    res = fm.haplotype_frequencies([(1, [[0, 1], [1, 1]]), (2, [[1, 0], [0, 0]])], windows=[(0, 1), (5, 9)])
    assert res.n_sites.tolist() == [1, 0] and res.start.tolist() == [1, -1] and res.distinct.tolist() == [2, 1]


def test_repeated_calls_and_threads_bit_identical():
    from ferromic_b200.api import _matrix_hapfreq
    a, miss, pos = _cohort(60, 200, 6000, missing=0.001)
    m = _matrix("u8", a, miss, pos)
    haps = _all_haps(200, 2)
    kw = dict(size=150, step=40, max_missing=0.01, counts=True)
    first = _matrix_hapfreq(m, haps, **kw)
    out, errs = [None] * 6, []

    def work(i):
        try:
            out[i] = _matrix_hapfreq(m, haps, **kw)
        except Exception as e:  # pragma: no cover - reported below
            errs.append(e)
    ts = [threading.Thread(target=work, args=(i,)) for i in range(6)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errs
    for r in out + [_matrix_hapfreq(m, haps, **kw)]:
        for k in ("h1", "h12", "h123", "h2_h1", "diversity"):
            assert _bits_equal(r[k], first[k]), k
        for k in ("distinct", "n_used", "sum_sq", "top_counts", "counts", "count_offsets"):
            assert np.array_equal(r[k], first[k]), k


def test_tie_to_per_site_pi():
    """size = 1 without missing data: each kept site has K = 2, and the haplotype diversity is the per-site pi of
    per_site_diversity_arrays, n / (n - 1) (1 - sum_sq / n^2), within 1e-12 relative."""
    import ferromic_b200 as fm
    from ferromic_b200.api import _Variants
    a, miss, pos = _cohort(70, 80, 1200)
    vs = _Variants(pos, a)
    haps = _all_haps(80, 2)
    res = fm.haplotype_frequencies(vs, haps, size=1)
    assert len(res.positions) > 500 and np.all(res.distinct == 2) and np.all(res.n_used == 160)
    ppos, pi, _ = fm.per_site_diversity_arrays(vs, haps, (int(pos[0]), int(pos[-1])))
    by_pos = dict(zip(ppos.tolist(), pi.tolist()))
    ref = np.array([by_pos[int(p) + 1] for p in res.start])
    np.testing.assert_allclose(res.diversity, ref, rtol=1e-12, atol=0)
