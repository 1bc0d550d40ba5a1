"""GPU haplotype LD pruning (fm_haplotype_ld_prune / haplotype_ld_prune) against the numpy restatement of
tests/ld_prune_reference.py: kept and retained rows, pairs, linked pairs, the retained count and the called-plane flag
exactly.  Every resident matrix form, ploidy 1 and 2, haplotype lists, the word and tile edges of the bit rows and of
the scan's 32-site blocks, thresholds 0 and 1, max_distance, regions, a long scan, threads, the size query, the
argument errors and the 8 GiB limit.  Also the site list of haplotype PCA and LD."""
import ctypes as C
import threading

import numpy as np
import pytest

from tests import ld_prune_reference as lp
from tests import ld_reference as lr
from tests import pca_reference as pr
from tests.test_gpu_pca import _compare as _compare_pca
from tests.test_gpu_pca import _matrix
from tests.test_ld_prune_reference import linked_cohort

pytestmark = pytest.mark.gpu


def _all_haps(S, P):
    return [(s, h) for s in range(S) for h in range(P)]


def _cohort(seed, S, V, ploidy=2, missing=0.0, flip=0.08):
    """Linked cohort as (alleles u8 [V, S, ploidy], missing bool, positions)."""
    x, called, pos = linked_cohort(seed, S * ploidy, V, missing, flip)
    return x.reshape(V, S, ploidy), ~called.reshape(V, S, ploidy), pos


def _run(m, a, miss, pos, haps, window, thr, region=None, max_distance=None, sites=None, **kw):
    from ferromic_b200.api import _matrix_ld_prune
    got = _matrix_ld_prune(m, haps, thr, window, max_distance, region, sites=sites, **kw)
    V, S, P = a.shape
    site_range = None
    if region is not None:
        site_range = (int(np.searchsorted(pos, region[0], "left")), int(np.searchsorted(pos, region[1], "right")))
    raw, called = a.reshape(V, -1), ~miss.reshape(V, -1)
    rows = pr.rows_from_arrays(raw, called)
    if sites is not None:
        rows = lp.subset_rows(rows, sites)
    off = lr.offsets(haps, S, P)
    ref = lp.ld_prune(rows, V, off, window, pos, thr, max_distance, site_range=site_range, **kw)
    info = got["info"]
    assert got["offsets"].tolist() == off.tolist()
    assert got["kept"].tolist() == ref["kept"].tolist()
    assert got["retained"].tolist() == ref["retained"].tolist()
    assert int(info.n_sites) == ref["M"] and int(info.n_haplotypes) == len(off)
    assert int(info.pairs) == ref["pairs"] and int(info.linked_pairs) == ref["linked_pairs"]
    assert int(info.n_retained) == len(ref["retained"])
    if ref["M"]:
        assert int(info.called_plane) == int(not called[ref["kept"]][:, off].all())
    return got, ref


@pytest.mark.parametrize("form", ["u8", "inband", "nomiss", "packed-dense", "packed-sparse", "lut"])
def test_matrix_forms(form):
    a, miss, pos = _cohort(41, 80, 900, missing=0.0 if form == "nomiss" else 0.01)
    if form == "lut":  # values above 15 go through the rank LUT; the filters and planes must see the raw values
        a[::7, :3, 0] = 254
        a[5::11] *= 17
    m = _matrix(form, a, miss, pos)
    got, ref = _run(m, a, miss, pos, _all_haps(80, 2), 70, 0.2, (int(pos[20]), int(pos[880])), max_missing=0.05,
                    min_maf=0.01)
    assert 500 < ref["M"] <= 861 and 0 < ref["linked_pairs"] and len(ref["retained"]) < ref["M"]
    assert int(got["info"].called_plane) == (0 if form == "nomiss" else 1)


@pytest.mark.parametrize("ploidy", [1, 2])
def test_ploidy_and_haplotype_lists(ploidy):
    a, miss, pos = _cohort(42 + ploidy, 100, 500, ploidy=ploidy, missing=0.01)
    for form in ("u8", "packed-dense"):
        m = _matrix(form, a, miss, pos)
        _run(m, a, miss, pos, _all_haps(100, 2), 100, 0.2, max_missing=0.05)
    m = _matrix("u8", a, miss, pos)
    for haps in ([(s, h) for s in (5, 9, 17, 40, 41, 77, 90) for h in (1, 0)],
                 [(s, h) for s in range(0, 100, 2) for h in (0, 1)] * 2 + [(3, 1)],
                 [(s, h) for s in range(60, 130) for h in (0, 1)]):
        _run(m, a, miss, pos, haps, 65, 0.2, max_missing=0.2)


@pytest.mark.parametrize("M", [1, 2, 63, 64, 65, 1000])
def test_sites_windows_thresholds(M):
    """Word and tile edges of the bit rows (window 31 / 32 / 33, 63 / 64 / 65) and of the scan's 32-site blocks."""
    a, miss, pos = _cohort(600 + M, 24, M, missing=0.02)
    m = _matrix("packed-dense", a, miss, pos)
    for window in sorted({1, 31, 32, 33, 63, 64, 65, 100, 1000, M - 1, M + 5} - {0}):
        for thr in (0.0, 0.2, 0.999, 1.0):
            got, ref = _run(m, a, miss, pos, _all_haps(24, 2), window, thr, max_missing=0.5)
            assert ref["M"] == M
    a0, miss0, pos0 = _cohort(700 + M, 24, M)  # no missing cell: the one-plane kernel
    got, _ = _run(_matrix("u8", a0, miss0, pos0), a0, miss0, pos0, _all_haps(24, 2), 65, 0.2)
    assert int(got["info"].called_plane) == 0


def test_max_distance_and_region():
    a, miss, pos = _cohort(44, 40, 1500, missing=0.01)
    pos = pos.copy()
    pos[100:110] = pos[100]          # duplicate positions
    pos[700:] += 10_000              # a gap no pair crosses at the limits below
    pos = np.maximum.accumulate(pos)
    m = _matrix("u8", a, miss, pos)
    for limit in (0, 25, 200, 5000):
        got, ref = _run(m, a, miss, pos, _all_haps(40, 2), 150, 0.2, max_distance=limit, max_missing=0.5)
        assert ref["pairs"] < ref["M"] * 150
    _run(m, a, miss, pos, _all_haps(40, 2), 80, 0.3, (int(pos[33]), int(pos[1222])), max_distance=400,
         max_missing=0.5)


def test_long_scan():
    """10^5 kept sites at window 2000: the scan crosses 3125 blocks with 63-word rows."""
    a, miss, pos = _cohort(45, 32, 100_000, missing=0.005, flip=0.15)
    m = _matrix("u8", a, miss, pos)
    got, ref = _run(m, a, miss, pos, _all_haps(32, 2), 2000, 0.2, max_missing=0.5)
    assert ref["M"] == 100_000 and 0.05 < len(ref["retained"]) / ref["M"] < 0.95


def test_pairs_equal_haplotype_ld():
    from ferromic_b200.api import _matrix_ld, _matrix_ld_prune
    a, miss, pos = _cohort(46, 30, 800, missing=0.01)
    m = _matrix("u8", a, miss, pos)
    haps = _all_haps(30, 2)
    for window, md in ((50, None), (300, 2000), (900, None)):
        ld = _matrix_ld(m, haps, window, md, max_missing=0.5)["info"]
        pr_ = _matrix_ld_prune(m, haps, 0.2, window, md, max_missing=0.5)["info"]
        assert int(pr_.pairs) == int(ld.pairs) and int(pr_.n_sites) == int(ld.n_sites)
        assert int(pr_.called_plane) == int(ld.called_plane)


def test_threads():
    from ferromic_b200.api import _matrix_ld_prune
    a, miss, pos = _cohort(47, 30, 20_000, missing=0.01)
    m = _matrix("u8", a, miss, pos)
    haps = _all_haps(30, 2)
    first = _matrix_ld_prune(m, haps, 0.2, 300, max_missing=0.5)
    out, errs = [None] * 4, []

    def work(i):
        try:
            out[i] = _matrix_ld_prune(m, haps, 0.2, 300, max_missing=0.5)
        except Exception as e:  # pragma: no cover - reported below
            errs.append(e)
    ts = [threading.Thread(target=work, args=(i,)) for i in range(4)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errs
    for r in out:
        assert np.array_equal(r["retained"], first["retained"])
        assert int(r["info"].linked_pairs) == int(first["info"].linked_pairs)


def _raw_call(m, haps, prm, thr=0.2, kept=None, ret=None, cap=0):
    from ferromic_b200 import _lib
    idx = np.asarray([h[0] for h in haps], np.uint64)
    side = np.asarray([h[1] for h in haps], np.uint8)
    info = _lib.LdPruneInfo()
    p = lambda x: None if x is None else x.ctypes.data  # noqa: E731
    st = _lib.lib().fm_haplotype_ld_prune(m.handle, p(idx), p(side), len(haps), C.byref(prm), thr, None, p(kept),
                                          p(ret), cap, C.byref(info))
    return st, info, _lib.lib().fm_last_error().decode()


def test_size_query_and_errors():
    import ferromic_b200 as fm
    from ferromic_b200 import _lib
    from ferromic_b200.api import _Matrix, _matrix_ld_prune
    a, miss, pos = _cohort(48, 40, 300, missing=0.01)
    m = _matrix("u8", a, miss, pos)
    haps = _all_haps(40, 2)
    prm = _lib.LdParams(20, -1, 0.0, 0.5, 0, 0, 0)
    st, info, msg = _raw_call(m, haps, prm)  # size query: no capacity, retained NULL
    assert st == _lib.FM_ERR_INVALID_ARG and "capacity too small" in msg
    assert info.n_sites == 300 and info.n_haplotypes == 80 and info.pairs == sum(min(20, 299 - i) for i in range(300))
    assert info.called_plane == 1 and info.band_launches == 0
    ret = np.zeros(300, np.uint64)
    st, info, msg = _raw_call(m, haps, prm, ret=ret, cap=299)
    assert st == _lib.FM_ERR_INVALID_ARG and "capacity too small" in msg
    st, info, msg = _raw_call(m, haps, prm, cap=300)
    assert st == _lib.FM_ERR_INVALID_ARG and "retained_sites" in msg
    kept = np.zeros(300, np.uint64)
    st, info, msg = _raw_call(m, haps, prm, kept=kept, ret=ret, cap=300)
    assert st == _lib.FM_OK and kept.tolist() == list(range(300)) and info.band_launches == 1
    ref = _matrix_ld_prune(m, haps, 0.2, 20, max_missing=0.5)
    assert ret[:info.n_retained].tolist() == ref["retained"].tolist()
    st, info, _ = _raw_call(m, [(0, 0)], prm)  # M == 0 is not an error
    assert st == _lib.FM_OK and info.n_sites == 0 and info.n_haplotypes == 1 and info.n_retained == 0
    for bad in (_lib.LdParams(0, -1, 0.0, 0.0, 0, 0, 0), _lib.LdParams(5, -1, 0.6, 0.0, 0, 0, 0),
                _lib.LdParams(5, -1, -0.1, 0.0, 0, 0, 0), _lib.LdParams(5, -1, 0.0, 1.0, 0, 0, 0),
                _lib.LdParams(5, -1, 0.0, -0.5, 0, 0, 0)):
        st, _, msg = _raw_call(m, haps, bad, kept=kept, ret=ret, cap=300)
        assert st == _lib.FM_ERR_INVALID_ARG, msg
    for thr in (-0.01, 1.0000001, float("nan"), float("inf")):
        st, _, msg = _raw_call(m, haps, prm, thr, kept=kept, ret=ret, cap=300)
        assert st == _lib.FM_ERR_INVALID_ARG and "r2_threshold" in msg
    with pytest.raises(ValueError, match="window"):
        _matrix_ld_prune(m, haps, 0.2, 0)
    a3 = np.zeros((50, 10, 3), np.uint8)
    a3[:, ::2] = 1
    with pytest.raises(NotImplementedError, match="ploidy"):
        _matrix_ld_prune(_Matrix(a3, None, np.arange(50), ingest="u8"), [(0, 0), (1, 0)], 0.2, 5)
    with pytest.raises(NotImplementedError, match="streamed"):
        _matrix_ld_prune(_Matrix.ingest(a, miss, pos, [haps]), haps, 0.2, 5)
    unsorted = _matrix("u8", a, miss, pos[::-1].copy())
    with pytest.raises(NotImplementedError, match="sorted"):
        _matrix_ld_prune(unsorted, haps, 0.2, 5, max_distance=10)
    for sites in ([5, 3, 9], [3, 3, 9], [3, 300]):
        with pytest.raises(ValueError, match="site_list"):
            _matrix_ld_prune(m, haps, 0.2, 5, sites=sites, max_missing=0.5)
    _run(m, a, miss, pos, haps, 7, 0.2, max_missing=0.5)  # the library is still usable
    res = fm.haplotype_ld_prune([(1, [[0, 1], [1, 1]]), (2, [[1, 0], [0, 0]])], window=1)
    assert res.n_kept == 2 and res.pairs == 1


def test_bit_row_limit():
    """A full-triangle window over 3 * 10^5 kept sites needs 3e5 * 9375 * 4 bytes > 8 GiB of bit rows: the call fails
    with both numbers in the message before any band launch."""
    from ferromic_b200 import _lib
    V, S = 300_000, 8
    rng = np.random.default_rng(49)
    a = (rng.random((V, S, 2)) < 0.5).astype(np.uint8)
    a[:, 0, 0], a[:, 1, 0] = 1, 0
    m = _matrix("nomiss", a, np.zeros_like(a, bool), np.arange(V, dtype=np.int64))
    prm = _lib.LdParams(V, -1, 0.0, 0.0, 0, 0, 0)
    ret = np.zeros(V, np.uint64)
    st, info, msg = _raw_call(m, _all_haps(S, 2), prm, ret=ret, cap=V)
    assert st == _lib.FM_ERR_UNSUPPORTED and "8 GiB" in msg and "M = 300000" in msg and f"window = {V}" in msg
    assert info.n_sites == V and info.band_launches == 0


# ------------------------------------------------------------------------------------ the site list of PCA and LD
def test_site_list_of_every_row_is_identity():
    from ferromic_b200.api import _matrix_ld, _matrix_pca
    a, miss, pos = _cohort(50, 60, 700, missing=0.01)
    m = _matrix("u8", a, miss, pos)
    haps = _all_haps(60, 2)
    every = np.arange(700)
    p0 = _matrix_pca(m, haps, 4, max_missing=0.1, loadings=True)
    p1 = _matrix_pca(m, haps, 4, max_missing=0.1, loadings=True, sites=every)
    for k in ("scores", "singular_values", "explained_variance_ratio", "loadings", "kept"):
        assert np.array_equal(p0[k].view(np.uint64), p1[k].view(np.uint64)), k
    l0 = _matrix_ld(m, haps, 40, max_missing=0.1, dprime=True)
    l1 = _matrix_ld(m, haps, 40, max_missing=0.1, dprime=True, sites=every)
    for k in ("r2", "dprime"):
        assert np.array_equal(l0[k].view(np.uint32), l1[k].view(np.uint32)), k
    assert np.array_equal(l0["kept"], l1["kept"])


def test_pca_and_ld_over_a_pruned_list():
    from ferromic_b200.api import _matrix_ld, _matrix_ld_prune, _matrix_pca
    a, miss, pos = _cohort(51, 60, 1200, missing=0.01)
    m = _matrix("packed-dense", a, miss, pos)
    haps = _all_haps(60, 2)
    V, S, P = a.shape
    raw, called = a.reshape(V, -1), ~miss.reshape(V, -1)
    off = pr.offsets(haps, S, P)
    sites = _matrix_ld_prune(m, haps, 0.2, 100, max_missing=0.1)["retained"]
    assert 50 < len(sites) < 1000
    sub = lp.subset_rows(pr.rows_from_arrays(raw, called), sites)
    got = _matrix_pca(m, haps, 5, max_missing=0.1, loadings=True, sites=sites)
    ref = pr.haplotype_pca(sub, V, off, 5, max_missing=0.1, loadings=True)
    assert ref["kept"].tolist() == sites.tolist()
    _compare_pca(got, off, ref, 5)
    region = (int(pos[100]), int(pos[1000]))
    got = _matrix_ld(m, haps, 30, 500, region, max_missing=0.1, dprime=True, sites=sites)
    site_range = (100, 1001)
    ref = lr.haplotype_ld(sub, V, off, 30, pos, 500, max_missing=0.1, site_range=site_range)
    assert got["kept"].tolist() == ref["kept"].tolist() and int(got["info"].pairs) == ref["pairs"]
    assert np.array_equal(got["r2"].view(np.uint32), ref["r2"].view(np.uint32))
    assert np.array_equal(got["dprime"].view(np.uint32), ref["dprime"].view(np.uint32))
    _run(m, a, miss, pos, haps, 50, 0.1, sites=sites[::2], max_missing=0.1)  # pruning over a list
    got = _matrix_ld(m, haps, 5, max_missing=0.1, sites=[])
    assert int(got["info"].n_sites) == 0


def test_bad_site_lists():
    from ferromic_b200.api import _matrix_ld, _matrix_pca
    a, miss, pos = _cohort(52, 20, 200, missing=0.01)
    m = _matrix("u8", a, miss, pos)
    haps = _all_haps(20, 2)
    for sites, what in (([5, 3, 9], "ascending"), ([3, 3, 9], "ascending"), ([3, 200], "beyond")):
        with pytest.raises(ValueError, match=what):
            _matrix_pca(m, haps, 2, max_missing=0.5, sites=sites)
        with pytest.raises(ValueError, match=what):
            _matrix_ld(m, haps, 5, max_missing=0.5, sites=sites)
    with pytest.raises(ValueError, match="negative"):
        _matrix_ld(m, haps, 5, sites=[-1, 3])


def test_public_prune_pca_chain():
    import ferromic_b200 as fm
    a, miss, pos = _cohort(53, 40, 600)
    variants = [(int(p), [list(map(int, g)) for g in row]) for p, row in zip(pos, a)]
    pruned = fm.haplotype_ld_prune(variants, r2_threshold=0.2, window=50, min_maf=0.05)
    V, S, P = a.shape
    off = lr.offsets(_all_haps(S, P), S, P)
    rows = pr.rows_from_arrays(a.reshape(V, -1), ~miss.reshape(V, -1))
    ref = lp.ld_prune(rows, V, off, 50, pos, 0.2, min_maf=0.05)
    assert pruned.sites.dtype == np.int64 and pruned.sites.tolist() == ref["retained"].tolist()
    assert pruned.positions.tolist() == pos[ref["retained"]].tolist()
    assert (pruned.n_kept, pruned.pairs, pruned.linked_pairs) == (ref["M"], ref["pairs"], ref["linked_pairs"])
    assert pruned.haplotypes == [(int(o) // 2, int(o) % 2) for o in off]
    res = fm.haplotype_pca(variants, n_components=3, sites=pruned.sites)
    assert res.positions.tolist() == pruned.positions.tolist()
    pref = pr.haplotype_pca(lp.subset_rows(rows, pruned.sites), V, off, 3)
    np.testing.assert_allclose(res.singular_values, pref["singular_values"], rtol=1e-9, atol=0)
    ld = fm.haplotype_ld(variants, window=5, sites=pruned.sites)
    assert ld.positions.tolist() == pruned.positions.tolist()
