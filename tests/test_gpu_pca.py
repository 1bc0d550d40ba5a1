"""GPU haplotype PCA (fm_haplotype_pca / haplotype_pca) against the numpy restatement of tests/pca_reference.py:
kept sites, M, T and the haplotype order exact; singular values and explained ratios within 1e-9 relative; scores
within 1e-7 of each component's largest score.  Every resident matrix form, ploidy 1 and 2, haplotype lists, the
edges of the tiling, regions, determinism, full width and the argument errors."""
import ctypes as C
import threading

import numpy as np
import pytest

from tests import pca_reference as pr

pytestmark = pytest.mark.gpu


def _matrix(form, a, miss, pos):
    from ferromic_b200.api import _Matrix
    if form == "inband":
        g = a.astype(np.int8)
        g[miss] = -1
        return _Matrix.from_int8(g, pos, max_allele=int(a.max()), ingest="u8")
    if form == "nomiss":
        return _Matrix(a, None, pos, ingest="u8")
    return _Matrix(a, miss, pos, ingest={"u8": "u8", "lut": "u8"}.get(form, form))


def _ref(a, miss, haps, k, site_range=None, **kw):
    V, S, P = a.shape
    raw, called = a.reshape(V, -1), ~miss.reshape(V, -1)
    off = pr.offsets(haps, S, P)
    return off, pr.haplotype_pca(pr.rows_from_arrays(raw, called), V, off, k, site_range=site_range, **kw)


def _compare(got, off, ref, k):
    assert got["offsets"].tolist() == off.tolist()
    assert got["kept"].tolist() == ref["kept"].tolist()
    assert int(got["info"].n_sites) == ref["M"] and int(got["info"].rank) == ref["l"]
    assert got["total_variance"] == ref["T"]
    np.testing.assert_allclose(got["singular_values"], ref["singular_values"], rtol=1e-9, atol=0)
    np.testing.assert_allclose(got["explained_variance_ratio"], ref["explained_variance_ratio"], rtol=1e-9, atol=0)
    scale = np.max(np.abs(ref["scores"]), axis=0)
    # the sign rule reads the entry of largest |score|; when two entries tie to rounding (two haplotypes with opposite
    # scores), summation order decides which one that is, so such a component is compared up to its sign
    top2 = -np.sort(-np.abs(ref["scores"]), axis=0)[:2] if ref["scores"].shape[0] > 1 else None
    tie = np.zeros(k, bool) if top2 is None else (top2[0] - top2[1] <= 1e-12 * top2[0])
    sign = np.where(tie & (np.sign(got["scores"][0]) != np.sign(ref["scores"][0])), -1.0, 1.0)
    assert np.all(np.abs(got["scores"] * sign - ref["scores"]) <= 1e-7 * scale)
    if ref["loadings"] is not None:
        lscale = np.max(np.abs(ref["loadings"]), axis=0)
        assert np.all(np.abs(got["loadings"] - ref["loadings"]) <= 1e-7 * lscale)


def _run(m, a, miss, pos, haps, k, region=None, **kw):
    from ferromic_b200.api import _matrix_pca
    got = _matrix_pca(m, haps, k, region, **kw)
    site_range = None
    if region is not None:
        site_range = (int(np.searchsorted(pos, region[0], "left")), int(np.searchsorted(pos, region[1], "right")))
    off, ref = _ref(a, miss, haps, k, site_range, **kw)
    _compare(got, off, ref, k)
    return got, ref


def _all_haps(S, P):
    return [(s, h) for s in range(S) for h in range(P)]


@pytest.mark.parametrize("form", ["u8", "inband", "nomiss", "packed-dense", "packed-sparse", "lut"])
def test_matrix_forms(form):
    a, miss, pos, _ = pr.cohort(11, 4, 40, 1100, missing=0.0 if form == "nomiss" else 0.01)
    if form == "lut":  # values above 15 go through the rank LUT; the filters must see the raw values
        a[::7, :3, 0] = 254       # an extra allele value: site dropped
        a[5::11] *= 17            # {0, 17}: no raw 1, although the ranks are {0, 1}
    m = _matrix(form, a, miss, pos)
    got, ref = _run(m, a, miss, pos, _all_haps(160, 2), 3, (int(pos[20]), int(pos[1050])), max_missing=0.05,
                    min_maf=0.01, loadings=True, seed=3)
    assert 600 < ref["M"] < 1031


def test_filter_boundaries():
    """The boundary sites of tests/test_pca_reference.py on the device: min_maf and max_missing * n met exactly, an
    extra allele value (also inside missing cells), the {0, 17} site of the rank LUT, a monomorphic site."""
    from tests.test_pca_reference import _one_site_cases
    cases = _one_site_cases()
    a = np.stack([c[0] for c in cases]).reshape(len(cases), 5, 2)
    miss = ~np.stack([c[1] for c in cases]).reshape(len(cases), 5, 2)
    pos = np.arange(len(cases), dtype=np.int64) * 3
    for form in ("u8", "inband"):
        got, ref = _run(_matrix(form, a, miss, pos), a, miss, pos, _all_haps(5, 2), 1, min_maf=0.2, max_missing=0.2)
        assert got["kept"].tolist() == [i for i, c in enumerate(cases) if c[2]]


def test_counts_match_group_summary():
    """On a biallelic matrix the kept sites and T follow from fm_group_summary's alt / called of the same list."""
    a, miss, pos, _ = pr.cohort(12, 3, 50, 900, missing=0.02)
    m = _matrix("u8", a, miss, pos)
    rng = np.random.default_rng(1)
    haps = [(int(s), int(h)) for s, h in zip(rng.integers(0, 150, 200), rng.integers(0, 2, 200))]
    from ferromic_b200.api import _matrix_pca
    got = _matrix_pca(m, haps, 2, max_missing=0.1, min_maf=0.05)
    summ = m.group(haps).summary(want_arrays=True)
    alt, called = summ["alt"].astype(np.int64), summ["called"].astype(np.int64)
    n = len(got["offsets"])
    keep = ((alt > 0) & (alt < called) & ((n - called) <= 0.1 * n) & (np.minimum(alt, called - alt) >= 0.05 * called))
    assert got["kept"].tolist() == np.flatnonzero(keep).tolist()
    assert got["total_variance"] == float(called[keep].sum())


@pytest.mark.parametrize("ploidy", [1, 2])
def test_ploidy(ploidy):
    a, miss, pos, _ = pr.cohort(13, 4, 70, 700, ploidy=ploidy, missing=0.01)
    for form in ("u8", "packed-dense"):
        m = _matrix(form, a, miss, pos)
        _run(m, a, miss, pos, _all_haps(280, 2), 3, max_missing=0.05)


def test_haplotype_lists():
    a, miss, pos, _ = pr.cohort(14, 4, 40, 800, missing=0.01)
    m = _matrix("u8", a, miss, pos)
    lists = {
        "duplicates": [(s, h) for s in range(0, 160, 2) for h in (0, 1)] * 2 + [(3, 1), (3, 1)],
        "out_of_range": [(s, h) for s in range(100, 190) for h in (0, 1)],
        "one_side": [(s, 1) for s in range(160)],
        "subset": [(s, h) for s in (5, 9, 17, 40, 41, 77, 90, 123, 150, 151, 152, 158) for h in (1, 0)],
    }
    for haps in lists.values():
        _run(m, a, miss, pos, haps, 2, max_missing=0.1)


def _polymorphic(n_haps_samples, V, seed, ploidy=2):
    """A cohort whose every site is polymorphic with no missing cell: M = V for min_maf = max_missing = 0."""
    a, miss, pos, _ = pr.cohort(seed, 4, (n_haps_samples + 3) // 4, V, ploidy=ploidy)
    a = a[:, :n_haps_samples].copy()
    miss = miss[:, :n_haps_samples].copy()
    a[:, 0, 0], a[:, -1, -1] = 1, 0
    return a, miss, pos


@pytest.mark.parametrize("n", [2, 63, 64, 65, 129])
def test_haplotype_tiling(n):
    a, miss, pos = _polymorphic(n, 700, 100 + n, ploidy=1)
    m = _matrix("u8", a, miss, pos)
    got, ref = _run(m, a, miss, pos, _all_haps(n, 1), 1 if n == 2 else 3)
    assert ref["M"] == 700


@pytest.mark.parametrize("M", [1, 255, 256, 257, 2100])
def test_site_tiling(M):
    a, miss, pos = _polymorphic(70, M, 200 + M)
    m = _matrix("packed-dense", a, miss, pos)
    got, ref = _run(m, a, miss, pos, _all_haps(70, 2), 1 if M == 1 else 4, oversampling=5)
    assert ref["M"] == M


@pytest.mark.parametrize("case", ["l64", "l_by_n", "l_by_m", "q0"])
def test_rank_edges(case):
    a, miss, pos = _polymorphic(20 if case == "l_by_n" else 120, 30 if case == "l_by_m" else 900, 300)
    m = _matrix("u8", a, miss, pos)
    P = 2
    kw = dict(l64=dict(k=10, oversampling=54), l_by_n=dict(k=5, oversampling=200), l_by_m=dict(k=5, oversampling=200),
              q0=dict(k=4, oversampling=6, power_iterations=0))[case]
    k = kw.pop("k")
    got, ref = _run(m, a, miss, pos, _all_haps(a.shape[1], P), k, **kw)
    assert ref["l"] == {"l64": 64, "l_by_n": 40, "l_by_m": 30, "q0": 10}[case]


def test_test_matrix_signs():
    """q = 0 and l = k: the result is fixed by G, so agreeing with the restatement checks the device's G (the first
    signs of seed 1 are pinned in tests/test_pca_reference.py); another seed must give another answer."""
    a, miss, pos, _ = pr.cohort(15, 6, 20, 500, missing=0.0)
    m = _matrix("u8", a, miss, pos)
    got, _ = _run(m, a, miss, pos, _all_haps(120, 2), 2, oversampling=0, power_iterations=0, seed=1)
    _, other = _ref(a, miss, _all_haps(120, 2), 2, oversampling=0, power_iterations=0, seed=2)
    assert np.max(np.abs(got["singular_values"] - other["singular_values"])) > 1e-6 * other["singular_values"][0]


def test_region_bounds():
    a, miss, pos, _ = pr.cohort(16, 4, 40, 1500, missing=0.02)
    m = _matrix("packed-sparse", a, miss, pos)
    for region in ((int(pos[37]), int(pos[700])), (int(pos[300]) + 1, int(pos[1299]) - 1)):
        _run(m, a, miss, pos, _all_haps(160, 2), 1, region, min_maf=0.1, max_missing=0.02)
    got, ref = _run(m, a, miss, pos, _all_haps(160, 2), 1, (0, int(pos[0])), max_missing=0.1)  # one site
    assert ref["M"] == 1


def test_determinism_and_threads():
    from ferromic_b200.api import _matrix_pca
    a, miss, pos, _ = pr.cohort(17, 5, 60, 3000, missing=0.01)
    m = _matrix("u8", a, miss, pos)
    haps = _all_haps(300, 2)
    first = _matrix_pca(m, haps, 4, max_missing=0.05, loadings=True)
    keys = ("scores", "singular_values", "explained_variance_ratio", "loadings")
    for _ in range(3):
        again = _matrix_pca(m, haps, 4, max_missing=0.05, loadings=True)
        for key in keys:
            assert np.array_equal(again[key], first[key])
    out, errs = [None] * 4, []

    def work(i):
        try:
            out[i] = _matrix_pca(m, haps, 4, max_missing=0.05, loadings=True)
        except Exception as e:  # pragma: no cover - reported below
            errs.append(e)
    ts = [threading.Thread(target=work, args=(i,)) for i in range(4)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errs
    for r in out:
        for key in keys:
            assert np.array_equal(r[key], first[key])


def test_public_api():
    import ferromic_b200 as fm
    a, miss, pos, _ = pr.cohort(18, 4, 30, 400, missing=0.0)
    variants = [(int(p), [list(map(int, g)) for g in row]) for p, row in zip(pos, a)]
    res = fm.haplotype_pca(variants, n_components=3, loadings=True)
    off, ref = _ref(a, miss, _all_haps(120, 2), 3, loadings=True)
    assert res.haplotypes == [(int(o) // 2, int(o) % 2) for o in off]
    assert res.positions.tolist() == pos[ref["kept"]].tolist()
    np.testing.assert_allclose(res.singular_values, ref["singular_values"], rtol=1e-9)
    assert res.loadings.shape == (ref["M"], 3) and res.total_variance == ref["T"]
    with pytest.raises(ValueError, match=r"n = 240 haplotypes, M = \d+ kept sites"):
        fm.haplotype_pca(variants, n_components=0)


def test_full_width_synth():
    """5008 haplotypes x 2e5 sites generated on the device (fm_synth_fill, 26 populations, 1 % missing)."""
    import torch
    from ferromic_b200 import _lib
    from ferromic_b200.api import _matrix_pca
    L = _lib.lib()
    V, S, seed = 200_000, 2504, 9
    pops = (np.arange(S) % 26).astype(np.uint16)
    total = V * S * 2
    d_data = torch.empty(total, dtype=torch.uint8, device="cuda:0")
    d_miss = torch.empty((total + 63) // 64, dtype=torch.int64, device="cuda:0")
    _lib.check(L.fm_set_device(0))
    _lib.check(L.fm_synth_fill(d_data.data_ptr(), d_miss.data_ptr(), V, S, 2, 0, seed, pops.ctypes.data, 0.05, 0.01))
    pos = np.arange(V, dtype=np.int64) * 5
    h = C.c_void_p()
    _lib.check(L.fm_matrix_create_device(d_data.data_ptr(), d_miss.data_ptr(), V, S, 2, 1, pos.ctypes.data, C.byref(h)))
    try:
        m = type("M", (), {"handle": h, "V": V, "P": 2})
        haps = _all_haps(S, 2)
        got = _matrix_pca(m, haps, 10, max_missing=0.02, min_maf=0.01, power_iterations=0)
        raw = d_data.view(V, S * 2).cpu().numpy()
        bits = np.unpackbits(d_miss.cpu().numpy().view(np.uint8), bitorder="little")[:total].reshape(V, S * 2)
        off = pr.offsets(haps, S, 2)
        ref = pr.haplotype_pca(lambda x, y: (raw[x:y], bits[x:y] == 0), V, off, 10, max_missing=0.02, min_maf=0.01,
                               power_iterations=0, chunk=8192)
        _compare(got, off, ref, 10)
    finally:
        L.fm_matrix_release(h)


def test_errors():
    import ferromic_b200 as fm
    from ferromic_b200 import _lib
    from ferromic_b200.api import _Matrix, _matrix_pca
    a, miss, pos = _polymorphic(40, 300, 400)
    m = _matrix("u8", a, miss, pos)
    haps = _all_haps(40, 2)
    for kw in (dict(n_components=0), dict(n_components=81), dict(n_components=10, oversampling=60),
               dict(n_components=2, min_maf=0.6), dict(n_components=2, min_maf=-0.1),
               dict(n_components=2, max_missing=1.0), dict(n_components=2, max_missing=-0.5)):
        k = kw.pop("n_components")
        with pytest.raises(ValueError, match=r"n = 80 haplotypes, M = \d+ kept sites"):
            _matrix_pca(m, haps, k, **kw)
    st = _lib.lib().fm_haplotype_pca(m.handle, None, None, 0, C.byref(_lib.PcaParams(1, 0, 0, 0.0, 0.0, 0, 0, 0, 0)),
                                     None, None, None, None, None, None, 0, C.byref(_lib.PcaInfo()))
    assert st == _lib.FM_ERR_INVALID_ARG and "n = 0 haplotypes" in _lib.lib().fm_last_error().decode()
    # too small a site capacity: counts are written so that the caller can retry
    idx = np.asarray([h[0] for h in haps], np.uint64)
    side = np.asarray([h[1] for h in haps], np.uint8)
    info = _lib.PcaInfo()
    kept = np.zeros(10, np.uint64)
    buf = np.zeros(80 * 2)
    st = _lib.lib().fm_haplotype_pca(m.handle, idx.ctypes.data, side.ctypes.data, len(haps),
                                     C.byref(_lib.PcaParams(2, 2, 1, 0.0, 0.0, 0, 0, 0, 0)), None, buf.ctypes.data,
                                     buf.ctypes.data, buf.ctypes.data, kept.ctypes.data, None, 10, C.byref(info))
    assert st == _lib.FM_ERR_INVALID_ARG and info.n_sites == 300 and info.n_haplotypes == 80
    a3 = np.zeros((50, 10, 3), np.uint8)
    a3[:, ::2] = 1
    with pytest.raises(NotImplementedError, match="ploidy"):
        _matrix_pca(_Matrix(a3, None, np.arange(50), ingest="u8"), [(0, 0), (1, 0)], 1)
    streamed = _Matrix.ingest(a, miss, pos, [haps])
    with pytest.raises(NotImplementedError, match="streamed"):
        _matrix_pca(streamed, haps, 2)
    _run(m, a, miss, pos, haps, 2)  # the library is still usable
    assert fm.haplotype_pca([(1, [[0, 1], [1, 1]]), (2, [[1, 0], [0, 0]])], n_components=1).scores.shape == (4, 1)
