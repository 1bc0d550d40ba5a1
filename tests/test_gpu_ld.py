"""GPU haplotype LD (fm_haplotype_ld / haplotype_ld) against the numpy restatement of tests/ld_reference.py: r^2 and
D' bit for bit (as uint32), kept sites, haplotype offsets and pair counts exactly.  Every resident matrix form,
ploidy 1 and 2, haplotype lists, the edges of the tiling in n, M and window, max_distance, regions and filters, the
NaN rules, several output slabs, the size-query protocol, the argument errors, threads and the public surface."""
import ctypes as C
import threading

import numpy as np
import pytest

from tests import ld_reference as lr
from tests import pca_reference as pr
from tests.test_gpu_pca import _matrix

pytestmark = pytest.mark.gpu


def _all_haps(S, P):
    return [(s, h) for s in range(S) for h in range(P)]


def _run(m, a, miss, pos, haps, window, region=None, max_distance=None, dprime=True, **kw):
    from ferromic_b200.api import _matrix_ld
    got = _matrix_ld(m, haps, window, max_distance, region, dprime=dprime, **kw)
    V, S, P = a.shape
    site_range = None
    if region is not None:
        site_range = (int(np.searchsorted(pos, region[0], "left")), int(np.searchsorted(pos, region[1], "right")))
    raw, called = a.reshape(V, -1), ~miss.reshape(V, -1)
    off = lr.offsets(haps, S, P)
    ref = lr.haplotype_ld(pr.rows_from_arrays(raw, called), V, off, window, pos, max_distance, site_range=site_range,
                          **kw)
    info = got["info"]
    assert got["offsets"].tolist() == off.tolist()
    assert got["kept"].tolist() == ref["kept"].tolist()
    assert int(info.n_sites) == ref["M"] and int(info.n_haplotypes) == len(off) and int(info.pairs) == ref["pairs"]
    assert got["r2"].shape == (ref["M"], window)
    assert np.array_equal(got["r2"].view(np.uint32), ref["r2"].view(np.uint32))
    if dprime:
        assert np.array_equal(got["dprime"].view(np.uint32), ref["dprime"].view(np.uint32))
    else:
        assert got["dprime"] is None
    if ref["M"]:
        incomplete = not called[ref["kept"]][:, off].all()
        assert int(info.called_plane) == int(incomplete)
    return got, ref


def _polymorphic(n_samples, V, seed, ploidy=2, missing=0.0):
    """Every site polymorphic (cell 0 alt, the last cell reference, both called): M = V at max_missing 0.5."""
    rng = np.random.default_rng(seed)
    a = (rng.random((V, n_samples, ploidy)) < rng.uniform(0.05, 0.95, size=V)[:, None, None]).astype(np.uint8)
    miss = rng.random((V, n_samples, ploidy)) < missing
    a[:, 0, 0], a[:, -1, -1] = 1, 0
    miss[:, 0, 0] = miss[:, -1, -1] = False
    a[miss] = 0
    return a, miss, np.cumsum(rng.integers(1, 30, size=V)).astype(np.int64)


@pytest.mark.parametrize("form", ["u8", "inband", "nomiss", "packed-dense", "packed-sparse", "lut"])
def test_matrix_forms(form):
    a, miss, pos, _ = pr.cohort(31, 4, 40, 900, missing=0.0 if form == "nomiss" else 0.01)
    if form == "lut":  # values above 15 go through the rank LUT; the filters and planes must see the raw values
        a[::7, :3, 0] = 254
        a[5::11] *= 17
    m = _matrix(form, a, miss, pos)
    got, ref = _run(m, a, miss, pos, _all_haps(160, 2), 70, (int(pos[20]), int(pos[880])), max_missing=0.05,
                    min_maf=0.01)
    assert 500 < ref["M"] <= 861 and (form != "lut" or ref["M"] < 861)
    assert int(got["info"].called_plane) == (0 if form == "nomiss" else 1)


@pytest.mark.parametrize("ploidy", [1, 2])
def test_ploidy(ploidy):
    a, miss, pos, _ = pr.cohort(32, 4, 50, 500, ploidy=ploidy, missing=0.01)
    for form in ("u8", "packed-dense"):
        _run(_matrix(form, a, miss, pos), a, miss, pos, _all_haps(200, 2), 100, max_missing=0.05)


def test_haplotype_lists():
    a, miss, pos, _ = pr.cohort(33, 4, 40, 600, missing=0.01)
    m = _matrix("u8", a, miss, pos)
    lists = {
        "subset": [(s, h) for s in (5, 9, 17, 40, 41, 77, 90, 123, 150, 151, 152, 158) for h in (1, 0)],
        "duplicates": [(s, h) for s in range(0, 160, 2) for h in (0, 1)] * 2 + [(3, 1), (3, 1)],
        "out_of_range": [(s, h) for s in range(100, 190) for h in (0, 1)],
    }
    for haps in lists.values():
        _run(m, a, miss, pos, haps, 65, max_missing=0.1)


@pytest.mark.parametrize("n", [1, 31, 32, 33, 255, 256, 257, 600])
def test_haplotype_counts(n):
    """Tail words of the last 32-haplotype word and of the last 8-word chunk; n = 1 keeps no site."""
    for missing in (0.0, 0.02):
        a, miss, pos = _polymorphic(n, 300, 500 + n, ploidy=1, missing=missing)
        got, ref = _run(_matrix("u8", a, miss, pos), a, miss, pos, _all_haps(n, 1), 70, max_missing=0.5)
        assert ref["M"] == (0 if n == 1 else 300)


@pytest.mark.parametrize("M", [1, 63, 64, 65, 1000])
def test_site_and_window_tiling(M):
    a, miss, pos = _polymorphic(40, M, 600 + M, missing=0.02)
    m = _matrix("packed-dense", a, miss, pos)
    for window in sorted({1, 63, 64, 65, 200, M - 1, M + 5} - {0}):
        got, ref = _run(m, a, miss, pos, _all_haps(40, 2), window, max_missing=0.5)
        assert ref["M"] == M
    a0, miss0, pos0 = _polymorphic(40, M, 700 + M)  # no missing cell: the one-plane kernel
    got, _ = _run(_matrix("u8", a0, miss0, pos0), a0, miss0, pos0, _all_haps(40, 2), 65)
    assert int(got["info"].called_plane) == 0


def test_max_distance():
    a, miss, pos = _polymorphic(50, 700, 800, missing=0.01)
    pos = pos.copy()
    pos[100:110] = pos[100]          # duplicate positions
    pos[300:] += 10_000              # a gap no pair crosses at the limits below
    pos[201] = pos[200] + 25         # a pair at exactly the limit
    pos = np.maximum.accumulate(pos)
    m = _matrix("u8", a, miss, pos)
    for limit in (0, 25, 200, 5000):
        got, ref = _run(m, a, miss, pos, _all_haps(50, 2), 150, max_distance=limit, max_missing=0.5)
        assert ref["pairs"] < ref["M"] * 150
    got, _ = _run(m, a, miss, pos, _all_haps(50, 2), 150, max_distance=25, max_missing=0.5)
    assert not np.isnan(got["r2"][200, 0])


def test_region_and_filters():
    """The boundary sites of tests/test_pca_reference.py (min_maf and max_missing met exactly, extra allele values,
    the {0, 17} site of the rank LUT, a monomorphic site) between polymorphic sites, inside a region."""
    from tests.test_pca_reference import _one_site_cases
    cases = _one_site_cases()
    rows = []
    rng = np.random.default_rng(7)
    for c in cases:
        fill = (rng.random(10) < 0.5).astype(np.uint8)
        fill[0], fill[1] = 1, 0
        rows += [(fill, np.ones(10, bool)), (c[0], c[1])]
    a = np.stack([r[0] for r in rows]).reshape(len(rows), 5, 2)
    miss = ~np.stack([r[1] for r in rows]).reshape(len(rows), 5, 2)
    pos = np.arange(len(rows), dtype=np.int64) * 3
    for form in ("u8", "inband"):
        m = _matrix(form, a, miss, pos)
        got, ref = _run(m, a, miss, pos, _all_haps(5, 2), 4, min_maf=0.2, max_missing=0.2)
        assert [int(k) for k in got["kept"] if k % 2] == [2 * i + 1 for i, c in enumerate(cases) if c[2]]
        _run(m, a, miss, pos, _all_haps(5, 2), 4, (int(pos[3]), int(pos[14])), min_maf=0.2, max_missing=0.2)


def test_jointly_called_nan_rules():
    """Site 0 and 1 are never called together (c = 0); site 2 is polymorphic but monomorphic among the haplotypes
    called at both 2 and 3."""
    a = np.zeros((4, 8, 1), np.uint8)
    miss = np.zeros((4, 8, 1), bool)
    a[0, :4, 0] = [1, 0, 1, 0]
    miss[0, 4:, 0] = True
    a[1, 4:, 0] = [1, 0, 1, 0]
    miss[1, :4, 0] = True
    a[2, :, 0] = [1, 1, 1, 1, 1, 1, 0, 0]
    miss[3, 6:, 0] = True
    a[3, :6, 0] = [1, 0, 1, 0, 1, 0]
    pos = np.arange(4, dtype=np.int64)
    got, ref = _run(_matrix("u8", a, miss, pos), a, miss, pos, _all_haps(8, 1), 3, max_missing=0.5)
    assert ref["M"] == 4 and np.isnan(got["r2"][0, 0]) and np.isnan(got["r2"][2, 0]) and np.isnan(got["dprime"][2, 0])
    assert not np.isnan(got["r2"][0, 2])


def test_many_slabs():
    """50k kept sites x window 1000: 200 MB of r^2 and as much D', in slabs of at most 64 MB."""
    a, miss, pos = _polymorphic(32, 50_000, 900, missing=0.01)
    got, _ = _run(_matrix("u8", a, miss, pos), a, miss, pos, _all_haps(32, 2), 1000, max_missing=0.5)
    assert int(got["info"].slabs) >= 6 and int(got["info"].band_launches) == int(got["info"].slabs)
    got, _ = _run(_matrix("packed-dense", a, miss, pos), a, miss, pos, _all_haps(32, 2), 1000, max_missing=0.5,
                  dprime=False)
    assert int(got["info"].slabs) >= 3


def _raw_call(m, haps, prm, kept=None, cap=0, r2=None, dp=None, pair_cap=0):
    from ferromic_b200 import _lib
    idx = np.asarray([h[0] for h in haps], np.uint64)
    side = np.asarray([h[1] for h in haps], np.uint8)
    info = _lib.LdInfo()
    p = lambda x: None if x is None else x.ctypes.data  # noqa: E731
    st = _lib.lib().fm_haplotype_ld(m.handle, p(idx), p(side), len(haps), C.byref(prm), None, p(kept), cap, p(r2),
                                    p(dp), pair_cap, C.byref(info))
    return st, info, _lib.lib().fm_last_error().decode()


def test_capacity_retry_and_errors():
    import ferromic_b200 as fm
    from ferromic_b200 import _lib
    from ferromic_b200.api import _Matrix, _matrix_ld
    a, miss, pos = _polymorphic(40, 300, 1000, missing=0.01)
    m = _matrix("u8", a, miss, pos)
    haps = _all_haps(40, 2)
    prm = _lib.LdParams(20, -1, 0.0, 0.5, 0, 0, 0)
    # size query: r2 NULL, no capacity -> the counts come back with FM_ERR_INVALID_ARG
    st, info, msg = _raw_call(m, haps, prm)
    assert st == _lib.FM_ERR_INVALID_ARG and "capacity too small" in msg
    assert info.n_sites == 300 and info.n_haplotypes == 80 and info.pairs == sum(min(20, 299 - i) for i in range(300))
    kept = np.zeros(299, np.uint64)
    r2 = np.zeros(300 * 20, np.float32)
    st, info, msg = _raw_call(m, haps, prm, kept, 299, r2, None, r2.size)
    assert st == _lib.FM_ERR_INVALID_ARG and "site capacity" in msg and info.n_sites == 300
    st, info, msg = _raw_call(m, haps, prm, None, 0, r2, None, r2.size - 1)
    assert st == _lib.FM_ERR_INVALID_ARG and "pair capacity" in msg
    kept = np.zeros(300, np.uint64)
    st, info, msg = _raw_call(m, haps, prm, kept, 300, r2, None, r2.size)
    assert st == _lib.FM_OK and kept.tolist() == list(range(300))
    ref = _matrix_ld(m, haps, 20, max_missing=0.5)
    assert np.array_equal(ref["r2"].reshape(-1).view(np.uint32), r2.view(np.uint32))
    # M == 0 is not an error
    st, info, _ = _raw_call(m, [(0, 0)], prm)
    assert st == _lib.FM_OK and info.n_sites == 0 and info.n_haplotypes == 1
    # argument errors
    for bad in (_lib.LdParams(0, -1, 0.0, 0.0, 0, 0, 0), _lib.LdParams(5, -1, 0.6, 0.0, 0, 0, 0),
                _lib.LdParams(5, -1, -0.1, 0.0, 0, 0, 0), _lib.LdParams(5, -1, 0.0, 1.0, 0, 0, 0),
                _lib.LdParams(5, -1, 0.0, -0.5, 0, 0, 0)):
        st, _, msg = _raw_call(m, haps, bad, kept, 300, r2, None, r2.size)
        assert st == _lib.FM_ERR_INVALID_ARG, msg
    with pytest.raises(ValueError, match="window"):
        _matrix_ld(m, haps, 0)
    a3 = np.zeros((50, 10, 3), np.uint8)
    a3[:, ::2] = 1
    with pytest.raises(NotImplementedError, match="ploidy"):
        _matrix_ld(_Matrix(a3, None, np.arange(50), ingest="u8"), [(0, 0), (1, 0)], 5)
    streamed = _Matrix.ingest(a, miss, pos, [haps])
    with pytest.raises(NotImplementedError, match="streamed"):
        _matrix_ld(streamed, haps, 5)
    unsorted = _matrix("u8", a, miss, pos[::-1].copy())
    with pytest.raises(NotImplementedError, match="sorted"):
        _matrix_ld(unsorted, haps, 5, max_distance=10)
    with pytest.raises(NotImplementedError, match="sorted"):
        _matrix_ld(unsorted, haps, 5, region=(0, 100))
    _matrix_ld(unsorted, haps, 5, max_missing=0.5)  # neither: positions are not read
    _run(m, a, miss, pos, haps, 7, max_missing=0.5)  # the library is still usable
    assert fm.haplotype_ld([(1, [[0, 1], [1, 1]]), (2, [[1, 0], [0, 0]])], window=1).r2.shape == (2, 1)


def test_threads():
    from ferromic_b200.api import _matrix_ld
    a, miss, pos = _polymorphic(60, 5000, 1100, missing=0.01)
    m = _matrix("u8", a, miss, pos)
    haps = _all_haps(60, 2)
    first = _matrix_ld(m, haps, 300, max_missing=0.5, dprime=True)
    out, errs = [None] * 4, []

    def work(i):
        try:
            out[i] = _matrix_ld(m, haps, 300, max_missing=0.5, dprime=True)
        except Exception as e:  # pragma: no cover - reported below
            errs.append(e)
    ts = [threading.Thread(target=work, args=(i,)) for i in range(4)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errs
    for r in out:
        assert np.array_equal(r["r2"].view(np.uint32), first["r2"].view(np.uint32))
        assert np.array_equal(r["dprime"].view(np.uint32), first["dprime"].view(np.uint32))


def test_public_api():
    import ferromic_b200 as fm
    a, miss, pos, _ = pr.cohort(34, 4, 30, 400, missing=0.0)
    variants = [(int(p), [list(map(int, g)) for g in row]) for p, row in zip(pos, a)]
    res = fm.haplotype_ld(variants, window=50, max_distance=200, dprime=True, min_maf=0.05)
    V, S, P = a.shape
    off = lr.offsets(_all_haps(S, P), S, P)
    ref = lr.haplotype_ld(pr.rows_from_arrays(a.reshape(V, -1), ~miss.reshape(V, -1)), V, off, 50, pos, 200,
                          min_maf=0.05)
    assert res.haplotypes == [(int(o) // 2, int(o) % 2) for o in off]
    assert res.positions.tolist() == pos[ref["kept"]].tolist()
    assert np.array_equal(res.r2.view(np.uint32), ref["r2"].view(np.uint32))
    assert np.array_equal(res.dprime.view(np.uint32), ref["dprime"].view(np.uint32))
    sub = fm.haplotype_ld(variants, haplotypes=[(0, 0), (3, 1), (7, 0), (7, 1), (20, 0)], window=5,
                          region=(int(pos[10]), int(pos[200])))
    assert sub.dprime is None and sub.haplotypes == [(0, 0), (3, 1), (7, 0), (7, 1), (20, 0)]
    assert all(pos[10] <= p <= pos[200] for p in sub.positions)
