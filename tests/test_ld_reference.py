"""CPU checks of the haplotype LD restatement (tests/ld_reference.py), independent of its own arithmetic: r^2 against
np.corrcoef over the jointly called haplotypes, worked two-site tables, every NaN rule and the band, distance and
window rules on hand-built positions; and the entry point's refusal to run without a device."""
import ctypes as C

import numpy as np
import pytest

from tests import ld_reference as lr
from tests import pca_reference as pr


def _flat(a, miss):
    V = a.shape[0]
    return a.reshape(V, -1), ~miss.reshape(V, -1)


@pytest.mark.parametrize("missing", [0.0, 0.05])
def test_r2_matches_corrcoef(missing):
    a, miss, pos, _ = pr.cohort(21, 3, 30, 300, missing=missing)
    raw, called = _flat(a, miss)
    off = pr.offsets([(s, h) for s in range(a.shape[1]) for h in (0, 1)], a.shape[1], 2)
    window = 40
    r = lr.haplotype_ld(pr.rows_from_arrays(raw, called), a.shape[0], off, window, pos, max_missing=0.2)
    M, kept = r["M"], r["kept"]
    assert M > 200
    x, c = raw[kept][:, off].astype(np.float64), called[kept][:, off]
    checked = 0
    for d in (1, 7, window):
        r64, _ = lr.stats(*r["counts"][d], fp64=True)
        for i in range(0, M - d, 5):
            j = i + d
            both = c[i] & c[j]
            want = np.corrcoef(x[i, both], x[j, both])[0, 1] ** 2
            assert abs(r64[i] - want) <= 1e-12
            assert r["r2"][i, d - 1] == np.float32(r64[i])
            checked += 1
    assert checked > 100


def _pair_counts(haps_i, haps_j):
    """(c, a, b, ab) from per-haplotype values with None for missing."""
    both = [(x, y) for x, y in zip(haps_i, haps_j) if x is not None and y is not None]
    return (len(both), sum(x for x, _ in both), sum(y for _, y in both), sum(x & y for x, y in both))


def _table(n_AB, n_Ab, n_aB, n_ab):
    """Haplotypes of two sites from a 2 x 2 table (A / B = alt)."""
    hi = [1] * (n_AB + n_Ab) + [0] * (n_aB + n_ab)
    hj = [1] * n_AB + [0] * n_Ab + [1] * n_aB + [0] * n_ab
    return hi, hj


def test_worked_tables():
    r2, dp = lr.stats(*_pair_counts(*_table(3, 1, 0, 4)), fp64=True)
    assert r2 == pytest.approx(0.6, abs=1e-15) and dp == 1.0
    # the same allele counts, coupling reversed: no haplotype carries both alt alleles
    hi = [1, 1, 1, 1, 0, 0, 0, 0]
    hj = [0, 0, 0, 0, 1, 1, 1, 0]
    assert _pair_counts(hi, hj) == (8, 4, 3, 0)
    r2, dp = lr.stats(*_pair_counts(hi, hj), fp64=True)
    assert r2 == pytest.approx(0.6, abs=1e-15) and dp == -1.0
    r2, dp = lr.stats(4, 2, 2, 1, fp64=True)
    assert r2 == 0.0 and dp == 0.0
    assert lr.stats(4, 2, 2, 1)[1].view(np.uint32) == np.float32(0.0).view(np.uint32)  # +0, not -0


def test_nan_rules():
    # c == 0; a in {0, c}; b in {0, c}
    cases = [(0, 0, 0, 0), (5, 0, 2, 0), (5, 5, 2, 2), (5, 2, 0, 0), (5, 2, 5, 2)]
    r2, dp = lr.stats(*np.array(cases).T)
    assert np.all(r2.view(np.uint32) == 0x7FC00000) and np.all(dp.view(np.uint32) == 0x7FC00000)
    # a site polymorphic overall but monomorphic among the haplotypes called at both sites
    hi = [1, 0, None, 1, 1]
    hj = [1, 1, 0, None, 1]
    assert _pair_counts(hi, hj) == (3, 2, 3, 2)
    assert np.isnan(lr.stats(*_pair_counts(hi, hj))[0])


def _grid(M, n=12, seed=3, missing=0.0):
    """M polymorphic sites over n haploid samples with given missingness (nothing filtered at max_missing 0.9)."""
    rng = np.random.default_rng(seed)
    raw = (rng.random((M, n)) < 0.5).astype(np.uint8)
    raw[:, 0], raw[:, 1] = 1, 0
    called = rng.random((M, n)) >= missing
    called[:, :2] = True
    return raw, called


def test_band_window_and_distance_rules():
    M = 9
    raw, called = _grid(M, missing=0.2)
    pos = np.array([0, 10, 10, 25, 40, 41, 100, 150, 151], np.int64)  # a gap, duplicates, a pair at exactly 15
    get = pr.rows_from_arrays(raw, called)
    off = np.arange(12)
    full = lr.haplotype_ld(get, M, off, M + 5, pos, max_missing=0.9)
    assert full["M"] == M and full["pairs"] == M * (M - 1) // 2
    r2 = full["r2"]
    for i in range(M):  # every cell with i + d >= M is NaN; the others are set when the counts allow it
        assert np.all(np.isnan(r2[i, M - 1 - i:]))
        assert not np.any(np.isnan(r2[i, :M - 1 - i]))
    band = lr.haplotype_ld(get, M, off, 3, pos, max_missing=0.9)
    assert band["r2"].shape == (M, 3) and band["pairs"] == 8 + 7 + 6
    assert np.array_equal(band["r2"].view(np.uint32), np.where(
        np.arange(3)[None, :] < (M - 1 - np.arange(M))[:, None], r2[:, :3].view(np.uint32), 0x7FC00000))
    near = lr.haplotype_ld(get, M, off, M - 1, pos, max_distance=15, max_missing=0.9)
    want = {(i, j) for i in range(M) for j in range(i + 1, M) if pos[j] - pos[i] <= 15}
    assert (3, 4) in want and (0, 1) in want and (2, 3) in want and (1, 3) in want and (0, 3) not in want
    got = {(i, i + d + 1) for i in range(M) for d in range(M - 1) if not np.isnan(near["r2"][i, d])}
    assert got == want and near["pairs"] == len(want)
    for i, j in want:
        assert near["r2"][i, j - i - 1].view(np.uint32) == r2[i, j - i - 1].view(np.uint32)


def test_filters_and_region():
    """Kept sites follow the PCA filters; pairs are counted between kept sites, in kept order."""
    from tests.test_pca_reference import _one_site_cases
    cases = _one_site_cases()
    raw = np.stack([c[0] for c in cases])
    called = np.stack([c[1] for c in cases])
    pos = np.arange(len(cases), dtype=np.int64) * 3
    r = lr.haplotype_ld(pr.rows_from_arrays(raw, called), len(cases), np.arange(10), 2, pos, min_maf=0.2,
                        max_missing=0.2)
    assert r["kept"].tolist() == [i for i, c in enumerate(cases) if c[2]] and r["M"] == 3
    sub = lr.haplotype_ld(pr.rows_from_arrays(raw, called), len(cases), np.arange(10), 2, pos, min_maf=0.2,
                          max_missing=0.2, site_range=(1, len(cases)))
    assert sub["kept"].tolist() == r["kept"].tolist()[1:]
    assert sub["r2"][0, 0].view(np.uint32) == r["r2"][1, 0].view(np.uint32)


def test_entry_point_fails_without_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device is present")
    import ferromic_b200 as fm
    from ferromic_b200 import _lib
    with pytest.raises(fm.FerromicGpuError) as exc:
        fm.haplotype_ld([(1, [[0, 1], [1, 1]]), (2, [[1, 0], [0, 0]])], window=1)
    assert exc.value.code == _lib.FM_ERR_NO_DEVICE
    info = _lib.LdInfo()
    prm = _lib.LdParams(1, -1, 0.0, 0.0, 0, 0, 0)
    assert _lib.lib().fm_haplotype_ld(None, None, None, 0, C.byref(prm), None, None, 0, None, None, 0,
                                      C.byref(info)) == _lib.FM_ERR_NO_DEVICE
