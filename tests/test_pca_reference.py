"""CPU checks of the haplotype PCA restatement (tests/pca_reference.py): its test matrix, its agreement with a
dense SVD, its total variance and its site filters at their boundaries; and the entry point's refusal to run
without a device."""
import ctypes as C

import numpy as np
import pytest

from tests import pca_reference as pr

# G[0, c], c = 0 .. 15, for seed 1 (computed once from fm_mix; tests/test_gpu_pca.py checks the device's G)
GOLDEN_SIGNS_SEED1 = [1, -1, -1, -1, -1, 1, 1, 1, 1, 1, -1, -1, 1, -1, 1, 1]


def _flat(a, miss):
    V = a.shape[0]
    return a.reshape(V, -1), ~miss.reshape(V, -1)


def test_test_matrix_golden_signs():
    assert pr.rademacher(1, [0], 16)[0].astype(int).tolist() == GOLDEN_SIGNS_SEED1
    g = pr.rademacher(1, np.arange(4096), 64)
    assert set(np.unique(g)) == {-1.0, 1.0} and abs(g.mean()) < 0.02


@pytest.mark.parametrize("missing", [0.0, 0.02])
def test_restatement_matches_dense_svd(missing):
    n_pops, k = 5, 3
    a, miss, pos, _ = pr.cohort(7, n_pops, 30, 1500, missing=missing)
    raw, called = _flat(a, miss)
    off = pr.offsets([(s, h) for s in range(a.shape[1]) for h in (0, 1)], a.shape[1], 2)
    r = pr.haplotype_pca(pr.rows_from_arrays(raw, called), a.shape[0], off, k, oversampling=10, power_iterations=8,
                         max_missing=0.2, dense=True)
    U, sv, _ = np.linalg.svd(r["Z"], full_matrices=False)
    assert np.all(sv[:k] / sv[1:k + 1] >= 1.01), "top-(k+1) singular values are not separated by 1 %"
    assert np.all(np.abs(r["singular_values"] - sv[:k]) <= 1e-8 * sv[:k])
    u = r["scores"] / r["singular_values"]
    assert np.all(np.abs(np.sum(u * U[:, :k], axis=0)) >= 1 - 1e-8)
    assert r["T"] == pytest.approx(float(np.sum(r["Z"] ** 2)), rel=1e-12)
    assert r["T"] == int(called[r["kept"]][:, off].sum())


def _one_site_cases():
    """Sites over n = 10 haplotypes (5 diploid samples) at their filter boundaries: (raw, called, kept?) with
    min_maf = 0.2 and max_missing = 0.2."""
    c10 = np.ones(10, bool)
    c8 = np.array([1] * 8 + [0] * 2, bool)
    c7 = np.array([1] * 7 + [0] * 3, bool)
    return [
        (np.array([1, 1] + [0] * 8, np.uint8), c10, True),            # minor 2 = 0.2 * 10: met exactly
        (np.array([1] + [0] * 9, np.uint8), c10, False),              # minor 1 < 2
        (np.array([1, 1, 1] + [0] * 7, np.uint8), c8, True),          # 2 missing = 0.2 * 10: met exactly
        (np.array([1, 1, 1] + [0] * 7, np.uint8), c7, False),         # 3 missing > 2
        (np.array([1, 1, 2] + [0] * 7, np.uint8), c10, False),        # an extra allele value
        (np.array([1, 1, 1] + [0] * 5 + [2, 2], np.uint8), c8, True),  # the extra value sits in missing cells
        (np.array([17, 17, 17] + [0] * 7, np.uint8), c10, False),     # {0, 17}: no raw 1 (ranks would be {0, 1})
        (np.array([1, 1, 17] + [0] * 7, np.uint8), c10, False),       # {0, 1, 17}
        (np.array([1] * 10, np.uint8), c10, False),                   # monomorphic
    ]


def test_filter_boundaries():
    cases = _one_site_cases()
    raw = np.stack([c[0] for c in cases])
    called = np.stack([c[1] for c in cases])
    kept, cal, alt = pr.site_stats(pr.rows_from_arrays(raw, called), 0, len(cases), np.arange(10), 0.2, 0.2)
    assert kept.tolist() == [i for i, c in enumerate(cases) if c[2]]
    assert cal.tolist() == [10, 8, 8] and alt.tolist() == [2, 3, 3]


def test_entry_point_fails_without_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device is present")
    import ferromic_b200 as fm
    from ferromic_b200 import _lib
    with pytest.raises(fm.FerromicGpuError) as exc:
        fm.haplotype_pca([(1, [[0, 1], [1, 1]]), (2, [[1, 0], [0, 0]])], n_components=1)
    assert exc.value.code == _lib.FM_ERR_NO_DEVICE
    info = _lib.PcaInfo()
    prm = _lib.PcaParams(1, 0, 0, 0.0, 0.0, 0, 0, 0, 0)
    assert _lib.lib().fm_haplotype_pca(None, None, None, 0, C.byref(prm), None, None, None, None, None, None, 0,
                                       C.byref(info)) == _lib.FM_ERR_NO_DEVICE
