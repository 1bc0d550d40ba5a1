"""The LD-pruning restatement (tests/ld_prune_reference.py) on the CPU: a plain per-pair Python loop on random data
with real linkage, and hand-built cases for the greedy rule, the strict threshold, the NaN rules and the pair rule."""
import numpy as np
import pytest

from tests import ld_prune_reference as lp
from tests import ld_reference as lr
from tests import pca_reference as pr


def linked_cohort(seed, n, V, missing=0.0, flip=0.08):
    """(raw u8 [V, n], called bool [V, n], positions): runs of sites that copy an earlier site with per-cell flips, so
    r^2 spans (0, 1] and chains of linked pairs occur; every site polymorphic."""
    rng = np.random.default_rng(seed)
    x = np.zeros((V, n), np.uint8)
    for v in range(V):
        if v and rng.random() < 0.7:
            src = x[v - int(rng.integers(1, min(v, 6) + 1))]
            x[v] = src ^ (rng.random(n) < rng.uniform(0.0, 2 * flip)).astype(np.uint8)
        else:
            x[v] = rng.random(n) < rng.uniform(0.1, 0.9)
        x[v, 0], x[v, 1] = 1, 0
    called = rng.random((V, n)) >= missing
    called[:, :2] = True
    x[~called] = 0
    return x, called, np.cumsum(rng.integers(1, 30, size=V)).astype(np.int64)


def plain_prune(x, called, window, pos, thr, max_distance=None):
    """O(M * window) loop over pairs from the per-cell definition; every site is kept (max_missing 1 - eps)."""
    M = x.shape[0]
    linked = set()
    n_linked = 0
    for i in range(M):
        for j in range(i + 1, min(M, i + window + 1)):
            if max_distance is not None and pos[j] - pos[i] > max_distance:
                continue
            both = called[i] & called[j]
            c = int(both.sum())
            a, b = int((x[i] & both).sum()), int((x[j] & both).sum())
            ab = int((x[i] & x[j] & both).sum())
            r2 = lr.stats(c, a, b, ab, fp64=True)[0]
            if r2 > thr:
                linked.add((i, j))
                n_linked += 1
    retained = []
    for j in range(M):
        if not any((i, j) in linked for i in retained):
            retained.append(j)
    return retained, n_linked


def _prune(x, called, pos, window, thr, max_distance=None):
    V, n = x.shape
    return lp.ld_prune(pr.rows_from_arrays(x, called), V, np.arange(n), window, pos, thr, max_distance,
                       max_missing=0.99)


@pytest.mark.parametrize("seed,missing,window,thr", [(1, 0.0, 20, 0.2), (2, 0.05, 7, 0.5), (3, 0.02, 40, 0.05),
                                                     (4, 0.0, 33, 0.9)])
def test_plain_loop_agrees(seed, missing, window, thr):
    x, called, pos = linked_cohort(seed, 40, 120, missing)
    got = _prune(x, called, pos, window, thr)
    assert got["M"] == 120
    ret, n_linked = plain_prune(x, called, window, pos, thr)
    assert got["retained"].tolist() == ret and got["linked_pairs"] == n_linked
    assert 0 < n_linked < got["pairs"] and 0 < len(ret) < 120


def test_perfect_ld_keeps_the_first_site():
    rng = np.random.default_rng(5)
    row = (rng.random(30) < 0.4).astype(np.uint8)
    row[0], row[1] = 1, 0
    x = np.tile(row, (50, 1))
    got = _prune(x, np.ones_like(x, bool), np.arange(50), 60, 0.2)  # window >= M - 1: the full triangle
    assert got["retained"].tolist() == [0] and got["linked_pairs"] == got["pairs"] == 50 * 49 // 2


def test_against_retained_not_kept():
    """A-B and B-C linked (r^2 = 0.25), A-C not (r^2 = 0): A and C are retained."""
    A = [1, 1, 1, 1, 0, 0, 0, 0]
    B = [1, 1, 1, 0, 1, 0, 0, 0]
    C = [1, 1, 0, 0, 1, 1, 0, 0]
    x = np.array([A, B, C], np.uint8)
    r2 = lambda i, j: lr.stats(8, x[i].sum(), x[j].sum(), (x[i] & x[j]).sum(), fp64=True)[0]  # noqa: E731
    assert r2(0, 1) == r2(1, 2) == 0.25 and r2(0, 2) == 0.0
    got = _prune(x, np.ones_like(x, bool), np.arange(3), 2, 0.2)
    assert got["retained"].tolist() == [0, 2] and got["linked_pairs"] == 2
    assert plain_prune(x, np.ones_like(x, bool), 2, np.arange(3), 0.2)[0] == [0, 2]


def test_threshold_is_strict():
    """The r^2 = 0.6 table of tests/test_ld_reference.py: not linked at its own FP64 r^2, linked one ulp below."""
    x = np.array([[1, 1, 1, 1, 0, 0, 0, 0], [1, 1, 1, 0, 0, 0, 0, 0]], np.uint8)
    r2 = lr.stats(8, 4, 3, 3, fp64=True)[0]
    assert r2 == pytest.approx(0.6, abs=1e-15)
    ones = np.ones_like(x, bool)
    assert _prune(x, ones, np.arange(2), 1, float(r2))["retained"].tolist() == [0, 1]
    got = _prune(x, ones, np.arange(2), 1, float(np.nextafter(r2, 0.0)))
    assert got["retained"].tolist() == [0] and got["linked_pairs"] == 1
    assert _prune(x, ones, np.arange(2), 1, 1.0)["linked_pairs"] == 0


def test_nan_pairs_never_link():
    """Sites 0 and 1 are never called together (c = 0); site 2 is monomorphic among the haplotypes called at both 2
    and 3; sites 3 and 4 have r^2 = 0 exactly.  At threshold 0 none of these pairs links."""
    x = np.zeros((5, 8), np.uint8)
    called = np.ones((5, 8), bool)
    x[0, :4] = [1, 0, 1, 0]
    called[0, 4:] = False
    x[1, 4:] = [1, 0, 1, 0]
    called[1, :4] = False
    x[2] = [1, 1, 1, 1, 1, 1, 0, 0]
    called[3, 6:] = False
    x[3, :6] = [1, 0, 1, 0, 1, 0]
    x[4] = [1, 1, 0, 0, 0, 0, 0, 0]  # with site 3: c = 6, a = 3, b = 2, ab = 1 -> Dn = 0
    got = _prune(x, called, np.arange(5), 1, 0.0)
    assert got["M"] == 5 and got["linked_pairs"] == 0 and got["retained"].tolist() == [0, 1, 2, 3, 4]
    assert plain_prune(x, called, 1, np.arange(5), 0.0) == ([0, 1, 2, 3, 4], 0)


def test_window_and_distance_limits():
    rng = np.random.default_rng(9)
    row = (rng.random(20) < 0.5).astype(np.uint8)
    row[0], row[1] = 1, 0
    x = np.tile(row, (10, 1))  # every pair has r^2 = 1
    ones = np.ones_like(x, bool)
    pos = np.array([0, 5, 10, 100, 105, 300, 301, 302, 1000, 1001], np.int64)
    for window, step in ((1, 2), (3, 4), (9, 10), (20, 10)):
        got = _prune(x, ones, pos, window, 0.5)
        assert got["retained"].tolist() == list(range(0, 10, step))
    got = _prune(x, ones, pos, 9, 0.5, max_distance=10)
    assert got["retained"].tolist() == [0, 3, 5, 8]
    assert got["retained"].tolist() == plain_prune(x, ones, 9, pos, 0.5, max_distance=10)[0]


def test_site_list_subset():
    """subset_rows leaves the listed rows as they are and keeps no other row."""
    x, called, pos = linked_cohort(11, 24, 60, 0.02)
    rows = pr.rows_from_arrays(x, called)
    listed = [3, 4, 10, 17, 30, 31, 59]
    sub = lp.subset_rows(rows, listed)
    kept = pr.site_stats(sub, 0, 60, np.arange(24), 0.0, 0.5)[0]
    assert kept.tolist() == listed
    full = lp.ld_prune(rows, 60, np.arange(24), 5, pos, 0.2, max_missing=0.5)
    part = lp.ld_prune(sub, 60, np.arange(24), 5, pos, 0.2, max_missing=0.5)
    assert part["kept"].tolist() == listed and set(part["retained"]) <= set(listed)
    assert full["M"] == 60
