"""The haplotype-frequency restatement (tests/hapfreq_reference.py) on the CPU: against a plain dict of key tuples,
hand-worked windows, scikit-allel's float formulas (garud_h, haplotype_diversity) written out, and the enumeration
of count windows with the dropped partial window."""
import math

import numpy as np

from tests import hapfreq_reference as hr


def _cohort(seed, V, cells, missing=0.0):
    rng = np.random.default_rng(seed)
    founders = rng.random((4, V)) < 0.4
    pick = rng.choice(4, size=cells, p=[0.55, 0.25, 0.15, 0.05])
    raw = founders[pick].T.astype(np.uint8)  # [V, cells]
    flip = rng.random((V, cells)) < 0.01
    raw ^= flip.astype(np.uint8)
    called = ~(rng.random((V, cells)) < missing)
    return raw, called


def _allel_garud_h(sizes):
    """scikit-allel's garud_h on the class counts of one window (allel.stats.selection.garud_h), written out."""
    n = float(np.sum(sizes))
    f = np.sort(np.asarray(sizes, np.float64))[::-1] / n
    h1 = np.sum(f ** 2)
    h12 = np.sum(f[:2]) ** 2 + np.sum(f[2:] ** 2)
    h123 = np.sum(f[:3]) ** 2 + np.sum(f[3:] ** 2)
    h2_h1 = (h1 - f[0] ** 2) / h1
    return h1, h12, h123, h2_h1


def _allel_haplotype_diversity(sizes):
    """allel.haplotype_diversity: (1 - sum p^2) * n / (n - 1)."""
    n = float(np.sum(sizes))
    f = np.asarray(sizes, np.float64) / n
    return (1 - np.sum(f ** 2)) * n / (n - 1)


def test_against_a_dict_of_key_tuples():
    raw, called = _cohort(1, 300, 90, missing=0.01)
    off = np.arange(90)
    ref = hr.haplotype_frequencies(raw, called, off, max_missing=0.05, size=37, step=11)
    kept = ref["kept"]
    for (f, s), counts, nu, k in zip(ref["windows"], ref["counts"], ref["n_used"], ref["distinct"]):
        d = {}
        rows = kept[f:f + s]
        for h in off:
            if not called[rows, h].all():
                continue
            key = tuple(int(raw[v, h] == 1) for v in rows)
            d[key] = d.get(key, 0) + 1
        assert sorted(d.values(), reverse=True) == counts.tolist()
        assert nu == sum(d.values()) and k == len(d)
    assert any(n < 90 for n in ref["n_used"])  # some windows drop a haplotype


def test_hand_worked_windows():
    # all identical: H1 = 1, H12 = 1, H2/H1 = 0, diversity 0
    N, K, top, s2, h1, h12, h123, h21, div = hr.statistics([7])
    assert (N, K, top, s2) == (7, 1, (7, 0, 0), 49) and (h1, h12, h123, h21, div) == (1.0, 1.0, 1.0, 0.0, 0.0)
    # all distinct (N = 8): H1 = 1/8, H12 = (2/8)^2 + 6/64, H123 = (3/8)^2 + 5/64, diversity 1
    N, K, top, s2, h1, h12, h123, h21, div = hr.statistics([1] * 8)
    assert (N, K, top, s2) == (8, 8, (1, 1, 1), 8)
    assert h1 == 1 / 8 and h12 == 10 / 64 and h123 == 14 / 64 and h21 == 7 / 8 and div == 1.0
    # N == 0: everything NaN; N == 1: only diversity NaN
    st = hr.statistics([])
    assert st[:4] == (0, 0, (0, 0, 0), 0) and all(math.isnan(x) for x in st[4:])
    st = hr.statistics([1])
    assert st[4:8] == (1.0, 1.0, 1.0, 0.0) and math.isnan(st[8])
    # two classes 3 + 1: s2 = 10, h12 = (10 + 6) / 16 = 1
    st = hr.statistics([1, 3])
    assert st[2:5] == ((3, 1, 0), 10, 10 / 16) and st[5] == 1.0 and st[7] == 1 / 10 and st[8] == 6 / 12
    # a window without kept sites: every used haplotype in one class
    assert hr.class_sizes(np.zeros((5, 0), bool)).tolist() == [5]
    assert hr.class_sizes(np.zeros((0, 3), bool)).tolist() == []


def test_against_scikit_allel_formulas():
    raw, called = _cohort(2, 400, 150)
    ref = hr.haplotype_frequencies(raw, called, np.arange(150), size=50, step=25)
    assert len(ref["windows"]) == (len(ref["kept"]) - 50) // 25 + 1
    for w, sizes in enumerate(ref["counts"]):
        a = _allel_garud_h(sizes)
        for got, exp in zip((ref["h1"][w], ref["h12"][w], ref["h123"][w], ref["h2_h1"][w]), a):
            assert abs(got - exp) <= 1e-12 * abs(exp) + 1e-15
        d = _allel_haplotype_diversity(sizes)
        assert abs(ref["diversity"][w] - d) <= 1e-12 * abs(d) + 1e-15
    assert min(ref["distinct"]) > 1 and max(ref["h12"]) > max(ref["h1"])


def test_count_window_enumeration():
    assert hr.count_windows(10, 3) == [(0, 3), (3, 3), (6, 3)]  # [9, 12) is partial: dropped
    assert hr.count_windows(10, 3, 2) == [(0, 3), (2, 3), (4, 3), (6, 3)]  # [8, 11) dropped
    assert hr.count_windows(10, 4, 5) == [(0, 4), (5, 4)]
    assert hr.count_windows(10, 10) == [(0, 10)] and hr.count_windows(9, 10) == []
    assert hr.count_windows(5, 1) == [(i, 1) for i in range(5)]
    pos = np.array([10, 20, 30, 40])
    assert hr.position_windows(pos, [(0, 9), (10, 10), (15, 35), (41, 100), (30, 20)]) == [
        (0, 0), (0, 1), (1, 2), (4, 0), (2, 0)]
