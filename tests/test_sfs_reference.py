"""The site-frequency-spectrum restatement (tests/sfs_reference.py) on the CPU: FP64 weights against exact rationals,
hand cases, the mass of the fold, the Tajima's D edge cases and the entry points without a device."""
import ctypes as C
import math
from fractions import Fraction

import numpy as np
import pytest

from tests import sfs_reference as sr


def test_fp64_weights_match_exact_rationals():
    """Every N in a grid up to 5008, every m (a stride of them at large N) and a spread of a: within 1e-12."""
    rng = np.random.default_rng(1)
    worst = 0.0
    for N in (1, 2, 3, 4, 5, 7, 16, 17, 33, 100, 257, 1000, 5008):
        ms = range(1, N + 1) if N <= 100 else sorted({1, 2, 3, N - 1, N, *rng.integers(1, N + 1, 6).tolist()})
        for m in ms:
            for a in sorted({0, 1, N // 2, N - 1, N, int(rng.integers(0, N + 1))} - {-1}):
                if not 0 <= a <= N:
                    continue
                lo, w = sr.weights_fp64(N, a, m)
                lo2, e = sr.weights_exact(N, a, m)
                assert lo == lo2 and len(w) == len(e)
                for x, f in zip(w, e):
                    if f > Fraction(1, 10 ** 290):
                        worst = max(worst, float(abs(Fraction(float(x)) - f) / f))
                    else:
                        assert x < 1e-280
    assert worst < 1e-12, worst


def test_hand_cases():
    lo, w = sr.weights_fp64(4, 2, 2)
    assert lo == 0 and w.tolist() == pytest.approx([1 / 6, 2 / 3, 1 / 6], rel=1e-15)
    assert [str(f) for f in sr.weights_exact(4, 2, 2)[1]] == ["1/6", "2/3", "1/6"]
    assert sr.weights_fp64(10, 4, 10) == (4, pytest.approx(np.array([1.0])))
    assert sr.weights_fp64(10, 4, 10)[1][0] == 1.0  # N == m: exactly one
    for N, a, m in ((50, 20, 13), (5008, 2500, 4900), (300, 1, 150), (1000, 999, 999)):
        lo, w = sr.weights_fp64(N, a, m)
        assert math.fsum(w) == pytest.approx(1.0, abs=1e-13)
        assert math.fsum(w * np.arange(lo, lo + len(w))) == pytest.approx(a * m / N, rel=1e-12)


def _cohort(seed, V, n, missing):
    rng = np.random.default_rng(seed)
    f = rng.beta(0.3, 0.3, V)
    raw = (rng.random((V, n)) < f[:, None]).astype(np.uint8)
    called = rng.random((V, n)) >= missing
    raw[~called] = 0
    return raw, called


def test_spectrum_mass_and_mean():
    """Each contributing row adds mass 1 and mean a m / N, so sum xi = n_sites and sum j xi_j = sum a m / N."""
    raw, called = _cohort(2, 400, 30, 0.1)
    raw[::37, 3] = 2
    off = np.arange(30)
    for m in (1, 5, 24, 30):
        r = sr.sfs(raw, called, off, m)
        cal, alt, oth = sr.site_counts(raw, called, off)
        keep = (oth == 0) & (cal >= m)
        assert r["n_sites"] == keep.sum() and r["non_biallelic"] == (oth > 0).sum()
        assert r["projected_out"] == ((oth == 0) & (cal < m)).sum()
        xi = r["spectrum"][0]
        assert math.fsum(xi) == pytest.approx(r["n_sites"], rel=1e-12)
        assert math.fsum(xi * np.arange(m + 1)) == pytest.approx(math.fsum(alt[keep] * m / cal[keep]), rel=1e-12)
    exact = sr.sfs(raw, called, off, 7, exact=True)["spectrum"]
    np.testing.assert_allclose(sr.sfs(raw, called, off, 7)["spectrum"], exact, rtol=1e-12, atol=0)


@pytest.mark.parametrize("m1,m2", [(6, 0), (7, 0), (1, 0), (4, 4), (3, 5), (4, 7), (5, 5), (0, 3)])
def test_fold_keeps_mass(m1, m2):
    rng = np.random.default_rng(m1 * 10 + m2)
    x = rng.random((m1 + 1) * (m2 + 1))
    f = sr.fold(x, m1, m2) if m2 else sr.fold(x, m1)
    assert math.fsum(np.ravel(f)) == pytest.approx(math.fsum(x), rel=1e-14)
    f = np.reshape(f, (m1 + 1, m2 + 1))
    X = x.reshape(m1 + 1, m2 + 1)
    if (m1 + m2) % 2 == 0 and m1 % 2 == 0 and m2 % 2 == 0:  # the centre entry stays as it is
        assert f[m1 // 2, m2 // 2] == X[m1 // 2, m2 // 2]
    assert f[0, 0] == X[0, 0] + X[m1, m2]
    assert f[m1, m2] == 0.0


def test_tajimas_d_edges():
    nan = lambda v: v != v  # noqa: E731
    for m in (1, 2, 3):
        xi = np.ones(m + 1)
        assert nan(sr.stats(xi, m)[3])
    xi = np.zeros(11)
    xi[0], xi[10] = 5.0, 2.0
    S, tp, tw, D = sr.stats(xi, 10)
    assert S == 0.0 and tp == 0.0 and tw == 0.0 and nan(D)
    xi = np.zeros(11)
    xi[5] = -0.5  # a negative radicand e1 S + e2 S (S - 1)
    assert nan(sr.stats(xi, 10)[3])
    xi = np.zeros(11)
    xi[1], xi[5] = 2.0, 3.0
    S, tp, tw, D = sr.stats(xi, 10)
    a1 = sum(1 / i for i in range(1, 10))
    assert S == 5.0 and tw == pytest.approx(5.0 / a1, rel=1e-15)
    assert tp == pytest.approx((9 * 2 + 25 * 3) / 45, rel=1e-15)
    # Tajima (1989) in exact rationals: n = 10, S = 5, k = 93 / 45
    n, Sf = 10, Fraction(5)
    A1 = sum(Fraction(1, i) for i in range(1, n))
    A2 = sum(Fraction(1, i * i) for i in range(1, n))
    B1, B2 = Fraction(n + 1, 3 * (n - 1)), Fraction(2 * (n * n + n + 3), 9 * n * (n - 1))
    C1, C2 = B1 - 1 / A1, B2 - Fraction(n + 2, n) / A1 + A2 / (A1 * A1)
    var = C1 / A1 * Sf + C2 / (A1 * A1 + A2) * Sf * (Sf - 1)
    assert D == pytest.approx(float(Fraction(93, 45) - Sf / A1) / math.sqrt(float(var)), rel=1e-13)


def test_entry_point_fails_without_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device is present")
    import ferromic_b200 as fm
    from ferromic_b200 import _lib
    variants = [(1, [[0, 1], [1, 1]]), (2, [[1, 0], [0, 0]])]
    for call in (lambda: fm.site_frequency_spectrum(variants),
                 lambda: fm.joint_site_frequency_spectrum(variants, [(0, 0)], [(1, 0)])):
        with pytest.raises(fm.FerromicGpuError) as exc:
            call()
        assert exc.value.code == _lib.FM_ERR_NO_DEVICE
    info = _lib.SfsInfo()
    prm = _lib.SfsParams(0, 0, 0, 0, 0)
    assert _lib.lib().fm_site_frequency_spectrum(None, None, None, 0, C.byref(prm), None, 0, None, None, 0, None, None,
                                                 None, None, None, C.byref(info)) == _lib.FM_ERR_NO_DEVICE
    jinfo = _lib.JointSfsInfo()
    jprm = _lib.JointSfsParams(0, 0, 0, 0, 0, 0)
    assert _lib.lib().fm_joint_site_frequency_spectrum(None, None, None, 0, None, None, 0, C.byref(jprm), None, 0,
                                                       C.byref(jinfo)) == _lib.FM_ERR_NO_DEVICE
