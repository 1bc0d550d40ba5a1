"""The FP64 building blocks that let K4 (csrc/fm_wc.cuh) drop the per-pair divisions of
calculate_variance_components (stats.rs:2034-2127) without changing a rounding: fm_div_recip (a / b from the
correctly rounded reciprocal, two residual corrections) and fm_recip_rn (branch-free reciprocal) must equal
IEEE division bit for bit on the divisors the kernel meets."""
import numpy as np
import pytest

from ferromic_b200 import _lib

pytestmark = pytest.mark.gpu


def probe(a, b):
    L = _lib.lib()
    a = np.ascontiguousarray(a, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    y, q, q3 = np.empty_like(a), np.empty_like(a), np.empty_like(a)
    _lib.check(L.fm_wc_arith_probe(a.ctypes.data, b.ctypes.data, y.ctypes.data, q.ctypes.data, q3.ctypes.data, a.size))
    probe.q_int = q3
    return y, q


def test_division_by_table_reciprocal_is_ieee_division():
    rng = np.random.default_rng(5)
    n = 1 << 24
    k = rng.integers(1, 400_000, size=n).astype(np.float64)
    b = np.where(np.arange(n) % 3 == 0, k, np.where(np.arange(n) % 3 == 1, k * 0.5, k * k * 0.5))
    a = np.concatenate([rng.integers(0, 400_000, size=n // 2).astype(np.float64), rng.random(n - n // 2) * 3.0 - 1.0])
    _, q = probe(a, b)
    assert np.array_equal(q.view(np.uint64), (a / b).view(np.uint64))
    # the one-correction form K4 uses for integer-like divisors (n, n/2, n^2/2 with n < 2^19): provably exact there
    assert np.array_equal(probe.q_int.view(np.uint64), (a / b).view(np.uint64))


def test_branch_free_reciprocal_is_ieee_reciprocal():
    rng = np.random.default_rng(6)
    n = 1 << 24
    # the a-denominator 1 - c^2 lies in (0, 1]; cover [2^-20, 2) densely plus exact powers of two and 1 - ulp
    b = np.concatenate([rng.random(n) * 0.999 + 0.001, np.ldexp(rng.random(n // 4) + 1.0, rng.integers(-20, 1, n // 4)),
                        np.array([1.0, 0.5, 0.25, np.nextafter(0.5, 1.0), 0.75, 1.0 - 2.0 ** -30, 1.0 - 1.0 / 452.0 ** 2])])
    y, q = probe(b, b)
    assert np.array_equal(y.view(np.uint64), (1.0 / b).view(np.uint64))
    assert np.all(q == 1.0)
    # the documented exception (Markstein): a divisor whose significand is all ones; K4's divisor 1 - c^2 is either 1
    # or at most 1 - 1/(n_i + n_j)^2 and never has that form
    ones = np.array([np.nextafter(1.0, 0.0)])
    y1, _ = probe(ones, ones)
    assert y1[0] == 1.0 and 1.0 / ones[0] == np.nextafter(1.0, 2.0)


def test_reciprocal_of_every_pair_a_denominator():
    """Every 1 - c^2 of a pair with n_i, n_j <= 2048, formed as fm_wc_pair_site forms it: fm_recip_rn equals IEEE
    1 / b bit for bit, and no such divisor has the all-ones significand the residual correction cannot round."""
    n1, n2 = np.meshgrid(np.arange(1, 2049, dtype=np.float64), np.arange(1, 2049, dtype=np.float64))
    keep = n1 <= n2  # 1 - c^2 is symmetric in (n_i, n_j)
    n1, n2 = n1[keep], n2[keep]
    nsd = n1 + n2
    n_bar = nsd / 2.0
    d1 = n1 - n_bar
    aden = 1.0 - (2.0 * (d1 * d1)) / (nsd * n_bar)
    mant = aden.view(np.uint64) & np.uint64((1 << 52) - 1)
    assert not np.any(mant == np.uint64((1 << 52) - 1))
    y, q = probe(aden, aden)
    assert np.array_equal(y.view(np.uint64), (1.0 / aden).view(np.uint64))
    assert np.all(q == 1.0)


def test_one_correction_quotients_up_to_4096():
    """fm_div_recip_int on every quotient of its integer-divisor kinds with n <= 4096: a / n for 0 <= a <= n (the
    allele frequencies), n_bar / (n_bar - 1) for n_i + n_j = 3 .. 4096, and the halved divisors n / 2."""
    n = np.repeat(np.arange(1, 4097, dtype=np.int64), np.arange(2, 4098))
    a = np.concatenate([np.arange(k + 1) for k in range(1, 4097)]).astype(np.float64)
    nsum = np.arange(3, 4097, dtype=np.float64)
    n_bar = nsum / 2.0
    num = np.concatenate([a, n_bar, a[: n_bar.size]])
    den = np.concatenate([n.astype(np.float64), n_bar - 1.0, n_bar])
    probe(num, den)
    assert np.array_equal(probe.q_int.view(np.uint64), (num / den).view(np.uint64))


@pytest.mark.parametrize("max_allele,n_pops", [(3, 5), (7, 4), (15, 3)])
def test_wc_multi_allelic_per_site_values_are_bit_identical_to_the_oracle(max_allele, n_pops):
    """fm_k_wc_multi evaluates orc_variance_components term for term (one IEEE division per quotient): per-site overall
    and pairwise (a, b) over every allele present equal the oracle's, not only within a tolerance."""
    import ferromic_b200 as F
    from oracle import pyoracle as orc
    from tests.test_gpu_parity import _to_python_variants, make_multi_cohort
    S = 40
    g, pos = make_multi_cohort(700, S, max_allele, 0.08, seed=400 + max_allele)
    g[:, :, 1][g[:, :, 0] < 0] = -1
    g[:, :, 0][g[:, :, 1] < 0] = -1
    bounds = np.linspace(0, S, n_pops + 1).astype(int)
    left = np.full(S, 0xFFFF, dtype=np.uint16)
    for p in range(n_pops):
        left[bounds[p]:bounds[p + 1]] = p
    right = left.copy()
    left[2] = 0xFFFF
    right[7] = (right[7] + 1) % n_pops
    labels = sorted(str(i) for i in range(n_pops))
    vs, _ = orc.from_numpy(g, pos)
    region = (int(pos[0]), int(pos[-1]))
    ref = orc.wc_fst(vs, left, right, n_pops, region)
    got = F.wc_fst_from_membership(_to_python_variants(g, pos), labels, left, right, region)
    keys = [f"{labels[i]}_vs_{labels[j]}" for i in range(n_pops) for j in range(i + 1, n_pops)]
    n_checked = 0
    for i, s in enumerate(got.site_fst):
        assert s.variance_components_a == float(ref["a"][i]) and s.variance_components_b == float(ref["b"][i]), i
        if not ref["has_maps"][i]:
            continue
        for k, key in enumerate(keys):
            a, b = s.pairwise_variance_components[key]
            ra, rb = float(ref["pair_a"][i][k]), float(ref["pair_b"][i][k])
            assert a == ra and b == rb, (i, key, a, ra, b, rb)
            n_checked += 1
    assert n_checked > 0


def test_wc_per_site_values_are_bit_identical_to_the_oracle():
    """Per-site overall and pairwise (a, b) of the GPU path against the C oracle, which divides with IEEE `/` in
    the reference's operation order (stats.rs:2034-2127): not a single bit may differ."""
    import ferromic_b200 as F
    from oracle import pyoracle as orc
    from tests.synth import make_cohort
    from tests.test_gpu_parity import _to_python_variants
    for n_pops, S, V, missing in ((2, 40, 1500, 0.1), (5, 60, 900, 0.05), (26, 130, 300, 0.08)):
        g, pos, pops = make_cohort(V, S, n_pops=n_pops, sigma=0.08, missing_rate=missing, seed=300 + n_pops)
        g[:, :, 1][g[:, :, 0] < 0] = -1
        g[:, :, 0][g[:, :, 1] < 0] = -1
        left = np.full(S, 0xFFFF, dtype=np.uint16)
        for p, members in enumerate(pops):
            left[members] = p
        labels = sorted(str(i) for i in range(n_pops))
        vs, _ = orc.from_numpy(g, pos)
        region = (int(pos[0]), int(pos[-1]))
        ref = orc.wc_fst(vs, left, left, n_pops, region)
        got = F.wc_fst_from_membership(_to_python_variants(g, pos), labels, left, left, region)
        keys = [f"{labels[i]}_vs_{labels[j]}" for i in range(n_pops) for j in range(i + 1, n_pops)]
        n_checked = 0
        for i, s in enumerate(got.site_fst):
            assert s.variance_components_a == float(ref["a"][i]) and s.variance_components_b == float(ref["b"][i])
            if not ref["has_maps"][i]:
                continue
            for k, key in enumerate(keys):
                a, b = s.pairwise_variance_components[key]
                ra, rb = float(ref["pair_a"][i][k]), float(ref["pair_b"][i][k])
                assert (a == ra or (np.isnan(a) and np.isnan(ra))) and (b == rb or (np.isnan(b) and np.isnan(rb))), \
                    (i, key, a, ra, b, rb)
                n_checked += 1
        assert n_checked > 0
