"""CPU checks of pairwise_differences (calculate_pairwise_differences, stats.rs:4106-4231; parity unpinned, see
DESIGN.md §3): the oracle's direct loop on hand-made cases, the bit-plane algebra the GPU kernels evaluate
(DESIGN.md §4 "Pairwise differences") against that loop, and the loud failure without a device."""
import ctypes as C

import numpy as np
import pytest

from oracle import pyoracle as orc
from tests import pairwise_oracle as po

WORKED = [(10, [[0, 0], [0, 1], [1, 1]]), (20, [[0, 0], [0, 0], [0, 1]]), (30, [[0, 1], None, [1, 0]])]


def _as_list(diff, start, pos, n):
    out, k = [], 0
    for i in range(n):
        for j in range(i + 1, n):
            out.append(((i, j), int(diff[k]), [int(p) for p in pos[start[k]:start[k + 1]]]))
            k += 1
    return out


def test_oracle_worked_example():
    d, c, s, p = po.pairwise_differences(orc.variants_from_python(WORKED), 3)
    assert _as_list(d, s, p, 3) == [((0, 1), 1, [10]), ((0, 2), 3, [10, 20, 30]), ((1, 2), 2, [10, 20])]
    assert list(c) == [2, 3, 2]


def test_oracle_short_genotypes_and_phase():
    # [1] != [1, 0] (length counts), [0, 1] != [1, 0] (phase counts), a sample past the row is None
    vs = orc.variants_from_python([(5, [[1], [1, 0], [1]]), (7, [[0, 1], [1, 0], [0, 1]]), (9, [[2, 2], [2, 2]])],
                                  n_samples=3)
    d, c, s, p = po.pairwise_differences(vs, 4)
    got = _as_list(d, s, p, 4)
    assert got == [((0, 1), 2, [5, 7]), ((0, 2), 0, []), ((0, 3), 0, []), ((1, 2), 2, [5, 7]), ((1, 3), 0, []),
                   ((2, 3), 0, [])]
    assert list(c) == [3, 2, 0, 2, 0, 0]


def test_oracle_multiallelic():
    vs = orc.variants_from_python([(0, [[3, 7], [3, 7], [7, 3]]), (1, [[200, 0], [200, 0], [200, 1]]),
                                   (2, [[15, 15], None, [15, 15]])])
    d, c, s, p = po.pairwise_differences(vs, 3)
    assert _as_list(d, s, p, 3) == [((0, 1), 0, []), ((0, 2), 2, [0, 1]), ((1, 2), 2, [0, 1])]
    assert list(c) == [2, 3, 2]


def test_oracle_threaded_form_matches():
    rng = np.random.default_rng(7)
    gt = rng.integers(0, 3, size=(300, 45, 2)).astype(np.uint8)
    gt[rng.random((300, 45)) < 0.1, 0] = 0xFF
    gt[rng.random((300, 45)) < 0.1, 1] = 0xFF
    vs = orc.Variants(np.arange(300, dtype=np.int64) * 3, gt)
    d1, c1, _, _ = po.pairwise_differences(vs, 45)
    d2, c2, _, _ = po.pairwise_differences(vs, 45, threads=4)
    assert np.array_equal(d1, d2) and np.array_equal(c1, c2)


def _planes(gt, n_bits, with_called):
    """Bit planes per (site, sample): pc_p = cells 0..p called, a_{p,k} = bit k of the allele rank of cell p masked
    by pc_p (ranks of the distinct values, as the matrix's rank table assigns them)."""
    called = np.logical_and.accumulate(gt != 0xFF, axis=2)
    values = np.unique(gt[gt != 0xFF])
    rank = np.zeros(256, dtype=np.int64)
    rank[values] = np.arange(values.size)
    r = rank[gt]
    out = [called[..., p] for p in range(gt.shape[2])] if with_called else []
    for p in range(gt.shape[2]):
        out += [((r[..., p] >> k) & 1).astype(bool) & called[..., p] for k in range(n_bits)]
    return out


@pytest.mark.parametrize("seed", range(40))
def test_bit_plane_algebra_matches_direct_loop(seed):
    """The identity the transpose + bit-GEMM kernels evaluate, on random None / haploid / diploid mixes with up to
    16 distinct allele values (including values above 15)."""
    rng = np.random.default_rng(seed)
    V, S = int(rng.integers(1, 60)), int(rng.integers(2, 12))
    pool = np.array([0, 1, 2, 3, 17, 40, 99, 254][: int(rng.integers(2, 9))], dtype=np.uint8)
    gt = pool[rng.integers(0, pool.size, size=(V, S, 2))]
    ln = rng.choice(3, size=(V, S), p=[0.2, 0.2, 0.6])  # genotype length 0 (None), 1 or 2
    gt[ln == 0, 0] = 0xFF
    gt[ln <= 1, 1] = 0xFF
    if seed % 3 == 0:  # a later cell may be called after a missing first cell: still None
        gt[rng.random((V, S)) < 0.1, 0] = 0xFF
    n_bits = max(1, int(np.ceil(np.log2(max(len(np.unique(gt[gt != 0xFF])), 2)))))
    pl = _planes(gt, n_bits, True)
    d, c, _, _ = po.pairwise_differences(orc.Variants(np.arange(V, dtype=np.int64), gt), S)
    k = 0
    for i in range(S):
        for j in range(i + 1, S):
            comp = pl[0][:, i] & pl[0][:, j]
            x = np.zeros(V, dtype=bool)
            for q in pl[1:]:
                x |= q[:, i] ^ q[:, j]
            assert int(comp.sum()) == c[k]
            assert int((comp & x).sum()) == d[k]
            k += 1


def test_pairwise_differences_fails_loudly_without_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device is present")
    import ferromic_b200 as fm
    from ferromic_b200 import _lib
    with pytest.raises(fm.FerromicGpuError) as exc:
        fm.pairwise_differences(WORKED, 3)
    assert exc.value.code == _lib.FM_ERR_NO_DEVICE
    with pytest.raises(fm.FerromicGpuError) as exc:
        fm.pairwise_difference_arrays(WORKED, 3)
    assert exc.value.code == _lib.FM_ERR_NO_DEVICE
    # the entry point itself refuses before touching its arguments
    n = C.c_size_t()
    assert _lib.lib().fm_pairwise_differences(None, 3, None, None, None, None, 0, C.byref(n)) == _lib.FM_ERR_NO_DEVICE


def test_pairwise_argument_checks_need_no_device():
    import ferromic_b200 as fm
    with pytest.raises(ValueError):
        fm.pairwise_differences(WORKED, -1)
    assert fm.pairwise_differences(WORKED, 1) == []
    d, c = fm.pairwise_difference_arrays(WORKED, 0)
    assert d.size == 0 and c.size == 0
