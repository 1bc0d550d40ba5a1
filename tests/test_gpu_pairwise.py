"""GPU parity of pairwise_differences / fm_pairwise_differences (calculate_pairwise_differences,
stats.rs:4106-4231) against the oracle's direct loop: counts and positions exact, over tile and word edges of
the sample-pair bit-GEMM, every resident matrix form and the error paths."""
import ctypes as C

import numpy as np
import pytest

from oracle import pyoracle as orc
from tests import pairwise_oracle as po

pytestmark = pytest.mark.gpu


def _random_gt(rng, V, S, max_allele=1, p_none=0.1, p_haploid=0.1, values=None):
    """gt[V, S, 2] with the 0xFF sentinel: None, haploid and diploid genotypes at the same site."""
    pool = np.arange(max_allele + 1, dtype=np.uint8) if values is None else np.asarray(values, dtype=np.uint8)
    gt = pool[rng.integers(0, pool.size, size=(V, S, 2))]
    u = rng.random((V, S))
    gt[u < p_none, 0] = 0xFF
    gt[u < p_none + p_haploid, 1] = 0xFF
    return gt


def _check(gt, positions, sample_count, positions_too=True):
    import ferromic_b200 as fm
    from ferromic_b200.api import _Variants
    od, oc, os_, op = po.pairwise_differences(orc.Variants(positions, gt), sample_count)
    d, c = fm.pairwise_difference_arrays(_Variants(positions, gt), sample_count)
    assert np.array_equal(d, od) and np.array_equal(c, oc)
    if positions_too:
        got = fm.pairwise_differences(_Variants(positions, gt), sample_count)
        assert [g[1] for g in got] == od.tolist()
        flat = [p for g in got for p in g[2]]
        assert flat == op.tolist()
        assert [g[0] for g in got] == [(i, j) for i in range(sample_count) for j in range(i + 1, sample_count)]


def test_worked_example(both_ingest_modes):
    import ferromic_b200 as fm
    got = fm.pairwise_differences([(10, [[0, 0], [0, 1], [1, 1]]), (20, [[0, 0], [0, 0], [0, 1]]),
                                   (30, [[0, 1], None, [1, 0]])], 3)
    assert got == [((0, 1), 1, [10]), ((0, 2), 3, [10, 20, 30]), ((1, 2), 2, [10, 20])]
    d, c = fm.pairwise_difference_arrays([(10, [[0, 0], [0, 1], [1, 1]]), (20, [[0, 0], [0, 0], [0, 1]]),
                                          (30, [[0, 1], None, [1, 0]])], 3)
    assert d.tolist() == [1, 3, 2] and c.tolist() == [2, 3, 2]


@pytest.mark.parametrize("S", [1, 2, 31, 33, 130, 257])
@pytest.mark.parametrize("V", [0, 1, 31, 33, 1000])
def test_sample_and_site_edges(both_ingest_modes, S, V):
    rng = np.random.default_rng(S * 1000 + V)
    gt = _random_gt(rng, V, S)
    _check(gt, np.cumsum(rng.integers(1, 9, size=V)).astype(np.int64), S, positions_too=S <= 130)


@pytest.mark.parametrize("S", [33, 130])
def test_long_rows(both_ingest_modes, S):
    rng = np.random.default_rng(S)
    V = 70001
    gt = _random_gt(rng, V, S, p_none=0.02, p_haploid=0.02)
    _check(gt, np.arange(V, dtype=np.int64) * 2, S, positions_too=S == 33)


@pytest.mark.parametrize("max_allele,values", [(1, None), (3, None), (15, None),
                                                (0, [0, 1, 2, 5, 16, 17, 30, 64, 100, 128, 150, 180, 200, 220, 240, 254])])
def test_allele_ranges(max_allele, values):
    rng = np.random.default_rng(max_allele + 11)
    gt = _random_gt(rng, 400, 70, max_allele=max_allele, values=values)
    _check(gt, np.arange(400, dtype=np.int64) * 5, 70)


def test_no_missing_haploid_and_diploid_rows(both_ingest_modes):
    import ferromic_b200 as fm
    rng = np.random.default_rng(3)
    for ploidy in (1, 2):
        g = rng.integers(0, 2, size=(500, 67, ploidy)).astype(np.uint8)
        gt = np.full((500, 67, 2), 0xFF, dtype=np.uint8)
        gt[:, :, :ploidy] = g
        _check(gt, np.arange(500, dtype=np.int64), 67)
    # a sample count beyond the rows: the extra samples are None
    got = fm.pairwise_difference_arrays([(1, [[0, 1], [1, 1]]), (2, [[0, 0]])], 4)
    assert got[0].tolist() == [1, 0, 0, 0, 0, 0] and got[1].tolist() == [1, 0, 0, 0, 0, 0]


def test_ragged_python_rows(both_ingest_modes):
    import ferromic_b200 as fm
    rng = np.random.default_rng(5)
    rows = []
    for v in range(120):
        n = int(rng.integers(0, 40))
        row = []
        for _ in range(n):
            k = int(rng.integers(0, 4))
            row.append(None if k == 0 else [int(x) for x in rng.integers(0, 2, size=min(k, 2))])
        rows.append((v * 7, row))
    S = 45
    od, oc, os_, op = po.pairwise_differences(orc.variants_from_python(rows, n_samples=S), S)
    got = fm.pairwise_differences(rows, S)
    assert [g[1] for g in got] == od.tolist()
    assert [p for g in got for p in g[2]] == op.tolist()
    assert np.array_equal(fm.pairwise_difference_arrays(rows, S)[1], oc)


def _call(m_handle, n, diff, comp, start, pos, cap):
    from ferromic_b200 import _lib
    total = C.c_size_t()
    ptr = (lambda a: None if a is None else a.ctypes.data)
    st = _lib.lib().fm_pairwise_differences(m_handle, n, ptr(diff), ptr(comp), ptr(start), ptr(pos), cap,
                                            C.byref(total))
    return st, total.value


def test_inband_int8_matrix():
    from ferromic_b200.api import _Matrix
    rng = np.random.default_rng(9)
    V, S = 900, 77
    g = rng.integers(0, 4, size=(V, S, 2)).astype(np.int8)
    g[rng.random(g.shape) < 0.08] = -1
    pos = np.arange(V, dtype=np.int64) * 3
    m = _Matrix.from_int8(g, pos, 3, ingest="u8")
    gt = np.where(g < 0, 0xFF, g).astype(np.uint8)  # a genotype is the run of leading called cells
    od, oc, os_, op = po.pairwise_differences(orc.Variants(pos, gt), S)
    n_pairs = S * (S - 1) // 2
    diff, comp = np.zeros(n_pairs, np.uint32), np.zeros(n_pairs, np.uint32)
    start, out = np.zeros(n_pairs + 1, np.uint64), np.zeros(int(od.sum()), np.int64)
    st, total = _call(m.handle, S, diff, comp, start, out, out.size)
    assert st == 0 and total == int(od.sum())
    assert np.array_equal(diff, od) and np.array_equal(comp, oc)
    assert np.array_equal(start, os_) and np.array_equal(out, op)


def test_capacity_retry_and_errors():
    from ferromic_b200 import _lib
    from ferromic_b200.api import _Matrix, _sparse_matrix, _Variants
    rng = np.random.default_rng(1)
    gt = _random_gt(rng, 200, 40)
    pos = np.arange(200, dtype=np.int64)
    od, oc, os_, op = po.pairwise_differences(orc.Variants(pos, gt), 40)
    m = _sparse_matrix(_Variants(pos, gt), 40)
    n_pairs = 40 * 39 // 2
    diff, comp = np.zeros(n_pairs, np.uint32), np.zeros(n_pairs, np.uint32)
    start, out = np.zeros(n_pairs + 1, np.uint64), np.zeros(10, np.int64)
    st, total = _call(m.handle, 40, diff, comp, start, out, 10)
    assert st == _lib.FM_ERR_INVALID_ARG and total == int(od.sum())
    assert np.array_equal(diff, od) and np.array_equal(comp, oc) and np.array_equal(start, os_)
    # fewer samples than the matrix holds: the leading sub-triangle
    d20 = np.zeros(190, np.uint32)
    assert _call(m.handle, 20, d20, None, None, None, 0)[0] == 0
    assert np.array_equal(d20, po.pairwise_differences(orc.Variants(pos, gt), 20)[0])
    assert _call(m.handle, 41, d20, None, None, None, 0)[0] == _lib.FM_ERR_INVALID_ARG
    # a matrix streamed as u8 rows keeps no rows to transpose
    a = rng.integers(0, 2, size=(64, 40, 2)).astype(np.uint8)
    ms = _Matrix.ingest(a, None, pos[:64], [[(0, 0), (1, 0)]])
    assert _call(ms.handle, 40, diff, None, None, None, 0)[0] == _lib.FM_ERR_UNSUPPORTED


def test_ploidy_three_is_not_implemented():
    import ferromic_b200 as fm
    with pytest.raises(NotImplementedError):
        fm.pairwise_differences([(1, [[0, 1, 1], [0, 0, 1]])], 2)


def test_fullsize_synthetic_cohort():
    """2504 samples x 1e5 sites generated on the device (fm_synth_fill, 1 % missing); 64 pairs from every tile
    class (diagonal tiles, the last partial tile, off-diagonal tiles, the first and last pair) against the oracle
    over all sites."""
    import torch
    from ferromic_b200 import _lib
    L = _lib.lib()
    V, S = 100_000, 2504
    total = V * S * 2
    d_data = torch.empty(total, dtype=torch.uint8, device="cuda:0")
    d_miss = torch.empty((total + 63) // 64, dtype=torch.int64, device="cuda:0")
    _lib.check(L.fm_set_device(0))
    _lib.check(L.fm_synth_fill(d_data.data_ptr(), d_miss.data_ptr(), V, S, 2, 0, 4106, None, 0.05, 0.01))
    pos = np.arange(V, dtype=np.int64) * 10
    m = C.c_void_p()
    _lib.check(L.fm_matrix_create_device(d_data.data_ptr(), d_miss.data_ptr(), V, S, 2, 1, pos.ctypes.data,
                                         C.byref(m)))
    try:
        n_pairs = S * (S - 1) // 2
        diff, comp = np.zeros(n_pairs, np.uint32), np.zeros(n_pairs, np.uint32)
        st, _ = _call(m, S, diff, comp, None, None, 0)
        assert st == 0
        rng = np.random.default_rng(2504)
        pairs = [(0, 1), (S - 2, S - 1), (0, S - 1), (63, 64), (2496, 2503), (2440, 2500)]
        while len(pairs) < 64:
            i, j = sorted(int(x) for x in rng.choice(S, size=2, replace=False))
            if len(pairs) % 3 == 0:  # same 64-sample block: a diagonal tile
                b = i // 64
                i, j = b * 64 + int(rng.integers(0, 32)), b * 64 + int(rng.integers(32, 64))
                if j >= S:
                    continue
            pairs.append((i, j))
        cols = sorted({c for p in pairs for c in p})
        cidx = torch.tensor(cols, device="cuda:0")
        g = d_data.view(V, S, 2)[:, cidx, :]
        e = ((torch.arange(V, device="cuda:0")[:, None, None] * S + cidx[None, :, None]) * 2 +
             torch.arange(2, device="cuda:0")[None, None, :])
        miss = ((d_miss[e >> 6] >> (e & 63)) & 1).bool()
        gt = torch.where(miss, torch.full_like(g, 0xFF), g).cpu().numpy()
        where = {c: k for k, c in enumerate(cols)}
        for i, j in pairs:
            sub = np.ascontiguousarray(gt[:, [where[i], where[j]], :])
            od, oc, _, _ = po.pairwise_differences(orc.Variants(pos, sub), 2)
            k = i * (2 * S - i - 1) // 2 + j - i - 1
            assert (diff[k], comp[k]) == (od[0], oc[0]), (i, j)
    finally:
        L.fm_matrix_release(m)
