"""fm_per_site_diversity{,_multi} store the pi / theta tracks (and the positions of large calls) straight into the
caller's arrays when these are page-locked (csrc/fm_gpu.cu: mapped_host_range); pageable arrays take device buffers
+ copies.  Both routes must give the same bits -- and match the oracle -- for whole arrays, for rows at an offset
inside a page-locked buffer (capacity > n, second group), for mixed page-locked / pageable arguments, for the
single-group entry point and for the cached-counts route."""
import ctypes as C

import numpy as np
import pytest

from oracle import pyoracle as orc
from tests.synth import both_sides, make_cohort

pytestmark = pytest.mark.gpu


def _pinned(shape, dtype):
    import torch
    t = torch.empty(shape, dtype=dtype, pin_memory=True)
    t.fill_(-7)
    return t


def _multi(L, _lib, groups, raw_n, pos, mask, p_out, pi_out, th_out, cap):
    gh = (C.c_void_p * len(groups))(*[g.handle for g in groups])
    rn = (C.c_size_t * len(groups))(*raw_n)
    n = C.c_size_t()
    _lib.check(L.fm_per_site_diversity_multi(gh, rn, len(groups), int(pos[0]), int(pos[-1]), mask.ctypes.data,
                                             mask.size // 2, None, 0, p_out, pi_out, th_out, cap, C.byref(n)))
    return n.value


@pytest.mark.parametrize("V", [3000, 70000])   # above 65536 sites the positions are produced on the device too
def test_page_locked_outputs_equal_pageable_outputs_and_the_oracle(V):
    import torch
    from ferromic_b200 import _lib
    from ferromic_b200.api import _Matrix
    L = _lib.lib()
    g, pos, pops = make_cohort(V, 40, n_pops=2, missing_rate=0.03, seed=4242 + V)
    miss = g < 0
    alle = np.where(miss, 0, g).astype(np.uint8)
    h1, h2 = both_sides(pops[0]), both_sides(pops[1])
    mask = np.array([int(pos[50]), int(pos[90]), int(pos[V // 2]), int(pos[V // 2 + 500])], dtype=np.int64)
    cap = V + 13  # rows of the output arrays are `capacity` apart: the second group's row starts at an odd offset

    def run(pinned_pi, pinned_th, pinned_pos):
        m = _Matrix(alle, miss, pos, max_allele=1, always_bitmap=True, ingest="packed")  # fresh groups: plane pass
        groups = [m.group(h1), m.group(h2)]
        if pinned_pi:
            t_pi = _pinned((2, cap), torch.float64)
            pi, pi_ptr = t_pi.numpy(), t_pi.data_ptr()
        else:
            pi = np.full((2, cap), -7.0)
            pi_ptr = pi.ctypes.data
        if pinned_th:
            t_th = _pinned((2, cap), torch.float64)
            th, th_ptr = t_th.numpy(), t_th.data_ptr()
        else:
            th = np.full((2, cap), -7.0)
            th_ptr = th.ctypes.data
        if pinned_pos:
            t_p = _pinned((cap,), torch.int64)
            p, p_ptr = t_p.numpy(), t_p.data_ptr()
        else:
            p = np.full(cap, -7, dtype=np.int64)
            p_ptr = p.ctypes.data
        n = _multi(L, _lib, groups, (len(h1), len(h2)), pos, mask, p_ptr, pi_ptr, th_ptr, cap)
        assert n == V
        # nothing beyond the n values of each row may be touched
        assert np.all(pi[:, n:] == -7.0) and np.all(th[:, n:] == -7.0) and np.all(p[n:] == -7)
        return p[:n].copy(), pi[:, :n].copy(), th[:, :n].copy()

    ref = run(False, False, False)
    for combo in [(True, True, True), (True, True, False), (True, False, True), (False, True, False)]:
        got = run(*combo)
        assert np.array_equal(got[0], ref[0])
        for a, b in zip(got[1:], ref[1:]):
            assert np.array_equal(np.isnan(a), np.isnan(b))
            assert np.array_equal(a[~np.isnan(a)], b[~np.isnan(b)])
    # and the oracle (sparse semantics need whole-genotype missingness; the dense counts are what both routes use, so
    # compare through the count formulas of the oracle's per-site call on a cohort without half-missing calls)
    vs, d = orc.from_numpy(g, pos)
    for k, haps in enumerate((h1, h2)):
        rp, rpi, rth = orc.per_site_diversity(vs, haps, (int(pos[0]), int(pos[-1])),
                                              mask=[(int(mask[0]), int(mask[1])), (int(mask[2]), int(mask[3]))])
        assert np.array_equal(ref[0], rp)
        whole = ~(miss[:, :, 0] ^ miss[:, :, 1]).any(axis=1)  # sites where dense and sparse missingness agree
        a, b = ref[1][k][whole], rpi[whole]
        assert np.array_equal(np.isnan(a), np.isnan(b))
        ok = ~np.isnan(b)
        assert np.all(np.abs(a[ok] - b[ok]) <= 1e-9 * np.abs(b[ok]))


def test_bench_hook_hands_back_the_tracks_of_its_last_step():
    """fm_bench_diversity (mode 1, the timed loop of bench.py) copies the tracks of its last step into the caller's
    arrays, host or device (bench.py --dump-outputs): the same bits as fm_per_site_diversity_multi for the same groups
    and mask.  Mode 0 computes no tracks and refuses the arrays."""
    import torch
    from ferromic_b200 import _lib
    from ferromic_b200.api import _Matrix
    L = _lib.lib()
    V = 70000
    g, pos, pops = make_cohort(V, 40, n_pops=2, missing_rate=0.03, seed=2024)
    miss = g < 0
    alle = np.where(miss, 0, g).astype(np.uint8)
    h1, h2 = both_sides(pops[0]), both_sides(pops[1])
    mask = np.array([int(pos[50]), int(pos[90]), int(pos[V // 2]), int(pos[V // 2 + 500])], dtype=np.int64)
    m = _Matrix(alle, miss, pos, max_allele=1, always_bitmap=True, ingest="packed")
    groups = [m.group(h1), m.group(h2)]
    p, pi, th = np.empty(V, dtype=np.int64), np.empty((2, V)), np.empty((2, V))
    assert _multi(L, _lib, groups, (len(h1), len(h2)), pos, mask, p.ctypes.data, pi.ctypes.data, th.ctypes.data, V) == V
    gh = (C.c_void_p * 2)(*[x.handle for x in groups])
    h_pi, h_th = np.full((2, V), -7.0), np.full((2, V), -7.0)
    d_pi = torch.full((2, V), -7.0, dtype=torch.float64, device="cuda")
    d_th = torch.full_like(d_pi, -7.0)
    for pi_ptr, th_ptr in ((h_pi.ctypes.data, h_th.ctypes.data), (d_pi.data_ptr(), d_th.data_ptr())):
        _lib.check(L.fm_bench_diversity(gh, 2, 1, mask.ctypes.data, mask.size // 2, 3, None,
                                        C.byref(_lib.BenchResult()), pi_ptr, th_ptr))
    for got, ref in ((h_pi, pi), (h_th, th), (d_pi.cpu().numpy(), pi), (d_th.cpu().numpy(), th)):
        assert np.array_equal(np.isnan(got), np.isnan(ref))
        assert np.array_equal(got[~np.isnan(got)], ref[~np.isnan(ref)])
    with pytest.raises(ValueError):
        _lib.check(L.fm_bench_diversity(gh, 2, 0, None, 0, 1, None, C.byref(_lib.BenchResult()), h_pi.ctypes.data,
                                        None))


def test_single_group_call_and_cached_counts_route_with_page_locked_outputs():
    """fm_per_site_diversity (one group) forwards to the multi-group call; once the group's counts are cached the tracks
    come from the light kernel -- both must store into page-locked arrays like the plane pass does."""
    import torch
    from ferromic_b200 import _lib
    from ferromic_b200.api import _Matrix
    L = _lib.lib()
    V = 70000
    g, pos, pops = make_cohort(V, 24, n_pops=2, missing_rate=0.02, seed=99)
    miss = g < 0
    alle = np.where(miss, 0, g).astype(np.uint8)
    h1 = both_sides(pops[0])
    m = _Matrix(alle, miss, pos, max_allele=1, always_bitmap=True, ingest="packed")
    grp = m.group(h1)
    mask = np.array([int(pos[10]), int(pos[400])], dtype=np.int64)
    lo, hi = int(pos[1000]), int(pos[V - 7])   # a sub-range: outputs start at site 1000

    def call(p_ptr, pi_ptr, th_ptr, cap):
        n = C.c_size_t()
        _lib.check(L.fm_per_site_diversity(grp.handle, len(h1), lo, hi, mask.ctypes.data, 1, None, 0, p_ptr, pi_ptr, th_ptr,
                                           cap, C.byref(n)))
        return n.value

    p0, pi0, th0 = np.zeros(V, dtype=np.int64), np.zeros(V), np.zeros(V)
    n0 = call(p0.ctypes.data, pi0.ctypes.data, th0.ctypes.data, V)         # pageable, plane pass
    assert n0 == V - 7 - 1000 + 1
    for cached in (False, True):
        if cached:
            grp.summary()                                                  # caches the counts: light kernel from here on
        tp, tpi, tth = _pinned((V,), torch.int64), _pinned((V,), torch.float64), _pinned((V,), torch.float64)
        n1 = call(tp.data_ptr(), tpi.data_ptr(), tth.data_ptr(), V)
        assert n1 == n0
        assert np.array_equal(tp.numpy()[:n1], p0[:n0]) and p0[0] == pos[1000] + 1
        for a, b in ((tpi.numpy(), pi0), (tth.numpy(), th0)):
            assert np.array_equal(np.isnan(a[:n1]), np.isnan(b[:n0]))
            assert np.array_equal(a[:n1][~np.isnan(a[:n1])], b[:n0][~np.isnan(b[:n0])])
            assert np.all(a[n1:] == -7)
