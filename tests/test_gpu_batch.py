"""The segment table of the row pass (fm_k_plane_pass_seq) through its two entry points: fm_groups_summary_batch
(many (matrix, group) units in one launch -- the CLI's per-region loop, process.rs:2169) and the fused first call of
fm_hudson_pair (both groups' counts + Hudson partials from one sweep, stats.rs:3179-3278).  Everything must equal the one-at-a-time calls
bit for bit, and the oracle."""
import ctypes as C

import numpy as np
import pytest

from oracle import pyoracle as orc
from tests.synth import both_sides, make_cohort

pytestmark = pytest.mark.gpu


def _fresh(alle, miss, pos, ingest):
    from ferromic_b200.api import _Matrix
    return _Matrix(alle, miss, pos, max_allele=int(alle.max()), ingest=ingest)


@pytest.mark.parametrize("ingest", ["packed", "u8"])
def test_groups_summary_batch_equals_single_calls(ingest):
    from ferromic_b200 import _lib
    L = _lib.lib()
    rng = np.random.default_rng(42)
    specs = [(1000, 40, 0.1), (33, 40, 0.0), (4097, 17, 0.05), (1, 5, 0.0), (700, 300, 0.02), (2500, 64, 0.3)]
    mats, groups_a, groups_b, refs = [], [], [], []
    for k, (V, S, missing) in enumerate(specs):
        g, pos, _ = make_cohort(V, S, missing_rate=missing, seed=500 + k)
        miss = g < 0
        alle = np.where(miss, 0, g).astype(np.uint8)
        vs, d = orc.from_numpy(g, pos)
        for haps in (both_sides(range(S)), [(int(s), int(rng.integers(0, 2))) for s in range(0, S, 2)]):
            ma, mb = _fresh(alle, miss, pos, ingest), _fresh(alle, miss, pos, ingest)
            mats += [ma, mb]
            groups_a.append(ma.group(haps))
            groups_b.append(mb.group(haps))
            refs.append(orc.build_summary(d, haps))
    n = len(groups_a)
    # one group already has its summary cached, one appears twice in the list
    groups_a[3].summary()
    handles = [g.handle for g in groups_a] + [groups_a[0].handle]
    arr = (C.c_void_p * len(handles))(*[h.value for h in handles])
    seg = np.zeros(len(handles), dtype=np.uint64)
    unc = np.zeros(len(handles), dtype=np.uint64)
    pis = np.zeros(len(handles))
    _lib.check(L.fm_groups_summary_batch(arr, len(handles), seg.ctypes.data, pis.ctypes.data, unc.ctypes.data))
    assert seg[n] == seg[0] and pis[n] == pis[0] and unc[n] == unc[0]
    for i in range(n):
        one = groups_b[i].summary(want_arrays=True)          # the per-group call on an identical fresh group
        got = groups_a[i].summary(want_arrays=True)          # cached by the batch call
        assert int(seg[i]) == one["segregating_sites"] == got["segregating_sites"] == refs[i].seg
        assert int(unc[i]) == one["uncallable_lt2"] == got["uncallable_lt2"]
        assert pis[i] == one["pi_sum"] == got["pi_sum"]
        assert np.array_equal(got["alt"], refs[i].alt) and np.array_equal(got["called"], refs[i].called)
        assert np.array_equal(one["alt"], refs[i].alt)
    _lib.check(L.fm_groups_summary_batch(arr, 0, None, None, None))


def test_groups_summary_batch_mixed_classes():
    """No-bitmap and bitmap matrices, a multi-allelic one and an empty one in the same call."""
    from ferromic_b200 import _lib
    from ferromic_b200.api import _Matrix
    L = _lib.lib()
    g1, pos1, _ = make_cohort(900, 30, missing_rate=0.0, seed=1)
    g2, pos2, _ = make_cohort(1100, 30, missing_rate=0.2, seed=2)
    g3 = g1.copy()
    g3[5, 3, 0] = 2  # multi-allelic: no dense summary in the reference; the library keeps per-allele counts
    mats = [_Matrix(np.where(g < 0, 0, g).astype(np.uint8), g < 0, p) for g, p in ((g1, pos1), (g2, pos2), (g3, pos1))]
    mats.append(_Matrix(np.zeros((0, 30, 2), dtype=np.uint8), None, np.zeros(0, dtype=np.int64), max_allele=0))
    haps = both_sides(range(30))
    grp = [m.group(haps) for m in mats]
    arr = (C.c_void_p * 4)(*[g.handle.value for g in grp])
    seg = np.zeros(4, dtype=np.uint64)
    _lib.check(L.fm_groups_summary_batch(arr, 4, seg.ctypes.data, None, None))
    for i, (g, p) in enumerate(((g1, pos1), (g2, pos2))):
        _, d = orc.from_numpy(g, p)
        assert int(seg[i]) == orc.build_summary(d, haps).seg
    assert int(seg[3]) == 0
    fresh = _Matrix(np.where(g3 < 0, 0, g3).astype(np.uint8), g3 < 0, pos1).group(haps)
    assert int(seg[2]) == fresh.segregating_sites()


@pytest.mark.parametrize("ingest", ["packed", "u8"])
@pytest.mark.parametrize("missing", [0.0, 0.1])
def test_fused_hudson_first_call_equals_cached_path_and_oracle(ingest, missing):
    import ferromic_b200 as F
    from ferromic_b200 import _lib
    from ferromic_b200.api import _Matrix
    V, S = 5000, 90
    g, pos, pops = make_cohort(V, S, n_pops=2, missing_rate=missing, seed=77)
    miss = g < 0
    alle = np.where(miss, 0, g).astype(np.uint8)
    h1, h2 = both_sides(pops[0]), both_sides(pops[1])
    Lseq = int(pos[-1] - pos[0] + 1)
    vs, d = orc.from_numpy(g, pos)
    o1 = orc.Pop(h1, vs, S, Lseq, dense=d, summary=orc.build_summary(d, h1))
    o2 = orc.Pop(h2, vs, S, Lseq, dense=d, summary=orc.build_summary(d, h2))
    rc, ref, _ = orc.hudson_pair(o1, o2)
    L = _lib.lib()

    def call(m):
        a, b = m.group(h1), m.group(h2)
        out = _lib.HudsonOutcome()
        n = C.c_size_t()
        _lib.check(L.fm_hudson_pair(a.handle, b.handle, Lseq, Lseq, _lib.FM_HUDSON_SUMMARIES, 0, 0, 0, len(h1), len(h2),
                                    C.byref(out), None, C.byref(n)))
        return out, a, b

    m_fused = _Matrix(alle, miss, pos, max_allele=1, ingest=ingest)
    fused, fa, fb = call(m_fused)                       # nothing cached: one table pass does everything
    m_cached = _Matrix(alle, miss, pos, max_allele=1, ingest=ingest)
    m_cached.group(h1).summary()
    m_cached.group(h2).summary()                        # counts cached first: light kernel on the counts
    cached, _, _ = call(m_cached)
    for k in ("fst", "d_xy", "pi_pop1", "pi_pop2", "pi_xy_avg", "some"):
        assert getattr(fused, k) == getattr(cached, k), k
    for k in ("fst", "d_xy", "pi_pop1", "pi_pop2"):
        assert abs(getattr(fused, k) - ref[k]) <= 1e-9 * abs(ref[k])
    # the fused pass cached both groups' summaries exactly as fm_group_summary computes them
    for grp, haps in ((fa, h1), (fb, h2)):
        s = grp.summary(want_arrays=True)
        r = orc.build_summary(d, haps)
        assert np.array_equal(s["alt"], r.alt) and np.array_equal(s["called"], r.called)
        assert s["segregating_sites"] == r.seg


@pytest.mark.parametrize("ingest", ["packed-dense", "packed-sparse", "u8"])
def test_tail_word_plane_layout_group_sizes(ingest):
    """Groups whose size is a few haplotypes past a multiple of 128 keep only their full 16-byte words in the streamed
    plane; the rest of the row lives in per-site tail words (fm_kernels.cuh GroupPlanes).  Every size class -- no tail,
    1 / 2 / 3 tail words, a tail too long to pay, below one word -- must count exactly like the oracle, through the
    single-group pass, the multi-group launch, the fused Hudson sweep and the per-site tracks."""
    import ferromic_b200 as F
    from ferromic_b200 import _lib
    from ferromic_b200.api import _Matrix
    L = _lib.lib()
    S = 1800
    g, pos, _ = make_cohort(1300, S, missing_rate=0.02, seed=4242)
    miss = g < 0
    alle = np.where(miss, 0, g).astype(np.uint8)
    vs, d = orc.from_numpy(g, pos)
    rng = np.random.default_rng(9)
    all_haps = both_sides(range(S))
    sizes = [100, 128, 129, 160, 200, 224, 225, 256 + 33, 1545, 3463]
    lists = []
    for n in sizes:
        pick = np.sort(rng.choice(len(all_haps), n, replace=False))
        lists.append([all_haps[i] for i in pick])
    m = _Matrix(alle, miss, pos, max_allele=1, always_bitmap=True, ingest=ingest)
    groups = m.groups(lists)
    refs = [orc.build_summary(d, h) for h in lists]
    for grp, ref in zip(groups, refs):
        got = grp.summary(want_arrays=True)
        assert np.array_equal(got["alt"], ref.alt) and np.array_equal(got["called"], ref.called)
        assert got["segregating_sites"] == ref.seg
    # fused Hudson sweep on fresh groups of tail sizes (1545 vs 3463: the bench's orientation-group sizes)
    m2 = _Matrix(alle, miss, pos, max_allele=1, always_bitmap=True, ingest=ingest)
    a, b = m2.group(lists[-2]), m2.group(lists[-1])
    Lseq = int(pos[-1] - pos[0] + 1)
    out = _lib.HudsonOutcome()
    n = C.c_size_t()
    _lib.check(L.fm_hudson_pair(a.handle, b.handle, Lseq, Lseq, _lib.FM_HUDSON_SUMMARIES, 0, 0, 0, len(lists[-2]),
                                len(lists[-1]), C.byref(out), None, C.byref(n)))
    o1 = orc.Pop(lists[-2], vs, S, Lseq, dense=d, summary=refs[-2])
    o2 = orc.Pop(lists[-1], vs, S, Lseq, dense=d, summary=refs[-1])
    rc, ref, _ = orc.hudson_pair(o1, o2)
    for k in ("fst", "d_xy", "pi_pop1", "pi_pop2"):
        assert abs(getattr(out, k) - ref[k]) <= 1e-9 * abs(ref[k])
    for grp, r in ((a, refs[-2]), (b, refs[-1])):
        s = grp.summary(want_arrays=True)
        assert np.array_equal(s["alt"], r.alt) and np.array_equal(s["called"], r.called)
