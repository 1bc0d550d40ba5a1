"""GPU parity tests: the CUDA path (through the C-ABI library and the Python mirror) against the
CPU oracle on the same seeded inputs.  Integer outputs are compared bit-exactly; FP64 outputs
within REL (the north-star tolerance is 1e-9 relative; per-site values normally agree to the
last bit because the kernels keep the reference's operation order)."""
import math

import numpy as np
import pytest

from oracle import pyoracle as orc
from tests.synth import both_sides, make_cohort

pytestmark = [pytest.mark.gpu, pytest.mark.usefixtures("both_ingest_modes")]

REL = 1e-9


def fm():
    import ferromic_b200 as m
    return m


def close(a, b, rel=REL):
    if a is None or b is None:
        return a is None and b is None
    if isinstance(a, float) and math.isnan(a):
        return isinstance(b, float) and math.isnan(b)
    if math.isinf(a) or math.isinf(b):
        return a == b
    return abs(a - b) <= rel * max(abs(a), abs(b)) + 1e-300


def assert_arrays_close(a, b, rel=REL):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape
    assert np.array_equal(np.isnan(a), np.isnan(b)), "NaN/None pattern differs"
    m = ~np.isnan(a)
    assert np.all(np.abs(a[m] - b[m]) <= rel * np.maximum(np.abs(a[m]), np.abs(b[m])) + 1e-300)


def dense_pair(g, positions):
    """Oracle dense matrix + device matrix with from_numpy (dense) semantics."""
    from ferromic_b200.api import _Matrix
    vs, d = orc.from_numpy(g, positions)
    miss = (g < 0)
    alle = np.where(miss, 0, g).astype(np.uint8)
    m = _Matrix(alle, miss, positions, max_allele=d.max_allele)
    return vs, d, m


# ------------------------------------------------------------------ K1 + K2: counts / summary
@pytest.mark.parametrize("n_samples,missing", [(1, 0.0), (3, 0.2), (40, 0.1), (64, 0.0), (65, 0.05),
                                               (700, 0.02), (2504, 0.0), (2504, 0.01)])
def test_summary_matches_oracle(n_samples, missing):
    V = 4100 if n_samples < 1000 else 700
    g, pos, _ = make_cohort(V, n_samples, missing_rate=missing, seed=7 + n_samples)
    vs, d, m = dense_pair(g, pos)
    rng = np.random.default_rng(n_samples)
    groups = [both_sides(range(n_samples)),
              [(int(s), int(rng.integers(0, 2))) for s in rng.choice(n_samples, max(1, n_samples // 2), replace=False)],
              both_sides(range(n_samples))[::3] + [(0, 0), (0, 0), (n_samples + 5, 1)]]  # dups + out of range
    for haps in groups:
        ref = orc.build_summary(d, haps)
        got = m.group(haps).summary(want_arrays=True)
        assert np.array_equal(got["alt"], ref.alt)
        assert np.array_equal(got["called"], ref.called)
        assert got["segregating_sites"] == ref.seg
        assert got["uncallable_lt2"] == int((ref.called < 2).sum())
        assert close(got["pi_sum"], ref.pi_sum, 1e-12)
        assert m.group(haps).capacity == ref.capacity


def test_wide_rows_chunked_mode():
    # plane rows wider than two sites per warp ring take the column-chunked pass: 52000 samples (13 KB rows) stream a
    # whole row per stage, 60000 samples (15 KB rows) two column chunks per row
    from ferromic_b200.api import _Variants
    for n_samples in (52000, 60000):
        g, pos, _ = make_cohort(70, n_samples, missing_rate=0.01, seed=3)
        vs, d, m = dense_pair(g, pos)
        haps = both_sides(range(n_samples))
        ref = orc.build_summary(d, haps)
        got = m.group(haps).summary(want_arrays=True)
        assert np.array_equal(got["alt"], ref.alt) and np.array_equal(got["called"], ref.called)
        assert got["segregating_sites"] == ref.seg and close(got["pi_sum"], ref.pi_sum, 1e-12)
        # per-site pi / theta tracks of the chunked pass under a mask (sparse semantics: whole-sample missingness)
        gs = g.copy()
        gs[:, :, 1][gs[:, :, 0] < 0] = -1
        gs[:, :, 0][gs[:, :, 1] < 0] = -1
        svs, _ = orc.from_numpy(gs, pos)
        region = (int(pos[3]), int(pos[66]))
        mask = [(int(pos[10]), int(pos[20])), (int(pos[40]), int(pos[40]) + 1)]
        rp, rpi, rth = orc.per_site_diversity(svs, haps, region, mask=mask)
        gp, gpi, gth = fm().per_site_diversity_arrays(_Variants(svs.positions, svs.gt), haps, region, mask=mask)
        assert np.array_equal(gp, rp)
        assert np.isnan(gpi).sum() >= 10  # the masked sites
        assert_arrays_close(gpi, rpi, 1e-12)
        assert_arrays_close(gth, rth, 1e-12)


@pytest.mark.parametrize("missing", [0.0, 0.15])
def test_pi_paths_match_oracle(missing):
    g, pos, pops = make_cohort(3000, 30, missing_rate=missing, seed=11)
    vs, d, m = dense_pair(g, pos)
    L = int(pos[-1] - pos[0] + 1)
    from ferromic_b200 import _lib
    for haps in (both_sides(pops[0]), both_sides(range(30)), [(2, 0)], []):
        grp = m.group(haps)
        # summary path (lib.rs:777-789 -> stats.rs:1476-1542)
        summ = orc.build_summary(d, haps)
        ref = orc.pi_for_population(orc.Pop(haps, vs, 30, L, dense=d, summary=summ))
        assert close(grp.pi(L, _lib.FM_PI_SUMMARY), ref, 1e-12)
        # dense path (CLI contexts: process.rs:970-983 -> stats.rs:4534-4597)
        ref = orc.pi_for_population(orc.Pop(haps, vs, 30, L, dense=d))
        assert close(grp.pi(L, _lib.FM_PI_DENSE), ref, 1e-12)
    for Lx, exp in ((-5, 0.0), (0, math.inf)):
        assert m.group(both_sides(pops[0])).pi(Lx, _lib.FM_PI_SUMMARY) == exp


def test_population_api_matches_oracle_paths():
    F = fm()
    for missing in (0.0, 0.1):
        g, pos, pops = make_cohort(2500, 24, missing_rate=missing, seed=5)
        L = int(pos[-1] - pos[0] + 1)
        haps = both_sides(range(24))
        vs, d = orc.from_numpy(g, pos)
        pop = F.Population.from_numpy("all", g, pos, haps, L, sample_names=[f"s{i}" for i in range(24)])
        summ = orc.build_summary(d, haps)
        ref_pop = orc.Pop(haps, vs, 24, L, dense=d, summary=summ)
        assert pop.segregating_sites() == orc.count_segregating_sites_for_population(ref_pop)
        assert close(pop.nucleotide_diversity(), orc.pi_for_population(ref_pop), 1e-12)
        sub = pop.with_haplotypes("p1", both_sides(pops[0]))
        summ1 = orc.build_summary(d, both_sides(pops[0]))
        ref1 = orc.Pop(both_sides(pops[0]), vs, 24, L, dense=d, summary=summ1)
        assert sub.segregating_sites() == orc.count_segregating_sites_for_population(ref1)
        assert close(sub.nucleotide_diversity(), orc.pi_for_population(ref1), 1e-12)
        # sparse free functions
        variants = [{"position": int(p), "genotypes": [None if (row < 0).any() else row.tolist() for row in site]}
                    for p, site in zip(pos[:400], g[:400])]
        ovs = orc.variants_from_python(variants)
        assert F.segregating_sites(variants) == orc.count_segregating_sites(ovs)
        assert close(F.nucleotide_diversity(variants, both_sides(pops[1]), 1000),
                     orc.pi_sparse(ovs, both_sides(pops[1]), 1000), 1e-12)


# ------------------------------------------------------------------ per-site tracks
@pytest.mark.parametrize("missing", [0.0, 0.2])
def test_per_site_diversity_matches_oracle(missing):
    F = fm()
    g, pos, pops = make_cohort(5000, 20, missing_rate=missing, seed=21)
    g[:, :, 1][g[:, :, 0] < 0] = -1  # whole-sample missingness (sparse semantics)
    g[:, :, 0][g[:, :, 1] < 0] = -1
    vs, _ = orc.from_numpy(g, pos)
    from ferromic_b200.api import _Variants
    fvs = _Variants(vs.positions, vs.gt)
    haps = both_sides(pops[0]) + [(3, 0)]
    region = (int(pos[100]), int(pos[4700]))
    mask = [(int(pos[500]), int(pos[650])), (int(pos[600]), int(pos[700]) + 1), (int(pos[3000]), int(pos[3000]) + 1)]
    filtered = [int(pos[200]), int(pos[201]), int(pos[4000]), 123456789]
    for kw in (dict(), dict(mask=mask), dict(mask=mask, filtered_positions=filtered), dict(mask=[])):
        rp, rpi, rth = orc.per_site_diversity(vs, haps, region, filtered=kw.get("filtered_positions", ()),
                                              mask=kw.get("mask"))
        gp, gpi, gth = F.per_site_diversity_arrays(fvs, haps, region, **kw)
        assert np.array_equal(gp, rp)
        assert_arrays_close(gpi, rpi, 1e-12)
        assert_arrays_close(gth, rth, 1e-12)
    # region = None -> min..max positions; fewer than two haplotypes -> ValueError (lib.rs:1653)
    gp, _, _ = F.per_site_diversity_arrays(fvs, haps, None)
    assert len(gp) == 5000
    with pytest.raises(ValueError):
        F.per_site_diversity(fvs, [(0, 0)], region)
    assert len(F.per_site_diversity_arrays(fvs, haps, (10**12, 10**12 + 5))[0]) == 0


# ------------------------------------------------------------------ Hudson
def _outcome_close(got, ref):
    for k in ("fst", "d_xy", "pi_pop1", "pi_pop2", "pi_xy_avg"):
        assert close(getattr(got, k), ref[k], REL), (k, getattr(got, k), ref[k])


@pytest.mark.parametrize("missing", [0.0, 0.12])
def test_hudson_summaries_path(missing):
    F = fm()
    g, pos, pops = make_cohort(6000, 32, missing_rate=missing, seed=31)
    L = int(pos[-1] - pos[0] + 1)
    names = [f"s{i}" for i in range(32)]
    base = F.Population.from_numpy("all", g, pos, both_sides(range(32)), L, sample_names=names)
    p1 = base.with_haplotypes("p1", both_sides(pops[0]))
    p2 = base.with_haplotypes("p2", both_sides(pops[1]))
    vs, d = orc.from_numpy(g, pos)
    o1 = orc.Pop(both_sides(pops[0]), vs, 32, L, dense=d, summary=orc.build_summary(d, both_sides(pops[0])))
    o2 = orc.Pop(both_sides(pops[1]), vs, 32, L, dense=d, summary=orc.build_summary(d, both_sides(pops[1])))
    rc, ref, _ = orc.hudson_pair(o1, o2)
    assert rc == 0
    _outcome_close(F.hudson_fst(p1, p2), ref)
    rc, rd = orc.dxy_hudson(o1, o2)
    assert close(F.hudson_dxy(p1, p2).d_xy, rd)
    # with a region: per-site sparse values + FST, auxiliary pi/Dxy from the summaries (SURVEY app. 13)
    region = (int(pos[50]), int(pos[5000]))
    rc, ref, rsites = orc.hudson_pair(o1, o2, region=region)
    got, gsites = F.hudson_fst_with_sites(p1, p2, region)
    _outcome_close(got, ref)
    assert len(gsites) == len(rsites)
    for a, b in zip(gsites[::37], rsites[::37]):
        assert a.position == b["position"] and a.n1_called == b["n1_called"] and a.n2_called == b["n2_called"]
        for k in ("fst", "d_xy", "pi_pop1", "pi_pop2", "numerator_component", "denominator_component"):
            assert close(getattr(a, k), b[k], 1e-12), k


@pytest.mark.parametrize("missing", [0.0, 0.1])
def test_hudson_dense_and_sparse_paths_c_abi(missing):
    """CLI-style contexts (dense matrix, no summaries: process.rs:3191-3215) and sparse contexts."""
    import ctypes as C
    from ferromic_b200 import _lib
    g, pos, pops = make_cohort(3000, 16, missing_rate=missing, seed=41)
    g[:, :, 1][g[:, :, 0] < 0] = -1
    g[:, :, 0][g[:, :, 1] < 0] = -1
    vs, _ = orc.from_numpy(g, pos)
    d = orc.dense_from_variants(vs, 16)  # from_variants: bitmap always present
    from ferromic_b200.api import _Matrix
    m = _Matrix(np.where(g < 0, 0, g).astype(np.uint8), g < 0, pos, always_bitmap=True)
    L = int(pos[-1] - pos[0] + 1)
    h1, h2 = both_sides(pops[0]), both_sides(pops[1])
    g1, g2 = m.group(h1), m.group(h2)
    for path, o1, o2 in ((_lib.FM_HUDSON_DENSE, orc.Pop(h1, vs, 16, L, dense=d), orc.Pop(h2, vs, 16, L, dense=d)),
                         (_lib.FM_HUDSON_SPARSE, orc.Pop(h1, vs, 16, L), orc.Pop(h2, vs, 16, L))):
        for region in (None, (int(pos[10]), int(pos[2500]))):
            rc, ref, rsites = orc.hudson_pair(o1, o2, region=region)
            out = _lib.HudsonOutcome()
            V = len(pos)
            arrs = [np.zeros(V) for _ in range(6)]
            p_ = np.zeros(V, dtype=np.int64)
            n1 = np.zeros(V, dtype=np.uint32)
            n2 = np.zeros(V, dtype=np.uint32)
            hs = _lib.HudsonSites(*[a.ctypes.data for a in [p_] + arrs + [n1, n2]], V)
            n = C.c_size_t()
            rs, re = region if region else (0, 0)
            _lib.check(_lib.lib().fm_hudson_pair(g1.handle, g2.handle, L, L, path, int(region is not None), rs, re,
                                                 len(h1), len(h2), C.byref(out), C.byref(hs), C.byref(n)))
            for bit, k in enumerate(("fst", "d_xy", "pi_pop1", "pi_pop2", "pi_xy_avg")):
                got = getattr(out, k) if (out.some >> bit) & 1 else None
                assert close(got, ref[k]), (path, region, k, got, ref[k])
            assert n.value == len(rsites)
            k = n.value
            assert np.array_equal(p_[:k], [s["position"] for s in rsites])
            assert np.array_equal(n1[:k], [s["n1_called"] for s in rsites])
            for arr, key in zip(arrs, ("fst", "d_xy", "pi_pop1", "pi_pop2", "numerator_component",
                                       "denominator_component")):
                refv = np.array([np.nan if s[key] is None else s[key] for s in rsites])
                assert_arrays_close(arr[:k], refv, 1e-12)


def test_hudson_error_behaviour():
    F = fm()
    g, pos, pops = make_cohort(50, 8, seed=2)
    names = [f"s{i}" for i in range(8)]
    a = F.Population.from_numpy("a", g, pos, both_sides(pops[0]), 100, sample_names=names)
    b = F.Population.from_numpy("b", g, pos, both_sides(pops[1]), 200, sample_names=names)
    with pytest.raises(ValueError, match="Parse"):
        F.hudson_fst(a, b)  # sequence length mismatch (stats.rs:3445-3450)
    c = F.Population.from_numpy("c", g, pos + 1, both_sides(pops[1]), 100, sample_names=names)
    with pytest.raises(ValueError, match="Parse"):
        F.hudson_fst(a, c)  # incompatible variant positions (stats.rs:3451-3455)
    assert F.hudson_fst_sites(a, c, (0, 10**6)) == []  # stats.rs:3027-3034
    with pytest.raises(ValueError):
        F.Population("demo", [], [], 0)


# ------------------------------------------------------------------ windows (K5)
def test_window_sums_match_per_site_oracle():
    import ctypes as C
    from ferromic_b200 import _lib
    g, pos, pops = make_cohort(20000, 12, missing_rate=0.05, seed=51)
    vs, d, m = dense_pair(g, pos)
    h1, h2 = both_sides(pops[0]), both_sides(pops[1])
    g1, g2 = m.group(h1), m.group(h2)
    edges = np.arange(int(pos[0]), int(pos[-1]) + 1, 10_000)
    windows = np.array([(int(s), int(s) + 9_999) for s in edges], dtype=np.int64)
    nw = len(windows)
    nv = np.zeros(nw, dtype=np.uint64); seg = np.zeros(nw, dtype=np.uint64); unc = np.zeros(nw, dtype=np.uint64)
    pis = np.zeros(nw)
    _lib.check(_lib.lib().fm_group_window_sums(g1.handle, windows.ctypes.data, nw, nv.ctypes.data, seg.ctypes.data,
                                               pis.ctypes.data, unc.ctypes.data))
    s1, s2 = orc.build_summary(d, h1), orc.build_summary(d, h2)
    for w, (ws, we) in enumerate(windows):
        sel = (pos >= ws) & (pos <= we)
        a, c = s1.alt[sel].astype(np.int64), s1.called[sel].astype(np.int64)
        assert nv[w] == sel.sum()
        assert seg[w] == int(((c >= 2) & (a > 0) & (a < c)).sum())
        assert unc[w] == int((c < 2).sum())
        ok = c >= 2
        n = c[ok].astype(np.float64); al = a[ok].astype(np.float64); rf = n - al
        ref = float(np.sum(n / (n - 1.0) * (1.0 - (rf * rf + al * al) / (n * n))))
        assert close(float(pis[w]), ref, 1e-10)
    num = np.zeros(nw); den = np.zeros(nw); dxy = np.zeros(nw); p1 = np.zeros(nw); p2 = np.zeros(nw)
    sk = np.zeros(nw, dtype=np.uint64)
    _lib.check(_lib.lib().fm_hudson_window_sums(g1.handle, g2.handle, windows.ctypes.data, nw, num.ctypes.data,
                                                den.ctypes.data, dxy.ctypes.data, sk.ctypes.data, p1.ctypes.data,
                                                p2.ctypes.data))
    for w, (ws, we) in enumerate(windows[:6]):
        sel = np.nonzero((pos >= ws) & (pos <= we))[0]
        sub1 = orc.Summary(s1.alt[sel], s1.called[sel], s1.capacity, 0, 0.0)
        sub2 = orc.Summary(s2.alt[sel], s2.called[sel], s2.capacity, 0, 0.0)
        L = 10_000
        rc, ref, _ = orc.hudson_pair(orc.Pop(h1, None, 12, L, summary=sub1), orc.Pop(h2, None, 12, L, summary=sub2))
        fst = num[w] / den[w] if den[w] > 1e-12 else None
        assert close(fst, ref["fst"], 1e-10)


# ------------------------------------------------------------------ Weir & Cockerham (K4)
def _wc_compare(F, variants_py, vs, left, right, labels, region, rel=REL):
    G = len(labels)
    ref = orc.wc_fst(vs, left, right, G, region)
    got = F.wc_fst_from_membership(variants_py, labels, left, right, region)
    keys = [f"{labels[i]}_vs_{labels[j]}" for i in range(G) for j in range(i + 1, G)]
    # region: overall
    assert got.overall_fst.state == ref["overall"]["state"]
    assert got.overall_fst.sites == ref["overall"]["sites"]
    assert close(got.overall_fst.sum_a, ref["overall"]["sum_a"], rel)
    assert close(got.overall_fst.sum_b, ref["overall"]["sum_b"], rel)
    assert close(got.overall_fst.value, ref["overall"]["value"], rel)
    # region: pairs
    for k, key in enumerate(keys):
        if not ref["pair_present"][k]:
            assert key not in got.pairwise_fst
            continue
        e, r = got.pairwise_fst[key], ref["pairs"][k]
        assert e.state == r["state"] and e.sites == r["sites"], key
        assert close(e.sum_a, r["sum_a"], rel) and close(e.sum_b, r["sum_b"], rel), key
        assert close(e.value, r["value"], rel), key
        assert got.pairwise_variance_components[key] == (e.sum_a, e.sum_b)
    # per site
    assert len(got.site_fst) == ref["n_sites"]
    for i, s in enumerate(got.site_fst):
        assert s.position == ref["position"][i]
        assert s.overall_fst.state == orc.STATE_NAMES[ref["state"][i]]
        assert close(s.variance_components_a, float(ref["a"][i]), 1e-12)
        assert close(s.variance_components_b, float(ref["b"][i]), 1e-12)
        exp_sizes = {labels[g]: int(n) for g, n in enumerate(ref["pop_sizes"][i]) if n > 0} if ref["has_maps"][i] else {}
        assert s.population_sizes == exp_sizes
        if ref["has_maps"][i]:
            for k, key in enumerate(keys):
                st = ref["pair_state"][i][k]
                assert s.pairwise_fst[key].state == orc.STATE_NAMES[st]
                a, b = s.pairwise_variance_components[key]
                assert close(a, float(ref["pair_a"][i][k]), 1e-12) and close(b, float(ref["pair_b"][i][k]), 1e-12)
        else:
            assert s.pairwise_fst == {} and s.pairwise_variance_components == {}
    return got, ref


def _to_python_variants(g, pos):
    return [{"position": int(p), "genotypes": [None if (row < 0).any() else row.tolist() for row in site]}
            for p, site in zip(pos, g)]


@pytest.mark.parametrize("n_pops,missing", [(2, 0.0), (2, 0.3), (5, 0.15), (26, 0.02), (40, 0.05)])
def test_wc_fst_matches_oracle(n_pops, missing):
    # 40 populations = 780 pairs: three chunks of the pairs kernel's 352 pair slots per segment
    F = fm()
    S = 60 if n_pops < 26 else (130 if n_pops == 26 else 170)
    V = 900 if n_pops < 26 else 300
    g, pos, pops = make_cohort(V, S, n_pops=n_pops, sigma=0.08, missing_rate=missing, seed=100 + n_pops)
    g[:, :, 1][g[:, :, 0] < 0] = -1
    g[:, :, 0][g[:, :, 1] < 0] = -1
    g[5] = 0          # monomorphic site
    g[6] = -1         # no data at all -> InsufficientData (stats.rs:1987-2001)
    g[7, : S // 2] = -1  # data only in some populations
    rng = np.random.default_rng(n_pops)
    left = np.full(S, 0xFFFF, dtype=np.uint16)
    right = np.full(S, 0xFFFF, dtype=np.uint16)
    for p, members in enumerate(pops):
        left[members] = p
        right[members] = p
    # a few samples without a group (their alleles still count as "present", stats.rs:1826-1833)
    # and a few whose two haplotypes sit in different groups
    left[rng.choice(S, 3, replace=False)] = 0xFFFF
    swap = rng.choice(S, 4, replace=False)
    right[swap] = (right[swap] + 1) % n_pops
    labels = sorted(str(i) for i in range(n_pops))  # lexicographic label order (stats.rs:1105-1107)
    vs, _ = orc.from_numpy(g, pos)
    variants_py = _to_python_variants(g, pos)
    region = (int(pos[3]), int(pos[-10]))
    _wc_compare(F, variants_py, vs, left, right, labels, region)


def test_wc_fst_public_api_and_edge_cases():
    F = fm()
    names = ["s0", "s1", "s2", "s3"]
    variants = [{"position": 10, "genotypes": [[0, 0], [0, 1], [1, 1], [0, 1]]},
                {"position": 20, "genotypes": [[0, 1], [0, 1], [0, 1], [0, 1]]},
                {"position": 30, "genotypes": [None, None, None, None]},
                {"position": 40, "genotypes": [[0, 0], [0, 0], [1, 1], [1, 1]]}]
    groups = {"s0": (0, 0), "s1": (0, 0), "s2_L": (1, 1), "s3": (1, 1), "unknown": (1, 0)}
    res = F.wc_fst(variants, names, groups, (0, 100))
    assert res.fst_type == "haplotype_groups"
    assert len(res.site_fst) == 4 and [s.position for s in res.site_fst] == [11, 21, 31, 41]
    assert res.site_fst[0].variance_components() == pytest.approx((0.125, 0.5), abs=1e-12)   # SURVEY §8c KATs
    assert res.site_fst[1].variance_components() == pytest.approx((-1 / 6, 2 / 3), abs=1e-12)
    assert res.site_fst[2].overall_fst.state == "insufficient_data_for_estimation"
    assert res.site_fst[3].overall_fst.value == pytest.approx(1.0, abs=1e-12)
    assert res.overall_fst.sites == 3 and set(res.pairwise_fst) == {"0_vs_1"}
    a = 0.125 - 1 / 6 + 1.0
    b = 0.5 + 2 / 3 + 0.0
    assert res.overall_fst.sum_a == pytest.approx(a, rel=1e-12) and res.overall_fst.sum_b == pytest.approx(b, rel=1e-12)
    assert res.overall_fst.value == pytest.approx(a / (a + b), rel=1e-12)
    assert F.wc_fst_components(res.overall_fst) == res.overall_fst.components()
    # empty region -> InsufficientData{sites_attempted: 0} and no pair keys (stats.rs:2152-2159)
    res = F.wc_fst(variants, names, groups, (1000, 2000))
    assert res.overall_fst.state == "insufficient_data_for_estimation" and res.overall_fst.sites == 0
    assert res.pairwise_fst == {} and res.site_fst == []
    with pytest.raises(ValueError):
        F.wc_fst(variants, [], groups, (0, 100))
    with pytest.raises(ValueError):
        F.wc_fst(variants, names, groups, (10, 5))


# ------------------------------------------------------------------ streaming ingest (f1)
@pytest.mark.parametrize("chunk_rows,calls,missing", [(0, 1, 0.1), (37, 3, 0.1), (1, 2, 0.0), (5000, 1, 0.3)])
def test_streaming_ingest_equals_resident_matrix(chunk_rows, calls, missing):
    """fm_ingest_* (chunked upload overlapped with the repack, u8 never resident) must build the
    same bitplanes as fm_matrix_create + fm_group_create: identical counts, summaries and W&C."""
    import ctypes as C
    from ferromic_b200 import _lib
    from ferromic_b200.api import _Matrix
    g, pos, pops = make_cohort(1500, 45, n_pops=3, missing_rate=missing, seed=7 + chunk_rows)
    miss = g < 0
    alle = np.where(miss, 0, g).astype(np.uint8)
    hap_lists = [both_sides(pops[0]), both_sides(pops[1]) + [(pops[2][0], 1)], [(s, 0) for s in pops[2]]]
    left = np.full(45, 0xFFFF, dtype=np.uint16)
    for p, members in enumerate(pops):
        left[members] = p
    resident = _Matrix(alle, miss, pos, max_allele=1)
    streamed = _Matrix.ingest(alle, miss, pos, hap_lists, partitions=[(left, left, 3)], chunk_rows=chunk_rows,
                              calls=calls)
    for haps in hap_lists:
        a, b = resident.group(haps).summary(True), streamed.group(haps).summary(True)
        assert np.array_equal(a["alt"], b["alt"]) and np.array_equal(a["called"], b["called"])
        assert a["segregating_sites"] == b["segregating_sites"] and a["pi_sum"] == b["pi_sum"]
        assert a["uncallable_lt2"] == b["uncallable_lt2"]
    # oracle cross-check of one group
    vs, d = orc.from_numpy(g, pos)
    s0 = orc.build_summary(d, hap_lists[0])
    got = streamed.group(hap_lists[0]).summary(True)
    assert np.array_equal(got["alt"], s0.alt) and np.array_equal(got["called"], s0.called)
    # the partition declared at ingest time gives the same W&C totals as one built afterwards
    L = _lib.lib()
    ph = C.c_void_p()
    _lib.check(L.fm_partition_create(resident.handle, left.ctypes.data, left.ctypes.data, 45, 3, C.byref(ph)))
    w = np.array([int(pos[0]), int(pos[-1])], dtype=np.int64)

    def totals(handle):
        oa, ob = np.zeros(1), np.zeros(1)
        pa, pb = np.zeros(3), np.zeros(3)
        pn, osz, nv = np.zeros(3, dtype=np.uint64), np.zeros(1, dtype=np.uint64), np.zeros(1, dtype=np.uint64)
        _lib.check(L.fm_wc_window_sums(handle, w.ctypes.data, 1, nv.ctypes.data, oa.ctypes.data, ob.ctypes.data,
                                       osz.ctypes.data, pa.ctypes.data, pb.ctypes.data, pn.ctypes.data))
        return (oa[0], ob[0], int(osz[0]), pa.tolist(), pb.tolist(), pn.tolist())

    assert totals(ph) == totals(streamed.partitions[0])
    L.fm_partition_release(ph)
    # a streamed matrix has no resident u8 rows: late group creation must fail loudly
    with pytest.raises(NotImplementedError):
        streamed.group([(0, 0), (1, 1)])


# ------------------------------------------------------------------ multi-allelic sites (general paths)
def make_multi_cohort(V, S, max_allele, missing, seed):
    rng = np.random.default_rng(seed)
    A = max_allele + 1
    w = rng.dirichlet(np.full(A, 0.6), size=V)                       # per-site allele frequencies
    cdf = np.cumsum(w, axis=1)
    u = rng.random((V, S, 2))
    g = (u[..., None] > cdf[:, None, None, :]).sum(axis=3).clip(0, max_allele).astype(np.int8)
    g[0] = 0                                                          # monomorphic
    g[1, :, :] = np.arange(S * 2).reshape(S, 2) % A                   # every allele present
    if missing > 0:
        g[rng.random(g.shape) < missing] = -1
    g[2] = -1                                                         # no data
    g[3, 1:, :] = -1                                                  # a single called sample
    g[4].flat[0] = max_allele                                         # make sure max_allele is reached
    pos = np.cumsum(rng.integers(1, 40, size=V, dtype=np.int64))
    return g, pos


@pytest.mark.parametrize("max_allele,missing", [(2, 0.0), (3, 0.12), (7, 0.05), (15, 0.1)])
def test_multi_allelic_dense_population_paths(max_allele, missing):
    """Population.from_numpy with max_allele > 1: the reference builds no summary (lib.rs:779) and takes
    count_segregating_sites_dense / calculate_pi_dense / dense_hudson_sites_general / calculate_dxy_dense."""
    F = fm()
    S = 22
    g, pos = make_multi_cohort(700, S, max_allele, missing, seed=90 + max_allele)
    L = int(pos[-1] - pos[0] + 1)
    names = [f"s{i}" for i in range(S)]
    h1 = both_sides(range(0, S // 2)) + [(S - 1, 0)]
    h2 = both_sides(range(S // 2, S - 1)) + [(S - 1, 1), (S // 2, 0)]  # one duplicate
    base = F.Population.from_numpy("all", g, pos, h1 + h2, L, sample_names=names)
    p1, p2 = base.with_haplotypes("p1", h1), base.with_haplotypes("p2", h2)
    vs, d = orc.from_numpy(g, pos)
    assert d.max_allele == max_allele
    o1 = orc.Pop(h1, vs, S, L, dense=d)
    o2 = orc.Pop(h2, vs, S, L, dense=d)
    assert p1.segregating_sites() == orc.count_segregating_sites_for_population(o1)
    assert p2.segregating_sites() == orc.count_segregating_sites_for_population(o2)
    assert close(p1.nucleotide_diversity(), orc.pi_for_population(o1))
    assert close(p2.nucleotide_diversity(), orc.pi_for_population(o2))
    rc, ref, _ = orc.hudson_pair(o1, o2)
    got = F.hudson_fst(p1, p2)
    assert rc == 0
    for k in ("fst", "d_xy", "pi_pop1", "pi_pop2", "pi_xy_avg"):
        assert close(getattr(got, k), ref[k]), k
    assert close(F.hudson_dxy(p1, p2).d_xy, orc.dxy_hudson(o1, o2)[1])
    # region => sparse per-site values + dense auxiliary pi / Dxy (stats.rs:3473-3475, 3562-3565)
    region = (int(pos[5]), int(pos[-7]))
    rc, ref, rsites = orc.hudson_pair(o1, o2, region=region)
    out, sites = F.hudson_fst_with_sites(p1, p2, region)
    assert rc == 0 and len(sites) == len(rsites)
    for k in ("fst", "d_xy", "pi_pop1", "pi_pop2", "pi_xy_avg"):
        assert close(getattr(out, k), ref[k]), k
    for s, r in zip(sites, rsites):
        assert s.position == r["position"] and s.n1_called == r["n1_called"] and s.n2_called == r["n2_called"]
        for a in ("fst", "d_xy", "pi_pop1", "pi_pop2", "numerator_component", "denominator_component"):
            assert close(getattr(s, a), r[a], 1e-12), (s.position, a)


@pytest.mark.parametrize("values,missing", [([0, 3, 17, 40, 200, 254], 0.1), ([0, 16], 0.0), ([0, 1, 2, 250], 0.05),
                                            (list(range(0, 160, 10)), 0.02)])
def test_allele_values_above_15_are_remapped(values, missing):
    """Allele indices up to 254 (stats.rs:4573-4589 counts in 256 bins): the GPU path bit-slices at most 4 bits per cell,
    so a matrix whose max_allele exceeds 15 has its DISTINCT values (up to 16, 0 always among them) mapped to ranks in
    ascending order before K1 -- the estimators only depend on allele identity and ascending order.  Dense population
    paths against the oracle on the original values."""
    F = fm()
    S = 22
    k = len(values) - 1
    g0, pos = make_multi_cohort(600, S, k, missing, seed=700 + k)
    lut = np.asarray(values, dtype=np.int16)
    g = np.where(g0 < 0, np.int16(-1), lut[np.clip(g0, 0, k)]).astype(np.int16)
    L = int(pos[-1] - pos[0] + 1)
    names = [f"s{i}" for i in range(S)]
    h1 = both_sides(range(0, S // 2)) + [(S - 1, 0)]
    h2 = both_sides(range(S // 2, S - 1)) + [(S - 1, 1)]
    base = F.Population.from_numpy("all", g, pos, h1 + h2, L, sample_names=names)
    p1, p2 = base.with_haplotypes("p1", h1), base.with_haplotypes("p2", h2)
    vs, d = orc.from_numpy(g, pos)
    assert d.max_allele == max(values)
    o1 = orc.Pop(h1, vs, S, L, dense=d)
    o2 = orc.Pop(h2, vs, S, L, dense=d)
    assert p1.segregating_sites() == orc.count_segregating_sites_for_population(o1)
    assert p2.segregating_sites() == orc.count_segregating_sites_for_population(o2)
    assert close(p1.nucleotide_diversity(), orc.pi_for_population(o1))
    rc, ref, _ = orc.hudson_pair(o1, o2)
    got = F.hudson_fst(p1, p2)
    assert rc == 0
    for key in ("fst", "d_xy", "pi_pop1", "pi_pop2", "pi_xy_avg"):
        assert close(getattr(got, key), ref[key]), key
    region = (int(pos[5]), int(pos[-7]))
    rc, ref, rsites = orc.hudson_pair(o1, o2, region=region)
    out, sites = F.hudson_fst_with_sites(p1, p2, region)
    assert rc == 0 and len(sites) == len(rsites)
    for s_, r in zip(sites, rsites):
        for a in ("fst", "d_xy", "pi_pop1", "pi_pop2"):
            assert close(getattr(s_, a), r[a], 1e-12), (s_.position, a)


def test_more_than_16_distinct_allele_values_fail_loudly():
    F = fm()
    S = 12
    rng = np.random.default_rng(1)
    g = rng.integers(0, 40, size=(50, S, 2)).astype(np.int16)  # 40 distinct values
    pos = np.arange(50, dtype=np.int64) * 7
    haps = both_sides(range(S))
    base = F.Population.from_numpy("all", g, pos, haps, 400, sample_names=[f"s{i}" for i in range(S)])
    with pytest.raises(NotImplementedError):
        base.segregating_sites()


@pytest.mark.parametrize("max_allele", [2, 5])
def test_multi_allelic_sparse_paths(max_allele):
    """Variant-list inputs (no dense matrix): calculate_pi, per-site diversity, cohort segregating sites and
    the sparse Hudson path on multi-allelic sites, incl. the reference's tri-allelic golden."""
    F = fm()
    S = 14
    g, pos = make_multi_cohort(300, S, max_allele, 0.1, seed=5 + max_allele)
    g[:, :, 1][g[:, :, 0] < 0] = -1
    g[:, :, 0][g[:, :, 1] < 0] = -1
    L = int(pos[-1] - pos[0] + 1)
    variants = _to_python_variants(g, pos)
    vs = orc.variants_from_python(variants, S)
    haps = both_sides(range(0, 9)) + [(9, 0)]
    assert F.segregating_sites(variants) == orc.count_segregating_sites(vs)
    assert close(F.nucleotide_diversity(variants, haps, L), orc.pi_sparse(vs, haps, L))
    region = (int(pos[2]), int(pos[-3]))
    gp, gpi, gth = F.per_site_diversity_arrays(variants, haps, region, mask=[(int(pos[50]), int(pos[60]))])
    rp, rpi, rth = orc.per_site_diversity(vs, haps, region, mask=[(int(pos[50]), int(pos[60]))])
    assert np.array_equal(gp, rp)
    assert_arrays_close(gpi, rpi, 1e-12)
    assert_arrays_close(gth, rth, 1e-12)
    names = [f"s{i}" for i in range(S)]
    h1, h2 = both_sides(range(0, 7)), both_sides(range(7, S))
    d1 = {"id": 0, "haplotypes": h1, "variants": variants, "sequence_length": L, "sample_names": names}
    d2 = {"id": 1, "haplotypes": h2, "variants": variants, "sequence_length": L, "sample_names": names}
    o1, o2 = orc.Pop(h1, vs, S, L), orc.Pop(h2, vs, S, L)
    rc, ref, _ = orc.hudson_pair(o1, o2)
    got = F.hudson_fst(d1, d2)
    for k in ("fst", "d_xy", "pi_pop1", "pi_pop2"):
        assert close(getattr(got, k), ref[k]), k
    # tests/hudson_fst_tests.rs:877-1006
    tri = [{"position": 100, "genotypes": [[0, 0], [1, 2], [0, 1], [2, 2]]}]
    a = {"id": 0, "haplotypes": both_sides([0, 1]), "variants": tri, "sequence_length": 1, "sample_names": names[:4]}
    b = {"id": 1, "haplotypes": both_sides([2, 3]), "variants": tri, "sequence_length": 1, "sample_names": names[:4]}
    _, sites = F.hudson_fst_with_sites(a, b, (100, 100))
    exp_pi = (4.0 / 3.0) * 0.625
    assert abs(sites[0].d_xy - 0.6875) < 1e-12 and abs(sites[0].pi_pop1 - exp_pi) < 1e-12
    assert abs(sites[0].fst - (0.6875 - exp_pi) / 0.6875) < 1e-12


def test_multi_allelic_unsupported_corners_fail_loudly():
    F = fm()
    g, pos = make_multi_cohort(50, 6, 20, 0.0, seed=1)  # allele index 20 > 15
    with pytest.raises(NotImplementedError):
        F.Population.from_numpy("x", g, pos, both_sides(range(6)), 100).segregating_sites()


@pytest.mark.parametrize("max_allele,n_pops", [(2, 2), (3, 4), (9, 3)])
def test_wc_fst_multi_allelic_matches_oracle(max_allele, n_pops):
    """W&C sums over EVERY allele present at a site (stats.rs:1849-1859): multi-allelic K4 variant."""
    F = fm()
    S = 36
    g, pos = make_multi_cohort(500, S, max_allele, 0.08, seed=31 + max_allele)
    g[:, :, 1][g[:, :, 0] < 0] = -1
    g[:, :, 0][g[:, :, 1] < 0] = -1
    bounds = np.linspace(0, S, n_pops + 1).astype(int)
    left = np.full(S, 0xFFFF, dtype=np.uint16)
    for p in range(n_pops):
        left[bounds[p]:bounds[p + 1]] = p
    right = left.copy()
    left[3] = 0xFFFF                      # a haplotype without a group still defines "alleles present"
    right[5] = (right[5] + 1) % n_pops
    labels = sorted(str(i) for i in range(n_pops))
    vs, _ = orc.from_numpy(g, pos)
    _wc_compare(F, _to_python_variants(g, pos), vs, left, right, labels, (int(pos[1]), int(pos[-2])))


# ------------------------------------------------------------------ in-band missingness (int8 cells < 0)
@pytest.mark.parametrize("max_allele", [1, 3])
def test_inband_missing_equals_bitmap(max_allele):
    """FM_MISSING_IN_BAND / fm_matrix_create_inband: the int8 array as the caller holds it (negative =
    missing) must give the same planes and counts as the converted u8 matrix + packed bitmap."""
    import ctypes as C
    from ferromic_b200 import _lib
    from ferromic_b200.api import _Matrix
    if max_allele == 1:
        g, pos, pops = make_cohort(2100, 37, n_pops=3, missing_rate=0.15, seed=77)
    else:
        g, pos = make_multi_cohort(900, 37, max_allele, 0.15, seed=78)
        pops = [list(range(0, 12)), list(range(12, 25)), list(range(25, 37))]
    miss = g < 0
    alle = np.where(miss, 0, g).astype(np.uint8)
    haps = [both_sides(pops[0]), both_sides(pops[1]) + [(pops[2][0], 1)], [(s, 1) for s in pops[2]]]
    bitmap = _Matrix(alle, miss, pos, max_allele=max_allele)
    inband = _Matrix.from_int8(g.astype(np.int8), pos, max_allele)
    for h in haps:
        a, b = bitmap.group(h), inband.group(h)
        if max_allele == 1:
            sa, sb = a.summary(True), b.summary(True)
            assert np.array_equal(sa["alt"], sb["alt"]) and np.array_equal(sa["called"], sb["called"])
            assert sa["pi_sum"] == sb["pi_sum"] and sa["segregating_sites"] == sb["segregating_sites"]
        else:
            assert a.segregating_sites() == b.segregating_sites()
            assert a.pi(5000, _lib.FM_PI_DENSE) == b.pi(5000, _lib.FM_PI_DENSE)
    if max_allele == 1:  # count-only partition groups (full-row bit words) and the streaming ingest
        left = np.full(37, 0xFFFF, dtype=np.uint16)
        for p, members in enumerate(pops):
            left[members] = p
        L = _lib.lib()
        w = np.array([int(pos[0]), int(pos[-1])], dtype=np.int64)

        def totals(m):
            ph = C.c_void_p()
            _lib.check(L.fm_partition_create(m.handle, left.ctypes.data, left.ctypes.data, 37, 3, C.byref(ph)))
            oa, ob = np.zeros(1), np.zeros(1)
            pa, pb = np.zeros(3), np.zeros(3)
            pn, osz, nv = np.zeros(3, dtype=np.uint64), np.zeros(1, dtype=np.uint64), np.zeros(1, dtype=np.uint64)
            _lib.check(L.fm_wc_window_sums(ph, w.ctypes.data, 1, nv.ctypes.data, oa.ctypes.data, ob.ctypes.data,
                                           osz.ctypes.data, pa.ctypes.data, pb.ctypes.data, pn.ctypes.data))
            L.fm_partition_release(ph)
            return (oa[0], ob[0], int(osz[0]), pa.tolist(), pb.tolist(), pn.tolist())

        assert totals(bitmap) == totals(inband)
        ih = C.c_void_p()
        g8 = np.ascontiguousarray(g.astype(np.int8))
        _lib.check(L.fm_ingest_begin(g.shape[0], 37, 2, 2, 1, pos.ctypes.data, 100, C.byref(ih)))  # FM_MISSING_IN_BAND
        idx = np.asarray([h[0] for h in haps[0]], dtype=np.uint64)
        side = np.asarray([h[1] for h in haps[0]], dtype=np.uint8)
        _lib.check(L.fm_ingest_add_group(ih, idx.ctypes.data, side.ctypes.data, len(idx), None))
        _lib.check(L.fm_ingest_rows(ih, g8.ctypes.data, None, 0, g.shape[0]))
        mh, gh = C.c_void_p(), (C.c_void_p * 1)()
        _lib.check(L.fm_ingest_finish(ih, C.byref(mh), gh, None))
        alt = np.zeros(g.shape[0], dtype=np.uint32)
        cnt = np.zeros(g.shape[0], dtype=np.uint32)
        seg, unc, pis = C.c_uint64(), C.c_uint64(), C.c_double()
        _lib.check(L.fm_group_summary(C.c_void_p(gh[0]), alt.ctypes.data, cnt.ctypes.data, C.byref(seg), C.byref(pis),
                                      C.byref(unc)))
        ref = bitmap.group(haps[0]).summary(True)
        assert np.array_equal(alt, ref["alt"]) and np.array_equal(cnt, ref["called"]) and pis.value == ref["pi_sum"]
        L.fm_group_release(C.c_void_p(gh[0]))
        L.fm_matrix_release(mh)


# ------------------------------------------------------------------ several groups in one launch
@pytest.mark.parametrize("S,missing,n_groups", [(40, 0.1, 2), (700, 0.02, 3), (2504, 0.01, 2), (300, 0.0, 4),
                                                (700, 0.02, 6)])
def test_per_site_diversity_multi_equals_per_group_calls(S, missing, n_groups):
    """fm_per_site_diversity_multi streams every group's planes in ONE persistent launch
    (fm_k_plane_pass_seq; more than four groups read their segment table from device memory); per-site values
    must equal the per-group calls bit for bit."""
    import ctypes as C
    from ferromic_b200 import _lib
    from ferromic_b200.api import _Matrix
    V = 3000 if S < 1000 else 900
    g, pos, _ = make_cohort(V, S, missing_rate=missing, seed=S + n_groups)
    miss = g < 0
    alle = np.where(miss, 0, g).astype(np.uint8)
    rng = np.random.default_rng(S)
    lab = rng.integers(0, n_groups, size=(S, 2))
    lab[: max(2, S // 20), :] = 0          # group 0 is never tiny
    hap_lists = [[(s, k) for s in range(S) for k in (0, 1) if lab[s, k] == gi] for gi in range(n_groups)]
    hap_lists[-1] = hap_lists[-1][: max(1, len(hap_lists[-1]) // 7)]  # a much narrower group (different row width)
    region = (int(pos[37]), int(pos[-41]))
    mask = np.array([[int(pos[100]), int(pos[180])], [int(pos[500]), int(pos[505])]], dtype=np.int64)
    L = _lib.lib()
    per_group = []
    m1 = _Matrix(alle, miss, pos, max_allele=1)
    for haps in hap_lists:
        grp = m1.group(haps)
        pp = np.zeros(V, dtype=np.int64)
        pi, th = np.zeros(V), np.zeros(V)
        n = C.c_size_t()
        _lib.check(L.fm_per_site_diversity(grp.handle, len(haps), region[0], region[1], mask.ctypes.data, len(mask), None,
                                           0, pp.ctypes.data, pi.ctypes.data, th.ctypes.data, V, C.byref(n)))
        per_group.append((pp[:n.value].copy(), pi[:n.value].copy(), th[:n.value].copy()))
    m2 = _Matrix(alle, miss, pos, max_allele=1)  # fresh groups: nothing cached, the fused launch is taken
    groups = [m2.group(h) for h in hap_lists]
    arr = (C.c_void_p * n_groups)(*[g_.handle.value for g_ in groups])
    raw = (C.c_size_t * n_groups)(*[len(h) for h in hap_lists])
    pp = np.zeros(V, dtype=np.int64)
    pi, th = np.zeros((n_groups, V)), np.zeros((n_groups, V))
    n = C.c_size_t()
    L.fm_timings_reset()
    _lib.check(L.fm_per_site_diversity_multi(arr, raw, n_groups, region[0], region[1], mask.ctypes.data, len(mask), None, 0,
                                             pp.ctypes.data, pi.ctypes.data, th.ctypes.data, V, C.byref(n)))
    tim = _lib.Timings()
    L.fm_timings_get(C.byref(tim))
    assert tim.stats_launches == 1, "the groups were expected to share one plane-pass launch"
    for gi in range(n_groups):
        rp, rpi, rth = per_group[gi]
        assert n.value == len(rp) and np.array_equal(pp[:n.value], rp)
        if len(hap_lists[gi]) < 2:
            assert np.isnan(pi[gi, :n.value]).all()
            continue
        assert np.array_equal(pi[gi, :n.value], rpi, equal_nan=True)
        assert np.array_equal(th[gi, :n.value], rth, equal_nan=True)
