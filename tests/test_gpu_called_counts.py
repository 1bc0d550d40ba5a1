"""Biallelic groups of a matrix with missing data keep the called count of every site (written by K1 when the rows
are repacked) instead of a called bitplane.  Right after a group is created, fm_group_summary's `called` array must
equal the oracle's build_summary(...).called, and the per-site pi / theta tracks of the plane pass that reads those
counts must match the oracle -- for every way a group comes to exist: u8 + bitmap (staged and direct rows), in-band
int8, packed rows with a called plane, packed rows with a sparse missing list (u16 columns and gap codes), streaming
ingest in several chunks with and without tracks requested at ingest time, rows wider than a warp slice and the VCF
packed batch."""
import ctypes as C

import numpy as np
import pytest

from oracle import pyoracle as orc
from tests.synth import both_sides, make_cohort

pytestmark = pytest.mark.gpu


def _cohort(V, S, seed, missing=0.03):
    g, pos, _ = make_cohort(V, S, missing_rate=missing, seed=seed)
    # whole genotypes are missing: the dense matrix then carries exactly the missingness the oracle's per-site
    # function (variant semantics: a genotype with a missing allele is None) sees
    g[(g < 0).any(axis=2)] = -1
    g[7] = -1  # a row without any call
    return g, pos


def _hap_lists(S):
    """Group sizes with n % 128 == 0, in 1..96 (tail words) and in 97..127 (padded rows), plus a group with
    duplicate haplotypes."""
    k = 119 if S >= 119 else 55  # 238 = 128 + 110 haplotypes (padded rows) or 110 (one padded word)
    return [both_sides(range(64)),                       # 128 haplotypes
            both_sides(range(84)),                       # 168 = 128 + 40: tail words
            both_sides(range(S - k, S)),
            both_sides(range(0, S, 2)) + [(0, 0), (2, 1), (0, 0)]]  # duplicates


def _tracks_match(group, haps, vs, pos, lo):
    """per-site tracks of the group over [pos[lo], pos[-1]] (a range that starts mid-batch) against the oracle"""
    from ferromic_b200 import _lib
    L = _lib.lib()
    region = (int(pos[lo]), int(pos[-1]))
    cap = len(pos)
    p = np.zeros(cap, dtype=np.int64)
    pi, th = np.zeros(cap), np.zeros(cap)
    n = C.c_size_t()
    _lib.check(L.fm_per_site_diversity(group.handle, len(haps), region[0], region[1], None, 0, None, 0, p.ctypes.data,
                                       pi.ctypes.data, th.ctypes.data, cap, C.byref(n)))
    rp, rpi, rth = orc.per_site_diversity(vs, haps, region)
    k = n.value
    assert k == len(rp) and np.array_equal(p[:k], rp)
    for got, ref in ((pi[:k], rpi), (th[:k], rth)):
        assert np.array_equal(np.isnan(got), np.isnan(ref))
        ok = ~np.isnan(ref)
        assert np.all(np.abs(got[ok] - ref[ok]) <= 1e-9 * np.abs(ref[ok]))


def _check(m, g, pos, lists, tracks=True):
    vs, d = orc.from_numpy(g, pos)
    for haps in lists:
        grp = m.group(haps)
        got = grp.summary(want_arrays=True)  # the first call on the group: its counts as K1 left them
        ref = orc.build_summary(d, haps)
        assert np.array_equal(got["called"], ref.called) and np.array_equal(got["alt"], ref.alt)
        assert got["segregating_sites"] == ref.seg
        if tracks and len(set(haps)) == len(haps):  # the sparse oracle counts a listed duplicate twice
            _tracks_match(grp, haps, vs, pos, 37)


@pytest.mark.parametrize("S", [96, 97])  # stride 192: direct rows; 194: staged rows
def test_u8_bitmap(S):
    from ferromic_b200.api import _Matrix
    g, pos = _cohort(1001, S, 10 + S)
    miss = g < 0
    m = _Matrix(np.where(miss, 0, g).astype(np.uint8), miss, pos, max_allele=1, always_bitmap=True, ingest="u8")
    _check(m, g, pos, _hap_lists(S))


def test_u8_groups_in_one_launch():
    from ferromic_b200.api import _Matrix
    g, pos = _cohort(999, 128, 5)
    miss = g < 0
    m = _Matrix(np.where(miss, 0, g).astype(np.uint8), miss, pos, max_allele=1, always_bitmap=True, ingest="u8")
    lists = _hap_lists(128)
    m.groups(lists)  # fm_groups_create: one K1 launch for all of them
    _check(m, g, pos, lists)


def test_in_band_int8():
    from ferromic_b200.api import _Matrix
    g, pos = _cohort(1003, 130, 21)
    m = _Matrix.from_int8(g.astype(np.int8), pos, 1, ingest="u8")
    _check(m, g, pos, _hap_lists(130))


def test_packed_called_plane():
    from ferromic_b200.api import _Matrix
    g, pos = _cohort(1005, 131, 22)
    miss = g < 0
    m = _Matrix(np.where(miss, 0, g).astype(np.uint8), miss, pos, max_allele=1, always_bitmap=True,
                ingest="packed-dense")
    assert m.ingest_mode == "packed-dense"
    _check(m, g, pos, _hap_lists(131))


@pytest.mark.parametrize("gap_code", [True, False])
def test_packed_sparse(gap_code, monkeypatch):
    from ferromic_b200 import api
    from ferromic_b200.api import _Matrix
    monkeypatch.setattr(api, "SPARSE_GAP_CODE", gap_code)
    g, pos = _cohort(1007, 129, 23, missing=0.01)
    miss = g < 0
    m = _Matrix(np.where(miss, 0, g).astype(np.uint8), miss, pos, max_allele=1, always_bitmap=True,
                ingest="packed-sparse")
    assert m.ingest_mode == "packed-sparse"
    _check(m, g, pos, _hap_lists(129))


@pytest.mark.parametrize("with_tracks", [False, True])
@pytest.mark.parametrize("packed", [False, True])
def test_streaming_ingest_in_chunks(packed, with_tracks):
    from ferromic_b200.api import _Matrix
    V, S = 2011, 128
    g, pos = _cohort(V, S, 24)
    miss = g < 0
    lists = [h for h in _hap_lists(S) if len(set(h)) == len(h)]
    cap = V
    req = None
    if with_tracks:
        req = {"groups": list(range(len(lists))), "raw_n": [len(h) for h in lists], "region": (int(pos[37]), int(pos[-1])),
               "mask": None, "filtered": None, "pos": np.zeros(cap, dtype=np.int64), "pi": np.zeros((len(lists), cap)),
               "theta": np.zeros((len(lists), cap)), "capacity": cap}
    m = _Matrix.ingest(np.where(miss, 0, g).astype(np.uint8), miss, pos, lists, chunk_rows=300, calls=3,
                       always_bitmap=True, packed=packed, tracks=req)
    _check(m, g, pos, lists)
    if with_tracks:
        vs, _ = orc.from_numpy(g, pos)
        n = m.track_sites
        for i, haps in enumerate(lists):
            rp, rpi, rth = orc.per_site_diversity(vs, haps, req["region"])
            assert n == len(rp) and np.array_equal(req["pos"][:n], rp)
            for got, ref in ((req["pi"][i, :n], rpi), (req["theta"][i, :n], rth)):
                assert np.array_equal(np.isnan(got), np.isnan(ref))
                ok = ~np.isnan(ref)
                assert np.all(np.abs(got[ok] - ref[ok]) <= 1e-9 * np.abs(ref[ok]))


def test_rows_wider_than_a_warp_slice():
    """40,000 samples: the u8 row does not fit the row-staged K1, so fm_k_repack writes the groups (several warps
    per row add up the row's called count)."""
    from ferromic_b200.api import _Matrix
    S = 40000
    g, pos = _cohort(40, S, 25, missing=0.01)
    miss = g < 0
    m = _Matrix(np.where(miss, 0, g).astype(np.uint8), miss, pos, max_allele=1, always_bitmap=True, ingest="u8")
    lists = [both_sides(range(S)), both_sides(range(0, S, 3)) + [(1, 1), (1, 1)], both_sides(range(119))]
    vs, d = orc.from_numpy(g, pos)
    for haps in lists:
        got = m.group(haps).summary(want_arrays=True)
        ref = orc.build_summary(d, haps)
        assert np.array_equal(got["called"], ref.called) and np.array_equal(got["alt"], ref.alt)
    _tracks_match(m.group(lists[0]), lists[0], vs, pos, 3)


def test_vcf_packed_batch():
    from ferromic_b200 import vcf
    from oracle import vcf as ov
    rng = np.random.default_rng(26)
    S, n_lines = 136, 700
    gts = ["0|0", "0|1", "1|0", "1|1", "./.", "0/1"]
    body = []
    for i in range(n_lines):
        p = rng.choice(len(gts), size=S, p=[0.4, 0.2, 0.2, 0.15, 0.03, 0.02])
        body.append("\t".join(["chr1", str(1000 + 3 * i), ".", "A", "T", ".", "PASS", ".", "GT:GQ"] +
                              [gts[k] + ":50" for k in p]))
    body = "\n".join(body) + "\n"
    text = "##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + \
        "\t".join(f"S{i}" for i in range(S)) + "\n" + body
    regions = [(900, 1000 + 3 * n_lines)]
    batch, _ = vcf.process_vcf_text(text.encode(), "1", regions, 30)
    kept = [9 + i for i in range(S)]
    out, _, _, _ = ov.process_lines(ov.split_lines(body), "1", regions, kept, 30)
    m = batch.matrix(packed=True)
    vs = orc.variants_from_python([{"position": v[0], "genotypes": v[1]} for v in out], S)
    d = orc.dense_from_variants(vs, S)
    for haps in _hap_lists(S):
        got = m.group(haps).summary(want_arrays=True)
        ref = orc.build_summary(d, haps)
        assert np.array_equal(got["called"], ref.called) and np.array_equal(got["alt"], ref.alt)


def test_plane_bytes_per_step():
    """fm_bench_result.plane_bytes_per_step counts what a step reads and writes: allele rows, tail words, 4 B of
    called count per site and group, 16 B of tracks per site and group."""
    from ferromic_b200 import _lib
    from ferromic_b200.api import _Matrix
    L = _lib.lib()
    V = 2000
    g, pos = _cohort(V, 200, 27, missing=0.01)
    miss = g < 0
    m = _Matrix(np.where(miss, 0, g).astype(np.uint8), miss, pos, max_allele=1, always_bitmap=True, ingest="u8")
    lists = [both_sides(range(84)), both_sides(range(84, 200))]  # 168 (tail layout: 1 row word + 2 tail words), 232
    gh = (C.c_void_p * 2)(*[m.group(h).handle.value for h in lists])
    res = _lib.BenchResult()
    _lib.check(L.fm_bench_diversity(gh, 2, 1, None, 0, 1, None, C.byref(res), None, None))
    row = [16 * 1 + 4 * 2, 16 * 2]
    assert res.plane_bytes_per_step == sum(V * (r + 4 + 16) for r in row)
    for i in range(2):
        assert res.group_bytes[i] == V * (row[i] + 4 + 16)
