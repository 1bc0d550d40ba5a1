"""BGZF output on the device: fm_bgzf_deflate, fm_falsta_tracks_bgzf (vcf.bgzf_deflate, the `bgzf=True` FALSTA
writers).

The encoder's phases are __host__ __device__ functions; tests/bgzf_deflate_host.cpp runs them serially on the CPU,
so the members the device must write are known here: the CPU tests check them under AddressSanitizer and UBSan
(round trips through gzip, zlib and the project's own decoder, the member walk, the stored bound, the ratio bar), and
the GPU tests check that the device writes exactly those bytes."""
import ctypes as C
import functools
import gzip
import json
import random
import struct
import threading
import zlib

import numpy as np
import pytest

from oracle import falsta as ofa
from tests.test_bgzf import assert_same_parse, fib_payload, text_payload, _vcf_text
from tests.test_falsta import _records

BLOCK = 0xff00
EOF_MEMBER = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def fst_corpus(region_len=1_000_000, n=30_000, tracks=6, seed=5) -> bytes:
    """FST tracks as append_fst_falsta writes them: 'NA' runs with a record at ~3 % of the positions."""
    rng = np.random.default_rng(seed)
    pos = np.sort(rng.choice(np.arange(1, region_len + 1), size=n, replace=False))
    vals = rng.random((tracks, n))
    vals[rng.random((tracks, n)) < 0.1] = np.nan
    vals[rng.random((tracks, n)) < 0.1] = 0.0
    out = []
    for t in range(tracks):
        tok = np.full(region_len, "NA", dtype=object)
        tok[pos - 1] = [ofa.fst_token(float(v)) for v in vals[t]]
        out.append(f">track_{t}_chr_1_start_1_end_{region_len}\n" + ",".join(tok) + "\n")
    return "".join(out).encode()


def far_repeat() -> bytes:
    """258 random bytes again at exactly distance 32768, with zeros between (nothing else to match them)."""
    x = random.Random(11).randbytes(258)
    return x + bytes(32768 - 258) + x


@functools.lru_cache(maxsize=None)
def corpus():
    """name -> input bytes."""
    text = text_payload(500)
    text = text * (6 * BLOCK // len(text) + 1)
    cases = {f"size_{n}": text[:n] for n in (0, 1, 2, 3, 257, 258, 259, BLOCK - 1, BLOCK, BLOCK + 1, 2 * BLOCK,
                                             3 * BLOCK + 7, 5 * BLOCK)}
    cases["run_1_byte"] = b"A" * 300_000
    cases["distance_32768"] = far_repeat()
    cases["random"] = random.Random(7).randbytes(200_000)
    cases["all_256_bytes"] = bytes(range(256)) * 300
    cases["fibonacci"] = fib_payload()
    return cases


@functools.lru_cache(maxsize=None)
def ratio_corpora():
    from tools.bench_vcf import synth_text
    return {"falsta_fst_1Mb": fst_corpus(), "vcf_gt_gq": synth_text(400, 2504)}


def members(gz: bytes):
    """(inflated size, member size) of every member, from the headers and trailers."""
    out, off = [], 0
    while off < len(gz):
        bsize = struct.unpack_from("<H", gz, off + 16)[0] + 1
        out.append((struct.unpack_from("<I", gz, off + bsize - 4)[0], bsize))
        off += bsize
    return out


def zlib_members(gz: bytes) -> bytes:
    out, rest = [], gz
    while rest:
        d = zlib.decompressobj(31)
        out.append(d.decompress(rest))
        rest = d.unused_data
    return b"".join(out)


def zlib1_bgzf_size(data: bytes) -> int:
    from tools.bench_bgzf import bgzf_compress
    return len(bgzf_compress(data, level=1))


def check_stream(gz: bytes, data: bytes, sanitize: bool = True):
    """Every property a stream of `data` must have; returns a list of failures."""
    from tests import bgzf_deflate_host as h
    bad = []
    if gzip.decompress(gz) != data:
        bad.append("gzip.decompress")
    if zlib_members(gz) != data:
        bad.append("zlib")
    st, n_mem = h.walk(gz, sanitize)
    if st or n_mem != (len(data) + BLOCK - 1) // BLOCK + 1:
        bad.append(f"bgzf_walk {st} {n_mem}")
    st, at, out = h.inflate(gz, sanitize)
    if st or out != data:
        bad.append(f"bh_inflate {st} member {at}")
    if not gz.endswith(EOF_MEMBER):
        bad.append("EOF member")
    for isize, bsize in members(gz):
        if bsize > isize + 31 and isize:
            bad.append(f"member of {isize} bytes is {bsize} bytes")
    return bad


def host_harness_results():
    """Runs every case through the sanitized CPU encoder (called in a child interpreter)."""
    from tests import bgzf_deflate_host as h
    res = {}
    for name, data in {**corpus(), **ratio_corpora()}.items():
        gz = h.deflate(data)
        res[name] = {"bad": check_stream(gz, data), "size": len(gz), "members": members(gz)}
    return res


# ------------------------------------------------------------------------------------------- CPU tests
@functools.lru_cache(maxsize=None)
def _host_results():
    from tests import bgzf_host, bgzf_deflate_host
    bgzf_deflate_host.build()
    r = bgzf_host.run_in_child("import json\nfrom tests import test_bgzf_deflate as t\n"
                               "print(json.dumps(t.host_harness_results()))")
    assert r.returncode == 0, r.stderr[-6000:]
    assert "Sanitizer" not in r.stderr and "runtime error" not in r.stderr, r.stderr[-6000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_host_encoder_under_sanitizers():
    """The encoder's host/device phases, serially on the CPU with ASan + UBSan: every output round-trips through
    gzip, zlib and the project's decoder, passes the member walk and ends with the EOF member; no member is larger
    than stored (n + 31 bytes)."""
    res = _host_results()
    assert set(res) == set(corpus()) | set(ratio_corpora())
    bad = {k: v["bad"] for k, v in res.items() if v["bad"]}
    assert not bad, bad
    assert res["size_0"]["size"] == len(EOF_MEMBER)
    # random bytes take the stored path: every member is exactly n + 31 bytes
    assert all(b == i + 31 for i, b in res["random"]["members"][:-1])
    # one byte repeated compresses to a few bytes per member; a 32768-distance repeat is found
    assert all(b < 200 for i, b in res["run_1_byte"]["members"])
    assert res["distance_32768"]["size"] < 32768 // 8


def test_ratio_within_bar_of_zlib_level_1():
    """On the FALSTA and VCF corpora the encoder's BGZF is at most 1.15x zlib level 1 in the same 0xff00 members."""
    res = _host_results()
    for name, data in ratio_corpora().items():
        ref = zlib1_bgzf_size(data)
        assert res[name]["size"] <= 1.15 * ref, (name, res[name]["size"], ref)


def test_deflate_entry_points_without_device():
    """fm_bgzf_deflate_bound is host-only; the two compressing entry points have no CPU path."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device is present")
    import ferromic_b200 as fm
    from ferromic_b200 import _lib, vcf
    L = _lib.lib()
    b = C.c_size_t()
    assert L.fm_bgzf_deflate_bound(0, 0, C.byref(b)) == 0 and b.value == 0
    assert L.fm_bgzf_deflate_bound(0, _lib.FM_BGZF_EOF, C.byref(b)) == 0 and b.value == 28
    assert L.fm_bgzf_deflate_bound(BLOCK + 1, _lib.FM_BGZF_EOF, C.byref(b)) == 0 and b.value == BLOCK + 1 + 62 + 28
    for data in (b"x" * 1000, b""):
        with pytest.raises(fm.FerromicGpuError) as exc:
            vcf.bgzf_deflate(data)
        assert exc.value.code == _lib.FM_ERR_NO_DEVICE
    pos = np.array([3], dtype=np.int64)
    val = np.array([0.5], dtype=np.float64)
    heads = (C.c_char_p * 1)(b">h\n")
    out = (C.c_uint8 * 4096)()
    n = C.c_size_t()
    st = L.fm_falsta_tracks_bgzf(pos.ctypes.data, val.ctypes.data, 1, 1, 1, 10, 1, C.cast(heads, C.c_void_p), out,
                                 4096, C.byref(n))
    assert st == _lib.FM_ERR_NO_DEVICE


# ------------------------------------------------------------------------------------------- GPU tests
def host_deflate(data: bytes, eof: bool = True) -> bytes:
    from tests import bgzf_deflate_host
    return bgzf_deflate_host.deflate(data, eof, sanitize=False)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(corpus()) + ["falsta_fst_1Mb", "vcf_gt_gq"])
def test_device_deflate_equals_host_build(name):
    from ferromic_b200 import vcf
    data = corpus()[name] if name in corpus() else ratio_corpora()[name]
    gz = vcf.bgzf_deflate(data)
    assert gz == host_deflate(data)
    assert vcf.bgzf_deflate(data) == gz  # and again
    assert gzip.decompress(gz) == data
    assert vcf.bgzf_inflate(gz) == data
    assert vcf.bgzf_deflate(data, eof=False) == gz[:-len(EOF_MEMBER)]


@pytest.mark.gpu
def test_device_deflate_large_and_threads():
    """352 MB of GT:GQ text: members are independent, so the stream equals its 0xff00-aligned parts' streams; four
    host threads compressing different inputs at once get what one thread gets."""
    from tools.bench_vcf import synth_text
    from ferromic_b200 import vcf
    text = synth_text(20000, 2504)
    gz = vcf.bgzf_deflate(text)
    assert vcf.bgzf_inflate(gz) == text
    assert zlib_members(gz) == text
    cut = (len(text) // 3) // BLOCK * BLOCK
    assert vcf.bgzf_deflate(text[:cut], eof=False) + vcf.bgzf_deflate(text[cut:]) == gz
    inputs = [text[k * 10_000_000 + k * 777:(k + 1) * 10_000_000] for k in range(4)]
    want = [vcf.bgzf_deflate(x) for x in inputs]
    got = [None] * 4

    def run(k):
        got[k] = [vcf.bgzf_deflate(inputs[k]) for _ in range(3)]

    ts = [threading.Thread(target=run, args=(k,)) for k in range(4)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    for k in range(4):
        assert got[k] == [want[k]] * 3, k
    assert want[1] == host_deflate(inputs[1])


@pytest.mark.gpu
@pytest.mark.parametrize("size", [997, BLOCK])
def test_parse_of_device_bgzf_equals_text_parse(size):
    from ferromic_b200 import vcf
    text = _vcf_text(51 + size, 400)
    assert_same_parse(text, vcf.bgzf_deflate(text))
    text = _vcf_text(61, 300, crlf=True, terminated=False)
    assert_same_parse(text, vcf.bgzf_deflate(text))


def _tracks_bgzf(pos, values, rs, re, mode, heads) -> bytes:
    from ferromic_b200 import falsta
    return falsta._render_bgzf(pos, values, rs, re, mode, heads)


@pytest.mark.gpu
def test_falsta_tracks_bgzf_inflates_to_headed_text():
    """fm_falsta_tracks_bgzf = heads + fm_falsta_tracks lines, deflated: for the shapes of the text tests, and the
    same members the host build writes for that text."""
    from ferromic_b200 import falsta, vcf
    rng = np.random.default_rng(11)
    for n, (rs, re) in ((0, (1, 9)), (1, (5, 5)), (300, (100, 900)), (5000, (-3, 2500)), (40000, (1000, 200000))):
        pos, v = _records(rng, n, rs - 50, re + 50)
        heads = [f">h{t}_{rs}_{re}\n" for t in range(6)]
        gz = _tracks_bgzf(pos, np.ascontiguousarray(v.T), rs, re, falsta.FST, heads)
        text = b"".join(h.encode() + line + b"\n" for h, line in
                        zip(heads, falsta.track_lines(pos, np.ascontiguousarray(v.T), rs, re, falsta.FST)))
        assert vcf.bgzf_inflate(gz) == gzip.decompress(gz) == text
        assert gz == host_deflate(text, eof=False)
        wc = [(int(p), *row) for p, row in zip(pos, v)]
        hud = [(int(p), row[0], row[1], row[2]) for p, row in zip(pos[::2], v[::2])]
        gz = falsta._fst("7", rs, re, wc, hud, falsta._render_bgzf)
        assert gzip.decompress(gz).decode() == ofa.fst_falsta_text("7", rs, re, wc, hud)
    rng = np.random.default_rng(12)
    n = 20000
    pos, v = _records(rng, n, 1, 60000)
    v = np.where(np.isinf(v), 0.25, v)
    gid = rng.integers(0, 2, size=n)
    flt = rng.random(n) < 0.4
    recs = [(int(p), float(a), float(b), int(g), bool(f)) for p, a, b, g, f in zip(pos, v[:, 0], v[:, 1], gid, flt)]
    for rs, re in ((1, 60000), (20000, 20100), (70000, 70010)):
        gz = falsta._diversity("chr2", rs, re, recs, falsta._render_bgzf)
        assert gzip.decompress(gz).decode() == ofa.diversity_falsta_text("chr2", rs, re, recs)


@pytest.mark.gpu
def test_bgzf_writers_append_members(tmp_path):
    from tests import bgzf_deflate_host as h
    from ferromic_b200 import falsta, vcf
    rng = np.random.default_rng(13)
    pos, v = _records(rng, 3000, 1, 90000)
    wc = [(int(p), *row) for p, row in zip(pos, v)]
    hud = [(int(p), row[0], row[1], row[2]) for p, row in zip(pos[::3], v[::3])]
    div = [(int(p), float(a), float(b), int(p) % 2, bool(p % 5 == 0)) for p, a, b in zip(pos, v[:, 0], v[:, 1])]
    rows = [("1", 1, 90000, 0, 1, 0.1, 0.2, float("nan"), 0.3, None), ("1", 1, 90000, "EUR", None, 1.0, 0.0, 0.5,
                                                                         float("inf"), 0.25)]
    paths = {k: tmp_path / f"{k}.gz" for k in ("fst", "div", "tsv")}
    want = {k: "" for k in paths}
    for rs, re in ((1, 90000), (500, 700), (95000, 96000)):
        falsta.append_fst_falsta(paths["fst"], "3", rs, re, wc, hud, bgzf=True)
        want["fst"] += ofa.fst_falsta_text("3", rs, re, wc, hud)
        falsta.append_diversity_falsta(paths["div"], "3", rs, re, div, bgzf=True)
        want["div"] += ofa.diversity_falsta_text("3", rs, re, div)
        falsta.append_hudson_tsv(paths["tsv"], rows, bgzf=True)
        want["tsv"] += falsta.hudson_tsv_text(rows).decode()
    falsta.append_fst_falsta(paths["fst"], "3", 1, 10, [], [], bgzf=True)  # nothing to write: no member
    for k, p in paths.items():
        with gzip.open(p, "rt") as f:
            assert f.read() == want[k], k
        raw = p.read_bytes()
        assert h.walk(raw, sanitize=False)[0] == 0
        assert vcf.bgzf_inflate(raw).decode() == want[k]
    # the default writes today's bytes: the same text, one gzip member per call
    falsta.append_fst_falsta(tmp_path / "plain.gz", "3", 1, 90000, wc, hud)
    assert gzip.decompress((tmp_path / "plain.gz").read_bytes()).decode() == ofa.fst_falsta_text("3", 1, 90000, wc,
                                                                                                   hud)


@pytest.mark.gpu
def test_deflate_capacity_and_argument_errors():
    from ferromic_b200 import _lib, vcf
    L = _lib.lib()
    data = corpus()[f"size_{3 * BLOCK + 7}"]
    gz = vcf.bgzf_deflate(data)
    n = C.c_size_t()
    small = (C.c_uint8 * 100)()
    for eof, need in ((1, len(gz)), (0, len(gz) - len(EOF_MEMBER))):
        assert L.fm_bgzf_deflate(data, len(data), eof, small, 100, C.byref(n)) == _lib.FM_ERR_INVALID_ARG
        assert n.value == need
    assert L.fm_bgzf_deflate(None, 10, 1, small, 100, C.byref(n)) == _lib.FM_ERR_INVALID_ARG
    assert L.fm_bgzf_deflate(data, len(data), 1, None, 100, C.byref(n)) == _lib.FM_ERR_INVALID_ARG
    assert L.fm_bgzf_deflate(data, len(data), 1, small, 100, None) == _lib.FM_ERR_INVALID_ARG
    assert L.fm_bgzf_deflate(data, len(data), 6, small, 100, C.byref(n)) == _lib.FM_ERR_INVALID_ARG
    assert L.fm_bgzf_deflate(b"", 0, 1, small, 100, C.byref(n)) == 0 and bytes(small)[:28] == EOF_MEMBER
    pos = np.array([3, 7, 9], dtype=np.int64)
    val = np.array([[0.5, 0.25, np.nan], [1.0, 0.0, 2.0]], dtype=np.float64)
    heads = (C.c_char_p * 2)(b">a\n", b">b\n")
    hp = C.cast(heads, C.c_void_p)
    out = (C.c_uint8 * 10)()
    args = (pos.ctypes.data, val.ctypes.data, 3, 2, 1, 10)
    assert L.fm_falsta_tracks_bgzf(*args, 1, hp, out, 10, C.byref(n)) == _lib.FM_ERR_INVALID_ARG
    need = n.value
    big = (C.c_uint8 * need)()
    assert L.fm_falsta_tracks_bgzf(*args, 1, hp, big, need, C.byref(n)) == 0 and n.value == need
    assert gzip.decompress(bytes(big)) == b">a\nNA,NA,0.500000,NA,NA,NA,0.250000,NA,NA,NA\n>b\n" \
                                          b"NA,NA,1.000000,NA,NA,NA,0,NA,2.000000,NA\n"
    assert L.fm_falsta_tracks_bgzf(*args, 5, hp, big, need, C.byref(n)) == _lib.FM_ERR_INVALID_ARG  # bad mode
    assert L.fm_falsta_tracks_bgzf(*args, 1, None, big, need, C.byref(n)) == _lib.FM_ERR_INVALID_ARG
    nul = (C.c_char_p * 2)(b">a\n", None)
    assert L.fm_falsta_tracks_bgzf(*args, 1, C.cast(nul, C.c_void_p), big, need, C.byref(n)) == _lib.FM_ERR_INVALID_ARG
    assert L.fm_falsta_tracks_bgzf(None, None, 3, 2, 1, 10, 1, hp, big, need, C.byref(n)) == _lib.FM_ERR_INVALID_ARG
    assert L.fm_falsta_tracks_bgzf(*args, 1, hp, big, need, None) == _lib.FM_ERR_INVALID_ARG
    assert vcf.bgzf_deflate(data) == gz  # the library stays usable
