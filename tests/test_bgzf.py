"""BGZF input on the device: fm_bgzf_inflate and fm_vcf_parse_bgzf (vcf.bgzf_inflate, vcf.process_vcf_bgzf).

Streams come from a small BGZF writer here (zlib raw deflate per member, the `BC` header, CRC32/ISIZE trailer, the
EOF member).  The decoder's __host__ __device__ functions also run on the CPU under AddressSanitizer and UBSan
(tests/bgzf_host.cpp) over every corpus and malformed case below, so a decoder bug shows there before a GPU runs."""
import ctypes as C
import functools
import gzip
import json
import random
import struct
import zlib

import numpy as np
import pytest

from tests.test_vcf import make_vcf


# ------------------------------------------------------------------------------------------- BGZF writer
def deflate(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, flushes=()):
    """Raw deflate; flushes: (offset, zlib flush mode) pairs applied mid-stream (several blocks, empty stored ones)."""
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 9, strategy)
    out, prev = [], 0
    for off, mode in flushes:
        out += [c.compress(data[prev:off]), c.flush(mode)]
        prev = off
    out += [c.compress(data[prev:]), c.flush()]
    return b"".join(out)


def member(payload, raw=None, crc=None, isize=None, **kw):
    raw = deflate(payload, **kw) if raw is None else raw
    bsize = 18 + len(raw) + 8
    assert bsize <= 65536
    head = b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + struct.pack("<H", bsize - 1)
    crc = zlib.crc32(payload) if crc is None else crc
    return head + raw + struct.pack("<II", crc, len(payload) if isize is None else isize)


EOF_MEMBER = member(b"")


def bgzf(data, size=0xff00, eof=True, cuts=None, **kw):
    """Members of `size` inflated bytes (bgzip writes 0xff00), or members ending at the offsets `cuts`."""
    cuts = list(range(size, len(data), size)) if cuts is None else sorted(cuts)
    bounds = [0] + [c for c in cuts if 0 < c < len(data)] + [len(data)]
    parts = [member(data[a:b], **kw) for a, b in zip(bounds, bounds[1:]) if b > a]
    return b"".join(parts) + (EOF_MEMBER if eof else b"")


class Bits:
    """LSB-first bit writer for hand-assembled deflate data."""

    def __init__(self):
        self.bits = []

    def put(self, value, n):
        self.bits += [(value >> i) & 1 for i in range(n)]

    def code(self, code, n):  # Huffman codes go most significant bit first
        self.bits += [(code >> (n - 1 - i)) & 1 for i in range(n)]

    def bytes(self):
        return np.packbits(np.array(self.bits + [0] * (-len(self.bits) % 8), dtype=np.uint8), bitorder="little").tobytes()

    def literal(self, b):  # fixed Huffman
        self.code(0x30 + b, 8) if b < 144 else self.code(0x190 + b - 144, 9)


def far_match_member():
    """One fixed-Huffman member with a distance-32768 match (zlib never emits a distance above 32506)."""
    rng = random.Random(5)
    lits = bytes(rng.randrange(256) for _ in range(32768))
    w = Bits()
    w.put(1, 1)
    w.put(1, 2)
    for b in lits:
        w.literal(b)
    w.code(0xc0 + 5, 8)  # litlen 285: length 258
    w.code(29, 5)  # distance code 29: 24577 + 13 extra bits
    w.put(32768 - 24577, 13)
    w.code(0, 7)  # end of block
    payload = lits + lits[:258]
    return member(payload, raw=w.bytes()), payload


def text_payload(n, seed=1):
    rng = np.random.default_rng(seed)
    return make_vcf(rng, n, 40, odd=0.02).encode()


def fib_payload():
    f = [1, 1]
    while len(f) < 22:
        f.append(f[-1] + f[-2])
    data = bytearray()
    for sym, k in enumerate(f):
        data += bytes([sym + 40]) * k
    random.Random(3).shuffle(data)
    return bytes(data)


@functools.lru_cache(maxsize=None)
def corpus():
    """name -> (BGZF stream, inflated bytes)."""
    text = text_payload(500)
    rnd = random.Random(7).randbytes(200_000)
    cases = {f"level{lv}": (bgzf(text, level=lv), text) for lv in (0, 1, 6, 9)}
    for name in ("Z_FIXED", "Z_HUFFMAN_ONLY", "Z_RLE", "Z_FILTERED"):
        cases[name.lower()] = (bgzf(text, strategy=getattr(zlib, name)), text)
    fl = [(100, zlib.Z_SYNC_FLUSH), (5000, zlib.Z_FULL_FLUSH), (5000, zlib.Z_SYNC_FLUSH), (20000, zlib.Z_SYNC_FLUSH)]
    cases["several_blocks"] = (bgzf(text, flushes=fl), text)
    cases["random_stored"] = (bgzf(rnd), rnd)
    run = b"A" * 300_000
    cases["one_byte_run"] = (bgzf(run), run)
    fib = fib_payload()
    cases["fibonacci_15_bit_codes"] = (bgzf(fib, strategy=zlib.Z_HUFFMAN_ONLY), fib)
    far, far_payload = far_match_member()
    cases["distance_32768"] = (far + EOF_MEMBER, far_payload)
    sized = text[:1] + text[:0xff00] + text[1000:1000 + 0xff00]
    cases["member_sizes_0_1_ff00"] = (EOF_MEMBER + member(text[:1]) + EOF_MEMBER + member(text[:0xff00])
                                      + member(text[1000:1000 + 0xff00]) + EOF_MEMBER, sized)
    full = (b"ab" * 32768)
    cases["isize_65536"] = (member(full) + member(text[:300]) + EOF_MEMBER, full + text[:300])
    cases["empty_stream"] = (b"", b"")
    cases["eof_only"] = (EOF_MEMBER, b"")
    return cases


def _dynamic_oversubscribed():
    w = Bits()
    w.put(1, 1)
    w.put(2, 2)  # dynamic
    w.put(0, 5)
    w.put(0, 5)
    w.put(15, 4)  # 19 code-length codes ...
    for _ in range(19):
        w.put(1, 3)  # ... all of length 1
    return w.bytes() + b"\0" * 8


def _fixed_far_distance():
    w = Bits()
    w.put(1, 1)
    w.put(1, 2)
    w.literal(ord("A"))
    w.code(1, 7)  # length 3
    w.code(1, 5)  # distance 2, one byte produced
    w.code(0, 7)
    return w.bytes()


HOST_PARSE, HOST_NOT_BGZF = 101, 102  # the harness's walk errors


@functools.lru_cache(maxsize=None)
def malformed():
    """name -> (stream, expected harness code, index of the bad member).  Two good members lead every stream."""
    text = text_payload(120, seed=9)
    lead = member(text[:3000]) + member(text[3000:6000])
    good = text[6000:9000]
    m = member(good)
    stored = member(text[:1000], level=0)
    cases = {
        "crc_flipped": (m[:-8] + bytes([m[-8] ^ 1]) + m[-7:], 9),
        "isize_larger": (member(good, isize=len(good) + 1), 8),
        "isize_smaller": (member(good, isize=len(good) - 1), 7),
        "truncated_member": (m[: len(m) // 2], HOST_PARSE),
        "truncated_deflate": (member(text[:1000], raw=stored[18:18 + 500]), 1),
        "block_type_3": (member(b"x", raw=b"\x07\x00"), 2),
        "stored_length": (member(b"abcde", raw=b"\x01" + struct.pack("<HH", 5, 5) + b"abcde"), 3),
        "oversubscribed_code_lengths": (member(b"x", raw=_dynamic_oversubscribed()), 4),
        "distance_beyond_output": (member(b"AAAA", raw=_fixed_far_distance()), 6),
        "trailing_bytes": (member(good, raw=deflate(good) + b"\0"), 10),
        "plain_gzip": (gzip.compress(good), HOST_NOT_BGZF),
        "not_gzip": (b"##fileformat=VCFv4.2\n" * 3, HOST_PARSE),
    }
    return {k: (lead + v + EOF_MEMBER, code, 2) for k, (v, code) in cases.items()}


def host_harness_results():
    """Runs every case through the sanitized CPU decoder (called in a child interpreter)."""
    from tests import bgzf_host
    res = {}
    for name, (gz, want) in corpus().items():
        st, bad, out = bgzf_host.inflate(gz)
        res[name] = [st, bad, out == want]
    for name, (gz, code, bad_member) in malformed().items():
        st, bad, _ = bgzf_host.inflate(gz)
        res["bad_" + name] = [st, bad, st == code and bad == bad_member]
    return res


# ------------------------------------------------------------------------------------------- CPU tests
def test_writer_round_trips_through_gzip():
    for name, (gz, want) in corpus().items():
        assert gzip.decompress(gz) == want, name


def test_host_decoder_under_sanitizers():
    """The decoder's host/device functions, serially on the CPU with ASan + UBSan: byte-equal to zlib on the corpus,
    and every malformed stream returns its code without a sanitizer report."""
    from tests import bgzf_host
    bgzf_host.build()
    r = bgzf_host.run_in_child("import json\nfrom tests import test_bgzf as t\n"
                               "print(json.dumps(t.host_harness_results()))")
    assert r.returncode == 0, r.stderr[-6000:]
    assert "Sanitizer" not in r.stderr and "runtime error" not in r.stderr, r.stderr[-6000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    assert len(res) == len(corpus()) + len(malformed())
    bad = {k: v for k, v in res.items() if not v[2]}
    assert not bad, bad


def test_bgzf_entry_points_fail_loudly_without_device():
    """Like the other stages: no CPU path behind the BGZF entry points, whatever the input (the device check comes
    before the member walk)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device is present")
    import ferromic_b200 as fm
    from ferromic_b200 import _lib, vcf
    gz = corpus()["level6"][0]
    for data in (gz, b"not gzip at all", gzip.compress(b"x"), b""):
        with pytest.raises(fm.FerromicGpuError) as exc:
            vcf.bgzf_inflate(data)
        assert exc.value.code == _lib.FM_ERR_NO_DEVICE
        kept = np.array([9], dtype=np.uint32)
        reg = np.array([[0, 10]], dtype=np.int64)
        h = C.c_void_p()
        st = _lib.lib().fm_vcf_parse_bgzf(data, len(data), 0, b"1", reg.ctypes.data, 1, kept.ctypes.data, 1, 30, 0,
                                          None, 0, 0, None, 0, 2, C.byref(h))
        assert st == _lib.FM_ERR_NO_DEVICE and not h


# ------------------------------------------------------------------------------------------- GPU tests
@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(corpus()))
def test_device_inflate_matches_gzip(name):
    from ferromic_b200 import vcf
    gz, want = corpus()[name]
    assert vcf.bgzf_inflate(gz) == want == gzip.decompress(gz)


@pytest.mark.gpu
def test_device_prefix_reads():
    from ferromic_b200 import _lib
    gz, want = corpus()["level6"]
    n = len(want)
    for cap in (0, 1, 1000, 0xff00 - 1, 0xff00, 0xff00 + 17, n - 1, n, n + 5):
        out = (C.c_uint8 * max(cap, 1))()
        total = C.c_uint64()
        _lib.check(_lib.lib().fm_bgzf_inflate(gz, len(gz), out, cap, C.byref(total)))
        assert total.value == n
        assert bytes(out)[:min(cap, n)] == want[:cap], cap


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(malformed()))
def test_device_rejects_malformed_streams(name):
    from ferromic_b200 import _lib, vcf
    gz, code, bad = malformed()[name]
    L = _lib.lib()
    out = (C.c_uint8 * (1 << 20))()
    total = C.c_uint64()
    st = L.fm_bgzf_inflate(gz, len(gz), out, len(out), C.byref(total))
    assert st == (_lib.FM_ERR_UNSUPPORTED if code == HOST_NOT_BGZF else _lib.FM_ERR_PARSE)
    msg = L.fm_last_error().decode()
    assert f"BGZF member {bad} at byte offset " in msg, msg
    if code == HOST_NOT_BGZF:
        assert "bgzip" in msg and "fm_vcf_parse" in msg
    good, want = corpus()["level6"]
    assert vcf.bgzf_inflate(good) == want  # the library stays usable


HEADER_COLS = 40


def vcf_header(n_cols=HEADER_COLS, meta_lines=2):
    meta = "".join(f"##INFO=<ID=X{i},Number=1,Type=String,Description=\"{'padding ' * 8}\">\n"
                   for i in range(meta_lines))
    return ("##fileformat=VCFv4.2\n" + meta + "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t"
            + "\t".join(f"S{i}" for i in range(n_cols)) + "\n")


def matrix_outcome(batch, packed):
    """What from_variants gives (None, the matrix's shape, or its refusal) and what a group over all haplotypes of
    that matrix gives (per-site counts, or the refusal: allele values above 15 are unsupported on the group path)."""
    try:
        m = batch.matrix(packed=packed)
    except NotImplementedError as e:
        return "unsupported: " + str(e)
    if m is None:
        return None
    shape = (m.V, m.S, m.P, m.max_allele, m.has_missing)
    try:
        s = m.group([(i, side) for i in range(m.S) for side in range(m.P)]).summary(True)
        return shape, s["alt"].tobytes(), s["called"].tobytes(), s["segregating_sites"]
    except NotImplementedError as e:
        return shape, "unsupported: " + str(e)


def assert_same_parse(text, gz, exclusion=("S3",), **kw):
    from ferromic_b200 import vcf
    regions = [(950, 1200), (1200, 1300), (1500, 2100)]
    allow = {"1": [(1000, 1100), (1050, 1250), (1600, 1900)]}
    mask = {"1": [(1020, 1030), (1700, 1705)]}
    # max_ploidy 2, as the estimators take it: longer genotypes become error lines, compared like the rest
    a, na = vcf.process_vcf_text(text, "chr1", regions, 30, allow, mask, exclusion, **kw)
    b, nb = vcf.process_vcf_bgzf(gz, "chr1", regions, 30, allow, mask, exclusion, **kw)
    assert na == nb
    assert a.stats() == b.stats() and a.errors == b.errors
    assert int(a.info.n_lines) == int(b.info.n_lines)
    assert np.array_equal(a.positions, b.positions) and np.array_equal(a.flags, b.flags)
    assert a.allele_info() == b.allele_info()
    assert np.array_equal(a.genotypes(), b.genotypes())
    assert np.array_equal(a.positions_with_missing(), b.positions_with_missing())
    assert np.array_equal(a.filtered_positions(), b.filtered_positions())
    assert float(a.info.inflate_ms) == 0.0  # the text path inflates nothing; the BGZF one whenever there are lines
    assert float(b.info.inflate_ms) > 0.0 or int(b.info.n_lines) == 0
    for packed in (True, False):
        assert matrix_outcome(a, packed) == matrix_outcome(b, packed)
    return a


def _vcf_text(seed, n_lines, n_cols=HEADER_COLS, crlf=False, meta_lines=2, terminated=True, odd=0.03):
    rng = np.random.default_rng(seed)
    body = make_vcf(rng, n_lines, n_cols, odd=odd, crlf=crlf, chrs=("chr1", "1", "chr2"))
    eol = "\r\n" if crlf else "\n"
    body = body.rstrip("\r\n") + (eol if terminated else "")
    return (vcf_header(n_cols, meta_lines) + body).encode()


@pytest.mark.gpu
@pytest.mark.parametrize("crlf", [False, True])
@pytest.mark.parametrize("size", [997, 4096, 0xff00])
def test_bgzf_parse_equals_text_parse(crlf, size):
    text = _vcf_text(11 + size, 400, crlf=crlf)
    assert_same_parse(text, bgzf(text, size=size))


@pytest.mark.gpu
def test_bgzf_parse_member_boundaries():
    """A header over several members; members ending inside a line, between '\\r' and '\\n', right after '\\n'; a
    line longer than a member; an unterminated last line."""
    text = _vcf_text(21, 60, n_cols=1500, crlf=True, meta_lines=300, terminated=False)
    crs = [i for i in range(len(text)) if text[i:i + 2] == b"\r\n"]
    cuts = set()
    for k, i in enumerate(crs[::3]):
        cuts |= {i + 1, i + 2 + 37 * (k % 5)} if k % 2 else {i + 2}
    cuts |= set(range(0, len(text), 0xff00))
    assert max(b - a for a, b in zip(sorted(crs), sorted(crs)[1:])) > 4096  # a line longer than a member below
    assert_same_parse(text, bgzf(text, cuts=sorted(cuts)))
    assert_same_parse(text, bgzf(text, size=4096))


@pytest.mark.gpu
def test_bgzf_parse_tiny_chunks(monkeypatch):
    """FM_VCF_CHUNK_BYTES below a member: every chunk is one member and carries a partial line to the next."""
    monkeypatch.setenv("FM_VCF_CHUNK_BYTES", "600")
    text = _vcf_text(31, 300, n_cols=30)
    assert_same_parse(text, bgzf(text, size=700))
    text = _vcf_text(32, 200, n_cols=30, crlf=True, terminated=False)
    assert_same_parse(text, bgzf(text, size=333))
    text = _vcf_text(33, 150, n_cols=24, odd=0.0)
    assert assert_same_parse(text, bgzf(text, size=500)).n_variants > 50


@pytest.mark.gpu
def test_bgzf_parse_empty_data_section():
    from ferromic_b200 import vcf
    for text in (vcf_header().encode(), vcf_header().encode().rstrip(b"\n")):
        b = assert_same_parse(text, bgzf(text, size=500))
        assert b.n_variants == 0 and int(b.info.n_lines) == 0
    header, off = vcf.read_bgzf_header(bgzf(vcf_header(meta_lines=400).encode(), size=1000))
    assert header == vcf_header(meta_lines=400).encode() and off == len(header)


@pytest.mark.gpu
def test_bgzf_parse_reports_bad_streams():
    from ferromic_b200 import vcf
    text = _vcf_text(41, 100)
    gz = bgzf(text, size=2000)
    cut = gz.rfind(b"\x1f\x8b\x08\x04", 0, len(gz) - len(EOF_MEMBER) - 1)
    bad = gz[:cut + 30] + bytes([gz[cut + 30] ^ 0x55]) + gz[cut + 31:]
    with pytest.raises(ValueError, match="BGZF member"):
        vcf.process_vcf_bgzf(bad, "chr1", [(0, 10 ** 9)], 30)
    with pytest.raises(NotImplementedError, match="bgzip"):
        vcf.process_vcf_bgzf(gzip.compress(text), "chr1", [(0, 10 ** 9)], 30)
    assert_same_parse(text, gz)


@pytest.mark.gpu
def test_bgzf_parse_full_size_pinned():
    """synth_text(20000, 2504): 352 MB of GT:GQ text as bgzip writes it, from a page-locked buffer."""
    import torch
    from tools.bench_vcf import synth_text
    from tools.bench_bgzf import bgzf_compress
    from ferromic_b200 import vcf
    text = vcf_header(2504).encode() + synth_text(20000, 2504)
    gz = bgzf_compress(text)
    pinned = torch.empty(len(gz), dtype=torch.uint8).pin_memory()
    pinned.numpy()[:] = np.frombuffer(gz, dtype=np.uint8)
    assert_same_parse(text, pinned.numpy(), exclusion=())
    assert vcf.bgzf_inflate(pinned.numpy()) == text
