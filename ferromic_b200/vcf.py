"""VCF parse/filter stage on the GPU (SURVEY §8f rank 4).

Host-side mirror of `process_vcf` (process.rs:4092-4468) for the text of one chromosome's VCF: the
header is consumed here like the reference does (sample names, exclusion set -> kept column
indices, :4181-4215); the data lines -- `process_variant` for every line, the merge of line-local
statistics, the (position, genotype bytes) sort -- run on the device through `fm_vcf_parse`.
Genotypes stay on the device; `VcfBatch.matrix()` is `DenseGenotypeMatrix::from_variants` without
a host round trip, ready for groups / partitions and the estimators.  BGZF input (`.vcf.gz`) is inflated
on the device too (`process_vcf_bgzf`)."""
from __future__ import annotations

import ctypes as C
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from ._lib import check, lib
from .api import _Matrix

FLAG_PASS, FLAG_MASK, FLAG_ALLOW, FLAG_LOW_GQ, FLAG_MISSING = 0, 1, 2, 4, 8  # process.rs:785-789
_WS = "\t\n\x0b\x0c\r "


def _normalize_chr(c: str) -> str:  # process.rs:4501-4514
    c = c.strip(_WS)
    for p in ("chr", "Chr", "CHR"):
        if c.startswith(p):
            return c[len(p):]
    return c


class VcfParseError(ValueError):
    """VcfError::Parse."""


def _message(code: int, aux: int, chr_: str, max_idx: int) -> str:
    if code == 10:
        return f"Invalid VCF line format: expected at least 9 fixed fields, found {aux}"
    if code == 11:
        return f"Invalid VCF line format: expected genotype field at column {max_idx + 1}, found {aux} columns"
    if code == 12:
        return "Invalid position"
    if code == 13:
        return f"Invalid 1-based pos: {aux}"
    if code == 14:
        return "GQ field not found in FORMAT"
    if code == 15:
        return f"GQ value missing in sample genotype field at chr{chr_}:{aux}"
    if code == 16:
        return f"unsupported: genotype longer than max_ploidy at position {aux}"
    return f"unsupported: more than 7 single-base ALT alleles at position {aux}"


class VcfBatch:
    """Result of one `fm_vcf_parse` call (one chunk of data lines)."""

    def __init__(self, handle, chr_: str, max_idx: int):
        self.handle = handle
        info = _lib.VcfInfo()
        check(lib().fm_vcf_batch_info(handle, C.byref(info)))
        self.info = info
        self.n_variants, self.n_samples, self.max_ploidy = int(info.n_variants), int(info.n_samples), int(info.max_ploidy)
        n = self.n_variants
        self.positions = np.zeros(n, dtype=np.int64)  # 0-based
        self.flags = np.zeros(n, dtype=np.uint8)
        self.stride = np.zeros(n, dtype=np.uint8)
        self._ref = np.zeros(n, dtype=np.uint8)
        self._n_alt = np.zeros(n, dtype=np.uint8)
        self._alts = np.zeros((n, 7), dtype=np.uint8)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        check(lib().fm_vcf_batch_variants(handle, p(self.positions), p(self.flags), p(self.stride), p(self._ref),
                                          p(self._n_alt), p(self._alts)))
        ne = int(info.n_errors)
        el, ec, ea = np.zeros(ne, dtype=np.uint64), np.zeros(ne, dtype=np.int32), np.zeros(ne, dtype=np.int64)
        check(lib().fm_vcf_batch_errors(handle, p(el), p(ec), p(ea), ne))
        self.error_codes = ec
        self.errors = [(int(l), _message(int(c), int(a), chr_, max_idx)) for l, c, a in zip(el, ec, ea)]

    def __del__(self):
        h, self.handle = getattr(self, "handle", None), None
        if h:
            lib().fm_vcf_batch_release(h)

    # FilteringStats / MissingDataInfo counters
    def stats(self) -> Dict[str, int]:
        keys = ("total_variants", "filtered_variants", "filtered_due_to_mask", "filtered_due_to_allow",
                "missing_data_variants", "low_gq_variants", "mnp_variants", "total_data_points", "missing_data_points")
        return {k: int(getattr(self.info, k)) for k in keys}

    def _positions(self, which: int, n: int) -> np.ndarray:
        out = np.zeros(n, dtype=np.int64)
        check(lib().fm_vcf_batch_positions(self.handle, which, out.ctypes.data_as(C.c_void_p), n))
        return out

    def positions_with_missing(self) -> np.ndarray:
        return self._positions(0, int(self.info.n_positions_with_missing))

    def filtered_positions(self) -> np.ndarray:
        return self._positions(1, int(self.info.n_filtered_positions))

    def allele_info(self) -> List[Tuple[str, List[str]]]:
        return [(chr(r), [chr(a) for a in alts[:n]]) for r, n, alts in zip(self._ref, self._n_alt, self._alts)]

    def genotypes(self) -> np.ndarray:
        """u8 [n_variants, n_samples, max_ploidy], CompressedGenotypes sentinel semantics (0xFF)."""
        gt = np.zeros((self.n_variants, self.n_samples, self.max_ploidy), dtype=np.uint8)
        if gt.size:
            check(lib().fm_vcf_batch_genotypes(self.handle, gt.ctypes.data_as(C.c_void_p)))
        return gt

    def matrix(self, pass_only: bool = False, packed: Optional[bool] = None) -> Optional[_Matrix]:
        """DenseGenotypeMatrix::from_variants over all variants (or the flags == 0 ones), on the device.
        packed (default: FERROMIC_GPU_INGEST != "u8"): the genotypes go straight to packed bit rows
        (fm_vcf_batch_matrix_packed) and the u8 matrix is never built; multi-allelic batches fall back to it."""
        import os
        from ._lib import FM_ERR_UNSUPPORTED
        if packed is None:
            packed = os.environ.get("FERROMIC_GPU_INGEST", "packed") != "u8"
        h = C.c_void_p()
        st = FM_ERR_UNSUPPORTED
        if packed:
            st = lib().fm_vcf_batch_matrix_packed(self.handle, int(bool(pass_only)), C.byref(h))
            if st != FM_ERR_UNSUPPORTED:
                check(st)
        if st == FM_ERR_UNSUPPORTED:
            h = C.c_void_p()
            check(lib().fm_vcf_batch_matrix(self.handle, int(bool(pass_only)), C.byref(h)))
        if not h:
            return None
        m = _Matrix.__new__(_Matrix)
        V, S, P, mx, hm = C.c_size_t(), C.c_size_t(), C.c_size_t(), C.c_uint8(), C.c_int()
        check(lib().fm_matrix_info(h, C.byref(V), C.byref(S), C.byref(P), C.byref(mx), C.byref(hm)))
        m.V, m.S, m.P, m.max_allele, m.has_missing = V.value, S.value, P.value, mx.value, bool(hm.value)
        m.handle = h
        m._groups = {}
        return m


def parse_header(header_line: str, exclusion_set: Iterable[str] = ()) -> Tuple[List[str], List[int]]:
    """#CHROM line -> (sample names, kept column indices), process.rs:4185-4213."""
    ex = set(exclusion_set)
    names, kept = [], []
    for idx, name in enumerate(header_line.split()):
        if idx >= 9 and name not in ex:
            names.append(name)
            kept.append(idx)
    if not names:
        raise VcfParseError("No samples remain after applying exclusions")
    return names, kept


def _pairs(v) -> np.ndarray:
    a = np.ascontiguousarray(np.asarray(v if v is not None else [], dtype=np.int64).reshape(-1, 2))
    return a


def _parse_args(chr_: str, regions, kept_col_indices, allow_regions, mask_regions):
    """The arguments after `chr` that fm_vcf_parse and fm_vcf_parse_bgzf share (arrays kept alive by the caller)."""
    key = _normalize_chr(chr_)

    def mode(m):
        if m is None:
            return 0, _pairs(None)
        if key in m:
            return 1, _pairs(m[key])
        return 2, _pairs(None)

    am, av = mode(allow_regions)
    mm, mv = mode(mask_regions)
    return _pairs(regions), np.ascontiguousarray(kept_col_indices, dtype=np.uint32), am, av, mm, mv


def _call_parse(fn, head, chr_, regions, kept_col_indices, min_gq, allow_regions, mask_regions, max_ploidy) -> VcfBatch:
    reg, kept, am, av, mm, mv = _parse_args(chr_, regions, kept_col_indices, allow_regions, mask_regions)
    h = C.c_void_p()
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    check(fn(*head, chr_.encode(), p(reg), len(reg), p(kept), len(kept), int(min_gq), am, p(av), len(av), mm, p(mv),
             len(mv), int(max_ploidy), C.byref(h)))
    return VcfBatch(h, chr_, int(kept.max()) if len(kept) else -1)


def process_lines(text: bytes, chr_: str, regions: Sequence[Tuple[int, int]], kept_col_indices: Sequence[int],
                  min_gq: int, allow_regions: Optional[Dict[str, Sequence[Tuple[int, int]]]] = None,
                  mask_regions: Optional[Dict[str, Sequence[Tuple[int, int]]]] = None, max_ploidy: int = 2) -> VcfBatch:
    """Data lines of a VCF (bytes, '\\n'-terminated) through the device parser.  regions are
    ZeroBasedHalfOpen (start, end) pairs; allow / mask maps are keyed by chromosome name without
    the chr prefix, as the reference's BED loaders store them."""
    if isinstance(text, str):
        text = text.encode()
    return _call_parse(lib().fm_vcf_parse, (text, len(text)), chr_, regions, kept_col_indices, min_gq, allow_regions,
                       mask_regions, max_ploidy)


def _scan_header(text: bytes, exclusion_set: Iterable[str]) -> Tuple[List[str], List[int], int]:
    """Header lines like process_vcf (:4181-4215): (sample names, kept column indices, offset of the first data
    line).  Raises when no sample remains."""
    off = 0
    names: List[str] = []
    kept: List[int] = []
    while off < len(text):
        nl = text.find(b"\n", off)
        end = len(text) if nl < 0 else nl + 1
        line = text[off:end]
        off = end
        if line.startswith(b"##"):
            continue
        if line.startswith(b"#CHROM"):
            names, kept = parse_header(line.decode(), exclusion_set)
            break
    if not names:
        raise VcfParseError("No samples remain after applying exclusions")
    return names, kept, off


def process_vcf_text(text: bytes, chr_: str, regions, min_gq: int, allow_regions=None, mask_regions=None,
                     exclusion_set: Iterable[str] = (), max_ploidy: int = 2) -> Tuple[VcfBatch, List[str]]:
    """A whole (uncompressed) VCF text: header handled like process_vcf (:4181-4215), data lines on the GPU."""
    if isinstance(text, str):
        text = text.encode()
    names, kept, off = _scan_header(text, exclusion_set)
    return process_lines(text[off:], chr_, regions, kept, min_gq, allow_regions, mask_regions, max_ploidy), names


# ------------------------------------------------------------------------------- BGZF input (.vcf.gz)
# bgzip / tabix write BGZF: independent gzip members of at most 64 KiB.  The device inflates them (fm_bgzf_inflate,
# fm_vcf_parse_bgzf), so only the compressed bytes cross the bus.  `data` is bytes or any contiguous bytes-like
# buffer (a numpy view of page-locked memory uploads without a bounce copy).
def _gz_buffer(data):
    if isinstance(data, bytes):
        return data, len(data)
    a = np.frombuffer(data, dtype=np.uint8)
    return a.ctypes.data_as(C.c_void_p), a.size


def _inflate_prefix(data, capacity: int) -> Tuple[bytes, int]:
    """(first min(capacity, total) inflated bytes, total inflated size)."""
    ptr, n = _gz_buffer(data)
    total = C.c_uint64()
    out = (C.c_uint8 * max(capacity, 1))()
    check(lib().fm_bgzf_inflate(ptr, n, out, capacity, C.byref(total)))
    return bytes(out)[:min(capacity, total.value)], total.value


def bgzf_inflate(data) -> bytes:
    """The whole inflated stream, decoded on the device."""
    ptr, n = _gz_buffer(data)
    total = C.c_uint64()
    check(lib().fm_bgzf_inflate(ptr, n, None, 0, C.byref(total)))
    return _inflate_prefix(data, total.value)[0]


def read_bgzf_header(data) -> Tuple[bytes, int]:
    """(header bytes up to and including the #CHROM line, offset of the first data line in the inflated stream).
    Inflates a prefix, doubling it until the #CHROM line ends (or the stream does)."""
    cap = 1 << 16
    while True:
        head, total = _inflate_prefix(data, cap)
        at = 0 if head.startswith(b"#CHROM") else head.find(b"\n#CHROM") + 1
        nl = head.find(b"\n", at) if at > 0 or head.startswith(b"#CHROM") else -1
        if nl >= 0:
            return head[:nl + 1], nl + 1
        if len(head) >= total:
            return head, len(head)
        cap *= 2


def process_vcf_bgzf(data, chr_: str, regions, min_gq: int, allow_regions=None, mask_regions=None,
                     exclusion_set: Iterable[str] = (), max_ploidy: int = 2) -> Tuple[VcfBatch, List[str]]:
    """process_vcf_text for a BGZF-compressed VCF (.vcf.gz as bgzip writes it): the same header rules, the same
    VcfBatch; the members are inflated and parsed on the device."""
    header, _ = read_bgzf_header(data)
    names, kept, off = _scan_header(header, exclusion_set)
    ptr, n = _gz_buffer(data)
    return _call_parse(lib().fm_vcf_parse_bgzf, (ptr, n, off), chr_, regions, kept, min_gq, allow_regions,
                       mask_regions, max_ploidy), names


# ------------------------------------------------------------------------------- multi-GPU (SURVEY §8e)
# The stage shards by LINE range: every line is independent, FilteringStats / MissingDataInfo counters add,
# the two position sets union, and the sorted variant lists of consecutive ranks concatenate (a position-sorted
# VCF gives every rank a contiguous site range, which is exactly how the estimator path shards).  Each rank
# uploads its own byte range over its own PCIe link; only the few counters travel.
STAT_KEYS = ("total_variants", "filtered_variants", "filtered_due_to_mask", "filtered_due_to_allow",
             "missing_data_variants", "low_gq_variants", "mnp_variants", "total_data_points", "missing_data_points")


def text_shard_bounds(text: bytes, world: int) -> List[int]:
    """Cut points of `world` contiguous byte ranges of data-line text, each ending on a line end."""
    n = len(text)
    cuts = [0]
    for r in range(1, world):
        c = max(n * r // world, cuts[-1])
        nl = text.find(b"\n", c - 1) if c > 0 else -1  # a cut right after a '\n' stays where it is
        c = n if nl < 0 else nl + 1
        cuts.append(min(max(c, cuts[-1]), n))
    cuts.append(n)
    return cuts


def merge_shard_stats(per_rank_counters: Sequence[Sequence[int]], per_rank_missing: Sequence[np.ndarray],
                      per_rank_filtered: Sequence[np.ndarray]) -> Tuple[Dict[str, int], np.ndarray, np.ndarray]:
    """Totals of a sharded parse: counters add in rank order, position sets union (sorted)."""
    tot = np.zeros(len(STAT_KEYS), dtype=np.int64)
    for c in per_rank_counters:
        tot += np.asarray(c, dtype=np.int64)
    pm = np.unique(np.concatenate([np.asarray(x, dtype=np.int64) for x in per_rank_missing] or [np.zeros(0, np.int64)]))
    pf = np.unique(np.concatenate([np.asarray(x, dtype=np.int64) for x in per_rank_filtered] or [np.zeros(0, np.int64)]))
    return {k: int(v) for k, v in zip(STAT_KEYS, tot)}, pm, pf


def gather_shard_stats(counters: Sequence[int], n_lines: int, pos_missing, pos_filtered, group=None):
    """The exchange step of a line-sharded parse under torch.distributed: ONE all_gather of each rank's nine counters,
    its line count and its two (small) position lists; merged in rank order on every rank.  Returns (global stats,
    positions_with_missing, filtered_positions, first global line index of this rank)."""
    import torch.distributed as dist
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    payload = (list(map(int, counters)) + [int(n_lines)], np.asarray(pos_missing), np.asarray(pos_filtered))
    gathered: List = [None] * world
    dist.all_gather_object(gathered, payload, group=group)
    stats, pm, pf = merge_shard_stats([g[0][:-1] for g in gathered], [g[1] for g in gathered], [g[2] for g in gathered])
    return stats, pm, pf, sum(g[0][-1] for g in gathered[:rank])


def process_lines_sharded(text: bytes, chr_: str, regions, kept_col_indices, min_gq, allow_regions=None,
                          mask_regions=None, max_ploidy: int = 2, group=None):
    """One rank of a line-sharded parse (one process per GPU).  Returns (this rank's VcfBatch, global stats dict,
    global positions_with_missing, global filtered_positions, first global line index of this rank)."""
    import torch.distributed as dist
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    cuts = text_shard_bounds(text, world)
    batch = process_lines(text[cuts[rank]:cuts[rank + 1]], chr_, regions, kept_col_indices, min_gq, allow_regions,
                          mask_regions, max_ploidy)
    s = batch.stats()
    stats, pm, pf, line0 = gather_shard_stats([s[k] for k in STAT_KEYS], int(batch.info.n_lines),
                                              batch.positions_with_missing(), batch.filtered_positions(), group)
    return batch, stats, pm, pf, line0
