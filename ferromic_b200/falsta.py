"""FALSTA per-site track writers fed by the GPU (SURVEY §8f rank 3).

Mirrors `append_diversity_falsta` / `append_fst_falsta` (process.rs:3740-4002): same headers,
same track order, same "omit a diversity track without records" rule, the same gzip-append file
convention.  The track bodies -- region_len comma-joined tokens per line, the O(tracks x sites)
string work of the reference -- are rendered on the device by `fm_falsta_tracks`
(scatter -> token lengths -> exclusive scan -> write); the host only splices headers in.

With `bgzf=True` a writer appends BGZF members instead of one gzip member per call: the device renders the headed
text and deflates it (`fm_falsta_tracks_bgzf`), so the text never crosses the bus uncompressed and no host gzip pass
runs.  The file decompresses to the same text; gzip.open, zcat and flate2's MultiGzDecoder read either form."""
from __future__ import annotations

import ctypes as C
import gzip
from typing import List, Sequence, Tuple

import numpy as np

from ._lib import check, lib

DIVERSITY, FST, TSV = 0, 1, 2  # FM_FALSTA_DIVERSITY / FM_FALSTA_FST / FM_FALSTA_TSV


def format_value(value: float, mode: int = FST) -> str:
    """One token exactly as the device renders it (host instance of the same routine)."""
    buf = C.create_string_buffer(64)
    n = C.c_size_t(0)
    check(lib().fm_falsta_format_value(float(value), mode, buf, 64, C.byref(n)))
    return buf.raw[: n.value].decode("ascii")


_SCRATCH = [np.empty(0, dtype=np.uint8)]


def _scratch(n: int) -> np.ndarray:
    """Grow-only host buffer for the rendered text: a writer renders track after track of similar size, and
    first-touch page faults of a fresh 100 MB buffer cost several times the rendering itself."""
    if _SCRATCH[0].size < n:
        _SCRATCH[0] = np.empty(int(n * 1.25) + 4096, dtype=np.uint8)
    return _SCRATCH[0]


def track_lines(pos1, values, region_start: int, region_end: int, mode: int) -> List[bytes]:
    """Bodies of the tracks `values[t]` (all sharing the 1-based record positions `pos1`)."""
    pos1 = np.ascontiguousarray(pos1, dtype=np.int64)
    values = np.ascontiguousarray(values, dtype=np.float64)
    if values.ndim == 1:
        values = values[None, :]
    T, n = values.shape
    if n != pos1.shape[0]:
        raise ValueError("values and positions differ in length")
    L = lib()
    total = C.c_size_t(0)
    lens = (C.c_size_t * T)()
    pp = pos1.ctypes.data_as(C.c_void_p)
    vp = values.ctypes.data_as(C.c_void_p)
    # one call with a generous capacity (default tokens are 1-2 bytes, `{:.6}` of these statistics stays far below
    # 24 bytes); an exact-length query + second call only if that was not enough
    s1 = max(region_start, 1)
    region_len = max(region_end, s1) - s1 + 1
    cap = T * (3 * region_len + 26 * min(n, region_len)) + 16
    out = _scratch(cap)  # not zero-filled: the library writes every byte it reports
    st = L.fm_falsta_tracks(pp, vp, n, T, region_start, region_end, mode, out.ctypes.data_as(C.c_void_p), cap, lens,
                            C.byref(total))
    if st != 0 and total.value > cap:
        out = _scratch(total.value)
        st = L.fm_falsta_tracks(pp, vp, n, T, region_start, region_end, mode, out.ctypes.data_as(C.c_void_p),
                                total.value, lens, C.byref(total))
    check(st)
    lines, o = [], 0
    for t in range(T):
        lines.append(out[o : o + lens[t]].tobytes())
        o += lens[t] + 1
    return lines


def _render_text(pos1, values, region_start: int, region_end: int, mode: int, heads: Sequence[str]) -> bytes:
    """heads[t] + line t + '\n' for every track."""
    lines = track_lines(pos1, values, region_start, region_end, mode)
    return b"".join(h.encode() + line + b"\n" for h, line in zip(heads, lines))


def _render_bgzf(pos1, values, region_start: int, region_end: int, mode: int, heads: Sequence[str]) -> bytes:
    """What _render_text gives, as BGZF members (no EOF member) rendered and deflated on the device."""
    pos1 = np.ascontiguousarray(pos1, dtype=np.int64)
    values = np.ascontiguousarray(values, dtype=np.float64)
    if values.ndim == 1:
        values = values[None, :]
    T, n = values.shape
    if n != pos1.shape[0]:
        raise ValueError("values and positions differ in length")
    enc = [h.encode() for h in heads]
    if len(enc) != T:
        raise ValueError("one head per track")
    c_heads = (C.c_char_p * T)(*enc)
    L = lib()
    s1 = max(region_start, 1)
    region_len = max(region_end, s1) - s1 + 1
    text = T * (3 * region_len + 26 * min(n, region_len)) + sum(map(len, enc)) + 16  # as in track_lines
    bound = C.c_size_t(0)
    check(L.fm_bgzf_deflate_bound(text, 0, C.byref(bound)))
    out = _scratch(bound.value)
    size = C.c_size_t(0)
    args = (pos1.ctypes.data_as(C.c_void_p), values.ctypes.data_as(C.c_void_p), n, T, region_start, region_end, mode,
            C.cast(c_heads, C.c_void_p))
    st = L.fm_falsta_tracks_bgzf(*args, out.ctypes.data_as(C.c_void_p), bound.value, C.byref(size))
    if st != 0 and size.value > bound.value:
        out = _scratch(size.value)
        st = L.fm_falsta_tracks_bgzf(*args, out.ctypes.data_as(C.c_void_p), size.value, C.byref(size))
    check(st)
    return out[: size.value].tobytes()


def _in_region(pos1: np.ndarray, region_start: int, region_end: int) -> np.ndarray:
    # from_1based_inclusive + relative_position_1based_inclusive (process.rs:193-206, 314-321)
    s1 = max(region_start, 1)
    e1 = max(region_end, s1)
    return (pos1 >= s1) & (pos1 <= e1)


def diversity_falsta_text(seqname: str, region_start: int, region_end: int,
                          per_site: Sequence[Tuple[int, float, float, int, bool]]) -> bytes:
    """Text `append_diversity_falsta` appends for one region (process.rs:3740-3806).
    per_site records: (pos_1based, pi, theta, group_id, is_filtered)."""
    return _diversity(seqname, region_start, region_end, per_site, _render_text)


def _diversity(seqname, region_start, region_end, per_site, render) -> bytes:
    if len(per_site) == 0:
        return b""
    pos = np.array([r[0] for r in per_site], dtype=np.int64)
    pi = np.array([r[1] for r in per_site], dtype=np.float64)
    th = np.array([r[2] for r in per_site], dtype=np.float64)
    gid = np.array([r[3] for r in per_site], dtype=np.int64)
    flt = np.array([bool(r[4]) for r in per_site], dtype=bool)
    inside = _in_region(pos, region_start, region_end)
    out = []
    for g in sorted(set(gid.tolist())):  # BTreeSet<u8> order
        for is_filtered, prefix in ((False, "unfiltered_"), (True, "filtered_")):  # pi then theta of each
            sel = (gid == g) & (flt == is_filtered)
            if not np.any(sel & inside):
                continue  # `any` stays false: the track is omitted
            heads = [f">{prefix}{stat}_chr_{seqname}_start_{region_start}_end_{region_end}_group_{g}\n"
                     for stat in ("pi", "theta")]
            out.append(render(pos[sel], np.stack([pi[sel], th[sel]]), region_start, region_end, DIVERSITY, heads))
    return b"".join(out)


def fst_falsta_text(seqname: str, region_start: int, region_end: int,
                    wc_sites: Sequence[Tuple[int, float, float, float, float, float, float]],
                    hudson_sites: Sequence[Tuple[int, float, float, float]]) -> bytes:
    """Text `append_fst_falsta` appends for one region (process.rs:3809-4002).
    wc_sites records: (position_1based, overall_fst, overall_numerator, overall_denominator,
    pairwise_fst, pairwise_numerator, pairwise_denominator) -- PerSiteWcOutput;
    hudson_sites records: (position_1based, fst, numerator, denominator)."""
    return _fst(seqname, region_start, region_end, wc_sites, hudson_sites, _render_text)


def _fst(seqname, region_start, region_end, wc_sites, hudson_sites, render) -> bytes:
    if len(wc_sites) == 0 and len(hudson_sites) == 0:
        return b""
    tail = f"chr_{seqname}_start_{region_start}_end_{region_end}\n"
    out = []

    def emit(records, heads):
        arr = np.array(records, dtype=np.float64).reshape(len(records), len(heads) + 1)
        pos = np.array([int(r[0]) for r in records], dtype=np.int64)
        out.append(render(pos, np.ascontiguousarray(arr[:, 1:].T), region_start, region_end, FST,
                          [">" + h + tail for h in heads]))

    if len(wc_sites):
        emit(wc_sites, ("haplotype_overall_fst_summary_", "haplotype_overall_fst_numerator_",
                        "haplotype_overall_fst_denominator_", "haplotype_0v1_pairwise_fst_summary_",
                        "haplotype_0v1_pairwise_fst_numerator_", "haplotype_0v1_pairwise_fst_denominator_"))
    if len(hudson_sites):
        emit(hudson_sites, ("hudson_pairwise_fst_hap_0v1_", "hudson_pairwise_fst_hap_0v1_numerator_",
                            "hudson_pairwise_fst_hap_0v1_denominator_"))
    return b"".join(out)


def _csv_field(f: str) -> str:
    # csv::Writer, QuoteStyle::Necessary with a tab delimiter
    if any(c in f for c in '\t"\n\r'):
        return '"' + f.replace('"', '""') + '"'
    return f


def hudson_tsv_text(rows) -> bytes:
    """Rows `append_hudson_tsv` writes (process.rs:4006-4041): chr, region_start, region_end, pop1 type, pop1 name,
    pop2 type, pop2 name, d_xy, pi_pop1, pi_pop2, pi_xy_avg, fst.  rows: (chr, region_start, region_end, pop1_id,
    pop2_id, d_xy, pi_pop1, pi_pop2, pi_xy_avg, fst); a population id is None, an int (HaplotypeGroup) or a str
    (Named) (format_population_id, :3692-3698); None / NaN floats print "NA" (format_optional_float, :3702-3713)."""
    def pop(p):
        if p is None:
            return "NA", "NA"
        if isinstance(p, str):
            return "NamedPopulation", p
        return "HaplotypeGroup", str(int(p))

    def flt(v):
        return "NA" if v is None else format_value(v, TSV)

    out = []
    for chr_, rs, re_, p1, p2, dxy, pi1, pi2, pixy, fst in rows:
        f = [str(chr_), str(int(rs)), str(int(re_)), *pop(p1), *pop(p2), flt(dxy), flt(pi1), flt(pi2), flt(pixy), flt(fst)]
        out.append("\t".join(_csv_field(x) for x in f) + "\n")
    return "".join(out).encode()


def _append_gz(path, text: bytes) -> None:
    # open_append_compressed (process.rs:3723-3729): every call appends one gzip member
    with gzip.open(path, "ab") as f:
        f.write(text)


def _append_bytes(path, members: bytes) -> None:
    # BGZF members are complete gzip members already: a plain append
    with open(path, "ab") as f:
        f.write(members)


def append_diversity_falsta(path, seqname, region_start, region_end, per_site, bgzf: bool = False) -> None:
    if len(per_site) == 0:  # process.rs:3745-3754: warns and returns before the file is opened
        return
    if bgzf:
        _append_bytes(path, _diversity(seqname, region_start, region_end, per_site, _render_bgzf))
    else:
        _append_gz(path, diversity_falsta_text(seqname, region_start, region_end, per_site))


def append_hudson_tsv(path, rows, bgzf: bool = False) -> None:
    if bgzf:
        from .vcf import bgzf_deflate
        _append_bytes(path, bgzf_deflate(hudson_tsv_text(rows), eof=False))
    else:
        _append_gz(path, hudson_tsv_text(rows))


def append_fst_falsta(path, seqname, region_start, region_end, wc_sites, hudson_sites, bgzf: bool = False) -> None:
    if len(wc_sites) == 0 and len(hudson_sites) == 0:  # process.rs:3835-3837
        return
    if bgzf:
        _append_bytes(path, _fst(seqname, region_start, region_end, wc_sites, hudson_sites, _render_bgzf))
    else:
        _append_gz(path, fst_falsta_text(seqname, region_start, region_end, wc_sites, hudson_sites))
