"""Host-side mirror of the reference's Python surface (`ferromic`, src/lib.rs) on top of the
C-ABI GPU library.  Names, argument meaning, return classes and error behaviour follow the PyO3
bindings (lib.rs:75-165, 259-814, 1082-1778, 2190-2225) so the reference's own pytests can be
pointed at `import ferromic_b200 as fm`.  All estimator arithmetic runs on the GPU through
libferromic_gpu.so; this module only does what lib.rs does on the host: parsing Python inputs
into genotype arrays, building haplotype memberships and choosing the code path the reference
would take (dense summary / dense / sparse)."""
from __future__ import annotations

import ctypes as C
import os
import math
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from ._lib import check, lib

MISSING = 0xFF  # process.rs:438
_U16_INVALID = 0xFFFF  # stats.rs:1080


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


# --------------------------------------------------------------------------- input parsing
def _field(obj, names):
    """extract_optional_field (lib.rs:1369-1379): item access first, then attribute."""
    for n in names:
        try:
            return obj[n]
        except Exception:
            pass
        if hasattr(obj, n):
            return getattr(obj, n)
    return None


def _parse_side(x) -> int:  # lib.rs:1334-1367
    if isinstance(x, (int, np.integer)) and not isinstance(x, bool):
        if int(x) in (0, 1):
            return int(x)
        raise ValueError("haplotype side must be 0 or 1")
    if isinstance(x, str):
        t = x.lower()
        if t in ("l", "left", "0"):
            return 0
        if t in ("r", "right", "1"):
            return 1
        raise ValueError("haplotype side must be one of 0, 1, 'L', 'R', 'left', 'right'")
    raise ValueError("haplotype side must be 0/1 or a left/right string")


def _parse_haplotypes(haplotypes) -> List[Tuple[int, int]]:  # lib.rs:887-923
    out = []
    for h in haplotypes:
        if isinstance(h, (tuple, list)):
            if len(h) < 2:
                raise ValueError("haplotypes must contain (sample_index, side)")
            idx, side = h[0], h[1]
        else:
            idx = _field(h, ("sample_index", "sample", "index"))
            side = _field(h, ("side", "haplotype", "haplotype_side"))
            if idx is None:
                raise ValueError("haplotype missing sample index")
            if side is None:
                raise ValueError("haplotype missing side")
        idx = int(idx)
        if idx < 0:
            raise OverflowError("can't convert negative int to unsigned")
        out.append((idx, _parse_side(side)))
    return out


class _Variants:
    """Sparse variants with CompressedGenotypes semantics (process.rs:430-536):
    gt[V, S, stride] u8, 0xFF in slot 0 = None, a later 0xFF ends the genotype."""

    def __init__(self, positions: np.ndarray, gt: np.ndarray, first_len: Optional[int] = None):
        self.positions = np.ascontiguousarray(positions, dtype=np.int64)
        self.gt = np.ascontiguousarray(gt, dtype=np.uint8)
        self.first_len = self.gt.shape[1] if first_len is None else first_len
        self._dense_cache: Dict[int, object] = {}

    @property
    def n_variants(self) -> int:
        return self.gt.shape[0]

    @property
    def n_samples(self) -> int:
        return self.gt.shape[1]


def _parse_variants(variants) -> _Variants:  # lib.rs:834-873, 1301-1332
    if isinstance(variants, _Variants):
        return variants
    pos, rows = [], []
    for v in variants:
        if isinstance(v, tuple):
            if len(v) != 2:
                raise ValueError("variant tuples must have length 2: (position, genotypes)")
            p, g = v
        else:
            p = _field(v, ("position", "pos", "site"))
            g = _field(v, ("genotypes", "calls"))
            if p is None:
                raise ValueError("variant is missing a position")
            if g is None:
                raise ValueError("variant is missing genotypes")
        pos.append(int(p))
        rows.append(list(g))
    S = max((len(r) for r in rows), default=0)
    stride = 1
    for r in rows:
        for g in r:
            if g is not None and not isinstance(g, (int, np.integer)):
                stride = max(stride, len(g))
    gt = np.full((len(rows), S, stride), MISSING, dtype=np.uint8)
    for vi, r in enumerate(rows):
        for si, g in enumerate(r):
            if g is None:
                continue
            if isinstance(g, (int, np.integer)):
                g = (g,)
            for k, a in enumerate(g):
                a = int(a)
                if not 0 <= a <= 255:
                    raise OverflowError("allele values must fit in u8")
                gt[vi, si, k] = a
    return _Variants(np.asarray(pos, dtype=np.int64), gt, first_len=len(rows[0]) if rows else 0)


def _pack_bits(mask_flat: np.ndarray) -> np.ndarray:
    total = mask_flat.size
    words = (total + 63) // 64
    padded = np.zeros(words * 64, dtype=np.uint8)
    padded[:total] = mask_flat
    return np.packbits(padded.reshape(words, 64), axis=1, bitorder="little").view(np.uint64).reshape(-1)


def _ingest_mode(max_allele: int) -> str:
    """How a host matrix reaches the device: "packed" (2 bits per genotype: the library's multi-threaded
    packer fm_pack_rows + fm_matrix_create_packed, biallelic matrices) or "u8" (the reference layout as it
    is, repacked on the device).  FERROMIC_GPU_INGEST overrides the default ("packed" when possible)."""
    mode = os.environ.get("FERROMIC_GPU_INGEST", "packed")
    if mode not in ("packed", "u8"):
        raise ValueError("FERROMIC_GPU_INGEST must be 'packed' or 'u8'")
    return mode if max_allele <= 1 else "u8"


def pack_rows(alleles2d: np.ndarray, missing_mode: int, bitmap: Optional[np.ndarray] = None, first_row: int = 0,
              n_total_rows: Optional[int] = None, threads: int = 0, generic: bool = False):
    """fm_pack_rows over a [rows, stride] u8 block -> (allele_bits, called_bits or None), each
    [rows, ceil(stride / 32)] u32 (SURVEY 8 f1: the 2-bit ingest format)."""
    a = np.ascontiguousarray(alleles2d).view(np.uint8)
    assert a.ndim == 2
    rows, stride = a.shape
    rw = (stride + 31) // 32
    ab = np.zeros((rows, rw), dtype=np.uint32)
    cb = np.zeros((rows, rw), dtype=np.uint32) if missing_mode != 0 else None
    total = rows + first_row if n_total_rows is None else n_total_rows
    L = lib()
    if generic:
        check(L.fm_pack_rows_generic(_ptr(a), _ptr(bitmap), missing_mode, first_row, rows, total, stride, _ptr(ab),
                                     _ptr(cb)))
    else:
        check(L.fm_pack_rows(_ptr(a), _ptr(bitmap), missing_mode, first_row, rows, total, stride, _ptr(ab), _ptr(cb),
                             threads))
    return ab, cb


# The sparse missing list of packed rows goes over PCIe as one-byte gap codes (include/ferromic_gpu.h) unless this is
# switched off (tests cover both forms).
SPARSE_GAP_CODE = True


def pack_rows_sparse(alleles2d: np.ndarray, missing_mode: int, bitmap: Optional[np.ndarray] = None, first_row: int = 0,
                     n_total_rows: Optional[int] = None, threads: int = 0, gap_code: bool = False):
    """fm_pack_rows_sparse: (allele_bits [rows, rw] u32, row_start [rows + 1] u64, missing_cols) -- the packed rows
    with a sparse missing list instead of a called plane.  missing_cols holds u16 / u32 column indices, or with
    gap_code=True the one-byte gap code (col_bytes == 1)."""
    a = np.ascontiguousarray(alleles2d).view(np.uint8)
    assert a.ndim == 2
    rows, stride = a.shape
    rw = (stride + 31) // 32
    ab = np.zeros((rows, rw), dtype=np.uint32)
    start = np.zeros(rows + 1, dtype=np.uint64)
    col_t = np.uint8 if gap_code else (np.uint16 if stride <= 65536 else np.uint32)
    total = rows + first_row if n_total_rows is None else n_total_rows
    L = lib()
    need = C.c_size_t()
    cols = np.zeros(max(16, rows * stride // 32), dtype=col_t)
    for _ in range(2):
        st = L.fm_pack_rows_sparse(_ptr(a), _ptr(bitmap), missing_mode, first_row, rows, total, stride, _ptr(ab),
                                   _ptr(start), _ptr(cols), cols.size, cols.itemsize, threads, C.byref(need))
        if st == _lib.FM_ERR_INVALID_ARG and need.value > cols.size:
            cols = np.zeros(need.value, dtype=col_t)  # the first call reported the size: retry
            continue
        check(st)
        break
    return ab, start, cols[:need.value]


def _sparse_missing_pays(missing_mask: Optional[np.ndarray]) -> bool:
    """The sparse list (2-4 bytes per missing cell) beats the called plane (1 bit per cell) below ~3 % missing."""
    return missing_mask is not None and missing_mask.size > 0 and float(missing_mask.mean()) < 1.0 / 40.0


# --------------------------------------------------------------------------- device handles
class _Matrix:
    def __init__(self, alleles: np.ndarray, missing_mask: Optional[np.ndarray], positions: np.ndarray,
                 max_allele: Optional[int] = None, always_bitmap: bool = False, ingest: Optional[str] = None):
        a = np.ascontiguousarray(alleles, dtype=np.uint8)
        assert a.ndim == 3
        self.V, self.S, self.P = a.shape
        bits = None
        if missing_mask is not None and (always_bitmap or missing_mask.any()):
            bits = _pack_bits(np.ascontiguousarray(missing_mask, dtype=np.uint8).reshape(-1))
        self.has_missing = bits is not None
        self.max_allele = int(a.max()) if (max_allele is None and a.size) else int(max_allele or 0)
        pos = np.ascontiguousarray(positions, dtype=np.int64)
        h = C.c_void_p()
        self.ingest_mode = ingest or _ingest_mode(self.max_allele)
        if self.ingest_mode in ("packed", "packed-dense", "packed-sparse"):
            # convert_numeric_array / from_variants seam (lib.rs:1135-1227, stats.rs:339-500): the host packs
            # bit words (several threads) and only 0.25 B per genotype cross PCIe ("packed-dense" keeps the called
            # plane even when the sparse missing list would be smaller)
            flat = a.reshape(self.V, self.S * self.P)
            if bits is not None and (self.ingest_mode == "packed-sparse" or
                                     (self.ingest_mode == "packed" and _sparse_missing_pays(missing_mask))):
                ab, start, cols = pack_rows_sparse(flat, 1, bits, gap_code=SPARSE_GAP_CODE)
                check(lib().fm_matrix_create_packed_sparse(_ptr(ab), _ptr(start), _ptr(cols), cols.itemsize, self.V, self.S,
                                                           self.P, _ptr(pos), C.byref(h)))
                self.ingest_mode = "packed-sparse"
            else:
                ab, cb = pack_rows(flat, 1 if bits is not None else 0, bits)
                check(lib().fm_matrix_create_packed(_ptr(ab), _ptr(cb), self.V, self.S, self.P, _ptr(pos), C.byref(h)))
        else:
            check(lib().fm_matrix_create(_ptr(a), _ptr(bits), self.V, self.S, self.P, self.max_allele, _ptr(pos),
                                         C.byref(h)))
        self.handle = h
        self._groups: Dict[tuple, "_Group"] = {}

    @classmethod
    def from_int8(cls, genotypes: np.ndarray, positions: np.ndarray, max_allele: int,
                  ingest: Optional[str] = None) -> "_Matrix":
        """Dense matrix straight from the caller's int8 array (negative = missing): the buffer is
        uploaded as it is and missingness stays in band (fm_matrix_create_inband) -- no host-side
        conversion pass, no bitmap packing (lib.rs:1135-1227 does both serially)."""
        g = np.ascontiguousarray(genotypes)
        assert g.ndim == 3 and g.dtype == np.int8
        self = cls.__new__(cls)
        self.V, self.S, self.P = g.shape
        self.has_missing = True
        self.max_allele = int(max_allele)
        pos = np.ascontiguousarray(positions, dtype=np.int64)
        h = C.c_void_p()
        self.ingest_mode = ingest or _ingest_mode(self.max_allele)
        if self.ingest_mode == "packed":  # packed straight from the int8 cells: sign bit = missing
            ab, cb = pack_rows(g.reshape(self.V, self.S * self.P), 2)
            check(lib().fm_matrix_create_packed(_ptr(ab), _ptr(cb), self.V, self.S, self.P, _ptr(pos), C.byref(h)))
        else:
            check(lib().fm_matrix_create_inband(g.ctypes.data, self.V, self.S, self.P, self.max_allele, _ptr(pos),
                                                C.byref(h)))
        self.handle = h
        self._groups = {}
        return self

    @classmethod
    def ingest(cls, alleles: np.ndarray, missing_mask: Optional[np.ndarray], positions: np.ndarray,
               group_haplotypes: Sequence[Sequence[Tuple[int, int]]], partitions=(), chunk_rows: int = 0,
               calls: int = 1, always_bitmap: bool = False, packed: bool = False, sparse: bool = False,
               tracks: Optional[dict] = None) -> "_Matrix":
        """Streaming ingestion (fm_ingest_*): the u8 rows are uploaded in chunks and repacked into
        the declared groups' bitplanes while the next chunk is in flight; the u8 matrix is never
        resident.  partitions: (left, right, n_groups) triples; their handles land in
        `self.partitions`.  calls > 1 pushes the rows in several fm_ingest_rows calls.  packed: False (u8 rows over
        PCIe), True (bit rows packed by the caller with fm_pack_rows / _sparse) or "library" (fm_ingest_rows_pack).
        tracks: per-site pi / theta of declared groups computed while the rows arrive (fm_ingest_request_tracks):
        {"groups": [indices], "raw_n": [...], "region": (start, end), "mask": int64 [k, 2] or None,
        "filtered": int64 [m] or None, "pos": int64 [cap], "pi": f64 [n_groups, cap], "theta": f64 [n_groups, cap]}
        (arrays or raw addresses); the number of sites lands in `self.track_sites`."""
        a = np.ascontiguousarray(alleles, dtype=np.uint8)
        assert a.ndim == 3
        self = cls.__new__(cls)
        self.V, self.S, self.P = a.shape
        bits = None
        if missing_mask is not None and (always_bitmap or missing_mask.any()):
            bits = _pack_bits(np.ascontiguousarray(missing_mask, dtype=np.uint8).reshape(-1))
        self.has_missing = bits is not None
        self.max_allele = int(a.max()) if a.size else 0
        pos = np.ascontiguousarray(positions, dtype=np.int64)
        self._groups = {}
        self.partitions = []
        self.handle = None
        L = lib()
        ih = C.c_void_p()
        check(L.fm_ingest_begin(self.V, self.S, self.P, int(self.has_missing), self.max_allele, _ptr(pos),
                                chunk_rows, C.byref(ih)))
        try:
            for haps in group_haplotypes:
                idx = np.asarray([h[0] for h in haps], dtype=np.uint64)
                side = np.asarray([h[1] for h in haps], dtype=np.uint8)
                check(L.fm_ingest_add_group(ih, _ptr(idx), _ptr(side), len(haps), None))
            for left, right, ng in partitions:
                lft = np.ascontiguousarray(left, dtype=np.uint16)
                rgt = np.ascontiguousarray(right, dtype=np.uint16)
                check(L.fm_ingest_add_partition(ih, _ptr(lft), _ptr(rgt), len(lft), ng, None))
            self.track_sites = None
            if tracks is not None:
                def addr(x):
                    return x if (x is None or isinstance(x, int)) else x.ctypes.data
                gi = np.ascontiguousarray(tracks["groups"], dtype=np.uint64)
                rn = np.ascontiguousarray(tracks["raw_n"], dtype=np.uint64)
                mk = tracks.get("mask")
                mk = None if mk is None else np.ascontiguousarray(mk, dtype=np.int64).reshape(-1)
                fl = tracks.get("filtered")
                fl = None if fl is None else np.ascontiguousarray(fl, dtype=np.int64)
                n = C.c_size_t()
                check(L.fm_ingest_request_tracks(ih, _ptr(gi), _ptr(rn), len(gi), int(tracks["region"][0]),
                                                 int(tracks["region"][1]), _ptr(mk), 0 if mk is None else mk.size // 2,
                                                 _ptr(fl), 0 if fl is None else fl.size, addr(tracks.get("pos")),
                                                 addr(tracks["pi"]), addr(tracks["theta"]), int(tracks["capacity"]),
                                                 C.byref(n)))
                self.track_sites = n.value
            flat = a.reshape(self.V, -1)
            cuts = np.linspace(0, self.V, max(1, calls) + 1).astype(int)
            for r0, r1 in zip(cuts[:-1], cuts[1:]):
                if r1 <= r0:
                    continue
                if packed and sparse and bits is not None:  # allele bits + sparse missing list
                    ab, start, cols = pack_rows_sparse(flat[r0:r1], 1, bits, first_row=int(r0), n_total_rows=self.V,
                                                       gap_code=SPARSE_GAP_CODE)
                    check(L.fm_ingest_rows_packed_sparse(ih, _ptr(ab), _ptr(start), _ptr(cols), cols.itemsize, int(r0),
                                                         int(r1 - r0)))
                elif packed == "library":  # u8 rows in, packed inside the call while the previous chunk uploads
                    check(L.fm_ingest_rows_pack(ih, flat[r0:r1].ctypes.data, _ptr(bits), int(r0), int(r1 - r0), 0))
                elif packed:  # fm_pack_rows on the host, 2 bits per genotype over PCIe (fm_ingest_rows_packed)
                    ab, cb = pack_rows(flat[r0:r1], 1 if bits is not None else 0, bits, first_row=int(r0),
                                       n_total_rows=self.V)
                    check(L.fm_ingest_rows_packed(ih, _ptr(ab), _ptr(cb), int(r0), int(r1 - r0)))
                else:
                    check(L.fm_ingest_rows(ih, flat[r0:r1].ctypes.data, _ptr(bits), int(r0), int(r1 - r0)))
            mh = C.c_void_p()
            gh = (C.c_void_p * max(1, len(group_haplotypes)))()
            ph = (C.c_void_p * max(1, len(partitions)))()
            check(L.fm_ingest_finish(ih, C.byref(mh), gh, ph))
            ih = None
        finally:
            if ih is not None:
                L.fm_ingest_abort(ih)
        self.handle = mh
        for i, haps in enumerate(group_haplotypes):
            self._groups[tuple(haps)] = _Group._adopt(self, haps, C.c_void_p(gh[i]))
        self.partitions = [C.c_void_p(ph[i]) for i in range(len(partitions))]
        return self

    def group(self, haplotypes: Sequence[Tuple[int, int]]) -> "_Group":
        key = tuple(haplotypes)
        g = self._groups.get(key)
        if g is None:
            g = _Group(self, haplotypes)
            self._groups[key] = g
        return g

    def groups(self, lists: Sequence[Sequence[Tuple[int, int]]]) -> List["_Group"]:
        """Several groups in one pass over the u8 rows (fm_groups_create); cached like `group`."""
        todo = [tuple(h) for h in lists if tuple(h) not in self._groups]
        todo = list(dict.fromkeys(todo))
        if len(todo) > 1:
            idx = np.asarray([h[0] for hs in todo for h in hs], dtype=np.uint64)
            side = np.asarray([h[1] for hs in todo for h in hs], dtype=np.uint8)
            sizes = (C.c_size_t * len(todo))(*[len(hs) for hs in todo])
            out = (C.c_void_p * len(todo))()
            check(lib().fm_groups_create(self.handle, _ptr(idx), _ptr(side), sizes, len(todo), out))
            for hs, h in zip(todo, out):
                self._groups[hs] = _Group._adopt(self, hs, C.c_void_p(h))
        return [self.group(h) for h in lists]

    def __del__(self):
        try:
            self._groups.clear()
            for ph in getattr(self, "partitions", []):
                lib().fm_partition_release(ph)
            self.partitions = []
            if getattr(self, "handle", None):
                lib().fm_matrix_release(self.handle)
                self.handle = None
        except Exception:
            pass


class _Group:
    def __init__(self, matrix: _Matrix, haplotypes: Sequence[Tuple[int, int]]):
        self.matrix = matrix
        self.raw_n = len(haplotypes)
        idx = np.asarray([h[0] for h in haplotypes], dtype=np.uint64)
        side = np.asarray([h[1] for h in haplotypes], dtype=np.uint8)
        h = C.c_void_p()
        check(lib().fm_group_create(matrix.handle, _ptr(idx), _ptr(side), len(haplotypes), C.byref(h)))
        self.handle = h

    @classmethod
    def _adopt(cls, matrix: _Matrix, haplotypes, handle) -> "_Group":
        self = cls.__new__(cls)
        self.matrix = matrix
        self.raw_n = len(haplotypes)
        self.handle = handle
        return self

    @property
    def capacity(self) -> int:
        c = C.c_size_t()
        check(lib().fm_group_capacity(self.handle, C.byref(c)))
        return c.value

    def summary(self, want_arrays: bool = False):
        V = self.matrix.V
        alt = np.zeros(V, dtype=np.uint32) if want_arrays else None
        called = np.zeros(V, dtype=np.uint32) if want_arrays else None
        seg, unc, pi = C.c_uint64(), C.c_uint64(), C.c_double()
        check(lib().fm_group_summary(self.handle, _ptr(alt), _ptr(called), C.byref(seg), C.byref(pi),
                                     C.byref(unc)))
        return dict(alt=alt, called=called, segregating_sites=seg.value, pi_sum=pi.value,
                    uncallable_lt2=unc.value)

    def segregating_sites(self) -> int:
        out = C.c_uint64()
        check(lib().fm_group_segregating_sites(self.handle, C.byref(out)))
        return out.value

    def pi(self, L: int, path: int, raw_n: Optional[int] = None) -> float:
        out = C.c_double()
        check(lib().fm_group_pi(self.handle, L, path, self.raw_n if raw_n is None else raw_n, C.byref(out)))
        return out.value

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                lib().fm_group_release(self.handle)
                self.handle = None
        except Exception:
            pass


def _dense_from_variants(vs: _Variants, sample_count: int):
    """DenseGenotypeMatrix::from_variants (stats.rs:339-500) as arrays: (alleles, missing mask)."""
    if vs.n_variants == 0:
        return None
    valid = np.logical_and.accumulate(vs.gt != MISSING, axis=2)
    found = int(valid.sum(axis=2).max()) if valid.size else 0
    if found == 0:
        return None
    # The sparse paths test membership with HapMembership (Left / Right per sample, stats.rs:1211-1238),
    # which counts a Right haplotype even when every genotype is haploid; keep two sides so that the
    # group capacity equals HapMembership::total and the absent side is simply missing.
    ploidy = max(found, 2)
    V, S = vs.n_variants, vs.n_samples
    alle = np.zeros((V, sample_count, ploidy), dtype=np.uint8)
    miss = np.ones((V, sample_count, ploidy), dtype=bool)
    k = min(S, sample_count)
    alle[:, :k, :found] = np.where(valid[:, :k, :found], vs.gt[:, :k, :found], 0)
    miss[:, :k, :found] = ~valid[:, :k, :found]
    return alle, miss


def _sparse_matrix(vs: _Variants, sample_count: Optional[int] = None) -> Optional[_Matrix]:
    """Device matrix carrying the sparse (from_variants) missingness of `vs`."""
    sc = vs.n_samples if sample_count is None else sample_count
    m = vs._dense_cache.get(sc)
    if m is None:
        d = _dense_from_variants(vs, sc)
        if d is None:
            # no genotype data at all: an all-missing two-sided matrix keeps every count at zero
            alle = np.zeros((vs.n_variants, sc, 2), dtype=np.uint8)
            miss = np.ones((vs.n_variants, sc, 2), dtype=bool)
            d = (alle, miss)
        m = _Matrix(d[0], d[1], vs.positions, always_bitmap=True)
        vs._dense_cache[sc] = m
    return m


# --------------------------------------------------------------------------- result classes
class FstEstimate:  # lib.rs:75-165
    __slots__ = ("state", "value", "sum_a", "sum_b", "sites")
    _STATES = ("calculable", "components_yield_indeterminate_ratio", "no_inter_population_variance",
               "insufficient_data_for_estimation")

    def __init__(self, state, value, sum_a, sum_b, sites):
        self.state, self.value, self.sum_a, self.sum_b, self.sites = state, value, sum_a, sum_b, sites

    @classmethod
    def _from_c(cls, e) -> "FstEstimate":
        return cls(cls._STATES[e.state], e.value if e.state == 0 else None, e.sum_a, e.sum_b, int(e.sites))

    def components(self):
        return (self.value, self.sum_a, self.sum_b, self.sites)

    def __repr__(self):
        v = "None" if self.value is None else f"{self.value:.6f}"
        return (f"FstEstimate(state='{self.state}', value={v}, sum_a={self.sum_a!r}, sum_b={self.sum_b!r}, "
                f"sites={self.sites!r})")


class DiversitySite:  # lib.rs:259-279
    __slots__ = ("position", "pi", "watterson_theta")

    def __init__(self, position, pi, watterson_theta):
        self.position, self.pi, self.watterson_theta = position, pi, watterson_theta

    def __repr__(self):
        return f"DiversitySite(position={self.position}, pi={self.pi:.6f}, watterson_theta={self.watterson_theta:.6f})"


class HudsonDxyResult:  # lib.rs:281-303
    __slots__ = ("d_xy",)

    def __init__(self, d_xy):
        self.d_xy = d_xy

    def __repr__(self):
        return "HudsonDxyResult(d_xy=None)" if self.d_xy is None else f"HudsonDxyResult(d_xy={self.d_xy:.6f})"


class HudsonFstSite:  # lib.rs:305-362
    __slots__ = ("position", "fst", "d_xy", "pi_pop1", "pi_pop2", "n1_called", "n2_called",
                 "numerator_component", "denominator_component")

    def __init__(self, *a):
        for k, v in zip(self.__slots__, a):
            setattr(self, k, v)

    def __repr__(self):
        return (f"HudsonFstSite(position={self.position}, fst={self.fst}, d_xy={self.d_xy}, "
                f"pi_pop1={self.pi_pop1}, pi_pop2={self.pi_pop2}, n1_called={self.n1_called}, "
                f"n2_called={self.n2_called})")


class HudsonFstResult:  # lib.rs:364-436
    __slots__ = ("fst", "d_xy", "pi_pop1", "pi_pop2", "pi_xy_avg", "population1_label",
                 "population1_haplotype_group", "population2_label", "population2_haplotype_group")

    def __init__(self, fst, d_xy, pi1, pi2, pi_avg, id1, id2):
        self.fst, self.d_xy, self.pi_pop1, self.pi_pop2, self.pi_xy_avg = fst, d_xy, pi1, pi2, pi_avg
        self.population1_label, self.population1_haplotype_group = _population_label(id1)
        self.population2_label, self.population2_haplotype_group = _population_label(id2)

    def __repr__(self):
        return (f"HudsonFstResult(fst={self.fst}, d_xy={self.d_xy}, pi_pop1={self.pi_pop1}, "
                f"pi_pop2={self.pi_pop2}, pi_xy_avg={self.pi_xy_avg}, pop1={self.population1_label}, "
                f"pop2={self.population2_label})")


class WcFstSite:  # lib.rs:438-498
    __slots__ = ("position", "overall_fst", "pairwise_fst", "variance_components_a", "variance_components_b",
                 "population_sizes", "pairwise_variance_components")

    def __init__(self, *a):
        for k, v in zip(self.__slots__, a):
            setattr(self, k, v)

    def variance_components(self):
        return (self.variance_components_a, self.variance_components_b)

    def __repr__(self):
        return f"WcFstSite(position={self.position}, overall_fst={self.overall_fst!r})"


class WcFstResult:  # lib.rs:500-545
    __slots__ = ("overall_fst", "pairwise_fst", "pairwise_variance_components", "site_fst", "fst_type")

    def __init__(self, *a):
        for k, v in zip(self.__slots__, a):
            setattr(self, k, v)

    def __repr__(self):
        return f"WcFstResult(overall_fst={self.overall_fst!r})"


def _parse_population_id(obj):  # lib.rs:928-965 -> ("group", int) | ("named", str)
    if isinstance(obj, dict):
        if "haplotype_group" in obj:
            return ("group", int(obj["haplotype_group"]))
        if "named" in obj:
            return ("named", str(obj["named"]))
        raise ValueError("population id dictionaries must provide 'haplotype_group' or 'named'")
    if isinstance(obj, (int, np.integer)) and not isinstance(obj, bool):
        if not 0 <= int(obj) <= 255:
            raise ValueError("haplotype_group ids must be <= 255")
        return ("group", int(obj))
    if isinstance(obj, str):
        return ("named", obj)
    raise ValueError("could not interpret population id; pass an int, string, or mapping")


def _population_label(pid):  # lib.rs:1393-1400
    kind, v = pid
    return (f"haplotype_group_{v}", v) if kind == "group" else (v, None)


# --------------------------------------------------------------------------- Population
class _Shared:
    """Variants + optional dense arrays shared by cloned Populations (lib.rs:731-775)."""

    def __init__(self, variants: _Variants, dense: Optional[tuple]):
        self.variants = variants
        self.dense = dense  # (alleles[V,S,2], missing mask bool, max_allele) or None
        self._dense_matrix: Optional[_Matrix] = None

    def dense_matrix(self) -> Optional[_Matrix]:
        if self.dense is None:
            return None
        if self._dense_matrix is None:
            a, miss, max_allele = self.dense[:3]
            raw = self.dense[3] if len(self.dense) > 3 else None
            if raw is not None and max_allele <= 127:
                # int8 input with missing cells: hand the caller's buffer over as it is (in-band missingness)
                self._dense_matrix = _Matrix.from_int8(raw, self.variants.positions, max_allele)
            else:
                self._dense_matrix = _Matrix(a, miss, self.variants.positions, max_allele=max_allele)
        return self._dense_matrix

    def sparse_matrix(self, sample_count: Optional[int] = None) -> _Matrix:
        # with no missing entries the dense matrix already carries the sparse semantics
        dm = self.dense_matrix()
        if dm is not None and not dm.has_missing and (sample_count in (None, dm.S)):
            return dm
        return _sparse_matrix(self.variants, sample_count)


class Population:
    """ferromic.Population (lib.rs:547-728)."""

    def __init__(self, id, variants, haplotypes, sequence_length, sample_names=None):
        if sequence_length <= 0:
            raise ValueError("sequence_length must be a positive integer")
        self._id = _parse_population_id(id)
        self._haps = _parse_haplotypes(haplotypes)
        self._L = int(sequence_length)
        self._names = list(sample_names) if sample_names is not None else []
        self._shared = _Shared(_parse_variants(variants), None)

    @staticmethod
    def from_numpy(id, genotypes, positions, haplotypes, sequence_length, sample_names=None):
        if sequence_length <= 0:
            raise ValueError("sequence_length must be a positive integer")
        self = Population.__new__(Population)
        self._id = _parse_population_id(id)
        self._haps = _parse_haplotypes(haplotypes)
        self._L = int(sequence_length)
        self._names = list(sample_names) if sample_names is not None else []
        self._shared = _shared_from_numpy(genotypes, positions)
        return self

    def with_haplotypes(self, id, haplotypes):
        p = Population.__new__(Population)
        p._id = _parse_population_id(id)
        p._haps = _parse_haplotypes(haplotypes)
        p._L, p._names, p._shared = self._L, self._names, self._shared
        return p

    # --- path selection: OwnedPopulationContext::as_population_context (lib.rs:777-799)
    def _summary_group(self) -> Optional[_Group]:
        dm = self._shared.dense_matrix()
        if dm is None or dm.max_allele > 1:  # no summary for multi-allelic matrices (lib.rs:779)
            return None
        return dm.group(self._haps)

    def _dense_group(self) -> Optional[_Group]:
        """dense_genotypes of the context (ploidy-2 numpy input); for a multi-allelic matrix it
        comes without a summary and the reference takes its general dense paths."""
        dm = self._shared.dense_matrix()
        return None if dm is None else dm.group(self._haps)

    def segregating_sites(self) -> int:  # lib.rs:636 -> stats.rs:3831-3851
        g = self._summary_group()
        if g is not None:
            return g.summary()["segregating_sites"]
        g = self._dense_group()
        if g is not None:  # count_segregating_sites_dense (stats.rs:3891-4026)
            return g.segregating_sites()
        # sparse: count_segregating_sites_for_haplotypes (raw list; duplicates are harmless)
        vs = self._shared.variants
        if vs.n_variants == 0:
            return 0
        return _sparse_matrix(vs).group(self._haps).summary()["segregating_sites"]

    def nucleotide_diversity(self) -> float:  # lib.rs:644 -> stats.rs:4599-4614
        g = self._summary_group()
        if g is not None:
            return g.pi(self._L, _lib.FM_PI_SUMMARY)
        g = self._dense_group()
        if g is not None:  # calculate_pi_dense (stats.rs:4534-4597)
            return g.pi(self._L, _lib.FM_PI_DENSE)
        return _sparse_pi(self._shared.variants, self._haps, self._L)

    @property
    def id(self):
        return self._id[1]

    @property
    def haplotype_group(self):
        return self._id[1] if self._id[0] == "group" else None

    @property
    def label(self):
        return self._id[1] if self._id[0] == "named" else None

    @property
    def sequence_length(self):
        return self._L

    @property
    def variant_count(self):
        return self._shared.variants.n_variants

    @property
    def sample_names(self):
        return list(self._names)

    @property
    def haplotypes(self):
        return list(self._haps)

    def __repr__(self):
        label = f"haplotype_group {self._id[1]}" if self._id[0] == "group" else f"named '{self._id[1]}'"
        return (f"Population({label}, haplotypes={len(self._haps)}, variants={self.variant_count}, "
                f"sequence_length={self._L})")


def _shared_from_numpy(genotypes, positions) -> _Shared:
    """build_variants_from_numpy / convert_numeric_array (lib.rs:1082-1227)."""
    g = np.asarray(genotypes)
    if g.ndim != 3 or g.dtype not in (np.uint8, np.int8, np.uint16, np.int16):
        raise ValueError("genotypes must be a numpy.ndarray with dtype uint8/int8/uint16/int16 and shape "
                         "(variants, samples, ploidy)")
    V, S, P = g.shape
    pos = np.asarray(positions)
    if pos.ndim != 1 or pos.shape[0] != V:
        raise ValueError(f"positions length {pos.shape[0] if pos.ndim == 1 else pos.size} does not match "
                         f"variant dimension {V}")
    pos = pos.astype(np.int64)
    if g.dtype in (np.uint16, np.int16) and g.size and int(g.max()) > 255:
        raise ValueError("allele values must be <= 255")
    miss = (g < 0) if g.dtype in (np.int8, np.int16) else np.zeros(g.shape, dtype=bool)
    alle = np.where(miss, 0, g).astype(np.uint8)
    # sparse view: a sample is None when ANY of its alleles is missing (lib.rs:1195-1199)
    gt = alle.copy() if P else np.full((V, S, 1), MISSING, dtype=np.uint8)
    if P:
        gt[np.broadcast_to(miss.any(axis=2, keepdims=True), g.shape)] = MISSING
    variants = _Variants(pos, gt)
    dense = None
    if P == 2:  # lib.rs:1208
        raw = g if (g.dtype == np.int8 and miss.any()) else None  # bitmap only when needed (lib.rs:1209-1213)
        dense = (alle, miss, int(alle.max()) if alle.size else 0, raw)
    return _Shared(variants, dense)


def _coerce_population(obj) -> Population:  # PopulationInput (lib.rs:978-1080)
    if isinstance(obj, Population):
        return obj
    get = (lambda names: next((obj[n] for n in names if n in obj), None)) if isinstance(obj, dict) else (
        lambda names: _field(obj, names))
    pid = get(("id", "population_id", "name"))
    variants = get(("variants",))
    haps = get(("haplotypes",))
    L = get(("sequence_length", "length", "L"))
    if pid is None:
        raise ValueError("population-like object missing 'id'")
    if variants is None:
        raise ValueError("population requires 'variants'")
    if haps is None:
        raise ValueError("population requires 'haplotypes'")
    if L is None:
        raise ValueError("population-like object missing 'sequence_length'")
    names = get(("sample_names", "samples") if not isinstance(obj, dict) else ("sample_names",))
    return Population(pid, variants, haps, int(L), list(names) if names is not None else None)


# --------------------------------------------------------------------------- free functions
def _sparse_pi(vs: _Variants, haps, L: int) -> float:
    """calculate_pi (stats.rs:4317-4432): membership sized max(first variant's samples, max idx+1)."""
    if len(haps) <= 1:
        return math.nan
    if L < 0:
        return 0.0
    if L == 0:
        return math.inf
    vsc = vs.first_len if vs.n_variants else 0
    sc = max(vsc, max((h[0] + 1 for h in haps), default=0))
    m = _sparse_matrix(vs, max(sc, vs.n_samples))
    return m.group(haps).pi(L, _lib.FM_PI_SPARSE, raw_n=len(haps))


def segregating_sites(variants) -> int:  # lib.rs:1556 -> count_segregating_sites (stats.rs:3808)
    vs = _parse_variants(variants)
    if vs.n_variants == 0 or vs.n_samples == 0:
        return 0
    m = _sparse_matrix(vs)
    haps = [(s, side) for s in range(m.S) for side in range(m.P)]
    if m.P > 2:
        raise NotImplementedError("ploidy > 2 is not on the GPU path")
    return m.group(haps).summary()["segregating_sites"]


def nucleotide_diversity(variants, haplotypes, sequence_length) -> float:  # lib.rs:1564
    if sequence_length <= 0:
        raise ValueError("sequence_length must be a positive integer")
    return _sparse_pi(_parse_variants(variants), _parse_haplotypes(haplotypes), int(sequence_length))


def watterson_theta(segregating_sites, sample_count, sequence_length) -> float:  # lib.rs:1589
    if sample_count <= 1:
        raise ValueError("sample_count must be greater than 1 for Watterson's theta")
    if sequence_length <= 0:
        raise ValueError("sequence_length must be a positive integer")
    out = C.c_double()
    check(lib().fm_watterson_theta(int(segregating_sites), int(sample_count), int(sequence_length), C.byref(out)))
    return out.value


def _build_optional_region(region, vs: _Variants):  # lib.rs:1402-1441
    if region is not None:
        start, end = int(region[0]), int(region[1])
        if end < start:
            raise ValueError("region end must be greater than or equal to region start")
        return start, end
    if vs.n_variants == 0:
        raise ValueError("region must be provided when no variants are supplied")
    return int(vs.positions.min()), int(vs.positions.max())


def per_site_diversity_arrays(variants, haplotypes, region=None, mask=None, filtered_positions=()):
    """Array form of calculate_per_site_diversity (stats.rs:4628-4806): (positions, pi, theta)."""
    vs = _parse_variants(variants)
    haps = _parse_haplotypes(haplotypes)
    region = _build_optional_region(region, vs)
    empty = (np.zeros(0, np.int64), np.zeros(0), np.zeros(0))
    if vs.n_variants == 0:
        return empty
    # membership is sized by the first variant's sample count (stats.rs:4650-4654)
    m = _sparse_matrix(vs)
    g = m.group([h for h in haps if h[0] < vs.first_len])
    V = vs.n_variants
    pos = np.zeros(V, dtype=np.int64)
    pi = np.zeros(V, dtype=np.float64)
    th = np.zeros(V, dtype=np.float64)
    miv = None if mask is None else np.ascontiguousarray(np.asarray(mask, dtype=np.int64).reshape(-1))
    filt = np.ascontiguousarray(np.asarray(list(filtered_positions), dtype=np.int64))
    n = C.c_size_t()
    if miv is not None and miv.size == 0:
        miv = np.zeros(2, dtype=np.int64)  # Some(&[]) -> non-NULL pointer, zero intervals
        n_mask = 0
    else:
        n_mask = 0 if miv is None else miv.size // 2
    check(lib().fm_per_site_diversity(g.handle, len(haps), region[0], region[1], _ptr(miv), n_mask,
                                      _ptr(filt) if filt.size else None, filt.size, _ptr(pos), _ptr(pi),
                                      _ptr(th), V, C.byref(n)))
    k = n.value
    return pos[:k], pi[:k], th[:k]


def per_site_diversity(variants, haplotypes, region=None):  # lib.rs:1639-1665
    haps = _parse_haplotypes(haplotypes)
    if len(haps) < 2:
        raise ValueError("at least two haplotypes are required for diversity calculations")
    pos, pi, th = per_site_diversity_arrays(variants, haps, region)
    return [DiversitySite(int(p), float(a), float(b)) for p, a, b in zip(pos, pi, th)]


def _pairwise(variants, sample_count, want_positions: bool):
    """fm_pairwise_differences over the first sample_count samples: (differences, comparable, pair_start,
    positions) as condensed arrays in pair order (0,1), (0,2), ..., (1,2), ...; the last two are None unless
    want_positions."""
    n = int(sample_count)
    if n < 0:
        raise ValueError("sample_count must not be negative")
    vs = _parse_variants(variants)
    n_pairs = n * (n - 1) // 2
    diff = np.zeros(n_pairs, dtype=np.uint32)
    comp = np.zeros(n_pairs, dtype=np.uint32)
    if n_pairs == 0:
        empty = (np.zeros(1, dtype=np.uint64), np.zeros(0, dtype=np.int64)) if want_positions else (None, None)
        return (diff, comp) + empty
    # samples beyond a variant's genotype list are None
    m = _sparse_matrix(vs, max(n, vs.n_samples))
    L = lib()
    total = C.c_size_t()
    if not want_positions:
        check(L.fm_pairwise_differences(m.handle, n, _ptr(diff), _ptr(comp), None, None, 0, C.byref(total)))
        return diff, comp, None, None
    start = np.zeros(n_pairs + 1, dtype=np.uint64)
    pos = np.zeros(1, dtype=np.int64)
    st = L.fm_pairwise_differences(m.handle, n, _ptr(diff), _ptr(comp), _ptr(start), _ptr(pos), 0, C.byref(total))
    if st == _lib.FM_ERR_INVALID_ARG and total.value > 0:
        pos = np.zeros(total.value, dtype=np.int64)  # the first call reported the size: retry
        st = L.fm_pairwise_differences(m.handle, n, _ptr(diff), _ptr(comp), _ptr(start), _ptr(pos), pos.size,
                                       C.byref(total))
    check(st)
    return diff, comp, start, pos[:total.value]


def pairwise_difference_arrays(variants, sample_count):
    """Array form of calculate_pairwise_differences (stats.rs:4106-4231): (differences, comparable) as
    condensed u32 arrays of the n (n - 1) / 2 sample pairs in scipy.spatial.distance.pdist order.  comparable
    counts the variants where neither genotype is None, differences those of them where the genotypes differ
    as ordered vectors."""
    diff, comp, _, _ = _pairwise(variants, sample_count, False)
    return diff, comp


def pairwise_differences(variants, sample_count):  # stats.rs:4106-4231
    """[((i, j), difference_count, differing_positions), ...] for every sample pair i < j of
    0 .. sample_count-1; positions are the variants' own (0-based) positions in site order."""
    diff, _, start, pos = _pairwise(variants, sample_count, True)
    n = int(sample_count)
    pos = pos.tolist()
    start = start.tolist()
    out, k = [], 0
    for i in range(n):
        for j in range(i + 1, n):
            out.append(((i, j), int(diff[k]), pos[start[k]:start[k + 1]]))
            k += 1
    return out


def _opt(value: float, some: int, bit: int):
    return value if (some >> bit) & 1 else None


def _variants_compatible(a: _Variants, b: _Variants) -> bool:  # stats.rs:3399-3401
    return a.n_variants == b.n_variants and bool(np.array_equal(a.positions, b.positions))


def _pop_pi(p: Population) -> float:  # calculate_pi_for_population (stats.rs:4599-4614)
    return p.nucleotide_diversity()


def _hudson_member_haps(p: Population):
    """HapMembership::build(sample_names.len(), haplotypes) (stats.rs:3047-3048, 2473-2474)."""
    return [h for h in p._haps if h[0] < len(p._names)]


def _sparse_pair_groups(p1: Population, p2: Population):
    m = p1._shared.sparse_matrix(max(p1._shared.variants.n_samples, len(p1._names), len(p2._names), 1))
    g1, g2 = m.groups([_hudson_member_haps(p1), _hudson_member_haps(p2)])  # one pass over the u8 rows for both
    return g1, g2


def _hudson_dxy_value(p1: Population, p2: Population):  # calculate_d_xy_hudson (stats.rs:2403-2524)
    if p1._L <= 0:
        raise ValueError('VCF error: InvalidRegion("Sequence length must be positive for Dxy calculation")')
    if p1._L != p2._L:
        raise ValueError('VCF error: Parse("Sequence length mismatch in Dxy calculation")')
    if not _variants_compatible(p1._shared.variants, p2._shared.variants):
        raise ValueError('VCF error: Parse("Variant slices differ in positions/length for Dxy calculation")')
    if not p1._haps or not p2._haps:
        return None
    s1, s2 = p1._summary_group(), p2._summary_group()
    d, some = C.c_double(), C.c_int()
    if s1 is not None and s2 is not None:
        check(lib().fm_hudson_dxy(s1.handle, s2.handle, p1._L, p2._L, _lib.FM_HUDSON_SUMMARIES, len(p1._haps),
                                  len(p2._haps), C.byref(d), C.byref(some)))
    elif p1._shared is p2._shared and p1._dense_group() is not None:
        # same dense matrix, ploidy 2, no summaries: calculate_dxy_dense (stats.rs:2456-2470, 2526-2611)
        check(lib().fm_hudson_dxy(p1._dense_group().handle, p2._dense_group().handle, p1._L, p2._L,
                                  _lib.FM_HUDSON_DENSE, len(p1._haps), len(p2._haps), C.byref(d), C.byref(some)))
    else:
        if p1._shared.variants.n_variants == 0:
            return 0.0 / p1._L if p1._L > 0 else None
        g1, g2 = _sparse_pair_groups(p1, p2)
        check(lib().fm_hudson_dxy(g1.handle, g2.handle, p1._L, p2._L, _lib.FM_HUDSON_SPARSE, len(p1._haps),
                                  len(p2._haps), C.byref(d), C.byref(some)))
    return d.value if some.value else None


def _hudson_sparse(p1: "Population", p2: "Population", region, L: int):
    """Sparse per-site Hudson path (stats.rs:3021-3058, 3490-3503): (regional fst, sites)."""
    v1 = p1._shared.variants
    sites: List[HudsonFstSite] = []
    if v1.n_variants == 0:
        return None, sites
    g1, g2 = _sparse_pair_groups(p1, p2)
    V = v1.n_variants
    arr = {k: np.zeros(V, dtype=np.float64) for k in ("fst", "d_xy", "pi1", "pi2", "num", "den")}
    pos = np.zeros(V, dtype=np.int64)
    n1 = np.zeros(V, dtype=np.uint32)
    n2 = np.zeros(V, dtype=np.uint32)
    hs = _lib.HudsonSites(_ptr(pos), _ptr(arr["fst"]), _ptr(arr["d_xy"]), _ptr(arr["pi1"]), _ptr(arr["pi2"]),
                          _ptr(arr["num"]), _ptr(arr["den"]), _ptr(n1), _ptr(n2), V)
    n = C.c_size_t()
    out = _lib.HudsonOutcome()
    rs, re = region if region is not None else (0, 0)
    check(lib().fm_hudson_pair(g1.handle, g2.handle, L, L, _lib.FM_HUDSON_SPARSE,
                               1 if region is not None else 0, rs, re, len(p1._haps), len(p2._haps),
                               C.byref(out), C.byref(hs), C.byref(n)))

    def o(x):
        return None if math.isnan(x) else float(x)
    for i in range(n.value):
        sites.append(HudsonFstSite(int(pos[i]), o(arr["fst"][i]), o(arr["d_xy"][i]), o(arr["pi1"][i]),
                                   o(arr["pi2"][i]), int(n1[i]), int(n2[i]), o(arr["num"][i]), o(arr["den"][i])))
    return _opt(out.fst, out.some, 0), sites


def _hudson_core(p1: Population, p2: Population, region):
    """calculate_hudson_fst_for_pair_core (stats.rs:3435-3599): returns (HudsonFstResult, sites)."""
    if p1._L <= 0:
        raise ValueError('VCF error: InvalidRegion("Sequence length must be positive for Hudson FST calculation.")')
    if p1._L != p2._L:
        raise ValueError('VCF error: Parse("Sequence length mismatch between population contexts for '
                         'Hudson FST calculation.")')
    v1 = p1._shared.variants
    if not _variants_compatible(v1, p2._shared.variants):
        raise ValueError('VCF error: Parse("Variant slices differ in positions/length.")')
    s1, s2 = p1._summary_group(), p2._summary_group()
    out = _lib.HudsonOutcome()
    sites: List[HudsonFstSite] = []
    if region is None and s1 is not None and s2 is not None:
        n = C.c_size_t()
        check(lib().fm_hudson_pair(s1.handle, s2.handle, p1._L, p2._L, _lib.FM_HUDSON_SUMMARIES, 0, 0, 0,
                                   len(p1._haps), len(p2._haps), C.byref(out), None, C.byref(n)))
        return HudsonFstResult(_opt(out.fst, out.some, 0), _opt(out.d_xy, out.some, 1), _opt(out.pi_pop1, out.some, 2),
                               _opt(out.pi_pop2, out.some, 3), _opt(out.pi_xy_avg, out.some, 4), p1._id, p2._id), sites
    if region is None and p1._shared is p2._shared and p1._dense_group() is not None:
        # shared dense matrix without summaries (multi-allelic): dense_hudson_sites (stats.rs:3481-3489)
        n = C.c_size_t()
        check(lib().fm_hudson_pair(p1._dense_group().handle, p2._dense_group().handle, p1._L, p2._L,
                                   _lib.FM_HUDSON_DENSE, 0, 0, 0, len(p1._haps), len(p2._haps), C.byref(out), None,
                                   C.byref(n)))
        return HudsonFstResult(_opt(out.fst, out.some, 0), _opt(out.d_xy, out.some, 1), _opt(out.pi_pop1, out.some, 2),
                               _opt(out.pi_pop2, out.some, 3), _opt(out.pi_xy_avg, out.some, 4), p1._id, p2._id), sites
    # per-site sparse path (region) or whole-slice sparse path
    fst, sites = _hudson_sparse(p1, p2, region, p1._L)
    # auxiliary pi / Dxy follow each context's own preferred backend (stats.rs:3562-3565)
    pi1_raw, pi2_raw = _pop_pi(p1), _pop_pi(p2)
    dxy = _hudson_dxy_value(p1, p2)
    pi1 = pi1_raw if math.isfinite(pi1_raw) else None
    pi2 = pi2_raw if math.isfinite(pi2_raw) else None
    avg = 0.5 * (pi1 + pi2) if (pi1 is not None and pi2 is not None) else None
    return HudsonFstResult(fst, dxy, pi1, pi2, avg, p1._id, p2._id), sites


def _build_region(region):  # lib.rs:1402-1410
    start, end = int(region[0]), int(region[1])
    if end < start:
        raise ValueError("region end must be greater than or equal to region start")
    return start, end


def hudson_dxy(population1, population2) -> HudsonDxyResult:  # lib.rs:1668
    return HudsonDxyResult(_hudson_dxy_value(_coerce_population(population1), _coerce_population(population2)))


def hudson_fst(population1, population2) -> HudsonFstResult:  # lib.rs:1685
    return _hudson_core(_coerce_population(population1), _coerce_population(population2), None)[0]


def hudson_fst_sites(population1, population2, region):  # lib.rs:1702 -> stats.rs:3021-3058
    p1, p2 = _coerce_population(population1), _coerce_population(population2)
    region = _build_region(region)
    if not _variants_compatible(p1._shared.variants, p2._shared.variants):
        return []
    # per-site values do not depend on L (stats.rs:3036-3045 only warns about a mismatch)
    return _hudson_sparse(p1, p2, region, 1)[1]


def hudson_fst_with_sites(population1, population2, region):  # lib.rs:1722
    return _hudson_core(_coerce_population(population1), _coerce_population(population2), _build_region(region))


def _normalize_sample_name(name: str) -> str:  # process.rs:1192-1196
    if name.endswith("_L") or name.endswith("_R"):
        return name[:-2]
    return name


def _map_sample_names_to_indices(sample_names: Sequence[str]) -> Dict[str, int]:  # process.rs:1198-1241
    exact: Dict[str, int] = {}
    alias: Dict[str, Optional[int]] = {}
    for i, name in enumerate(sample_names):
        exact[name] = i
        suffix = name.rsplit("_", 1)[-1]
        if suffix != name:
            if suffix not in alias:
                alias[suffix] = i
            elif alias[suffix] != i:
                alias[suffix] = None
    for a, idx in alias.items():
        if idx is not None and a not in exact:
            exact[a] = idx
    return exact


def _membership_from_labels(n_samples: int, hap_to_label: Dict[Tuple[int, int], str]):
    """SubpopulationMembership::from_map (stats.rs:1103-1150)."""
    labels = sorted(set(hap_to_label.values()))
    index = {l: i for i, l in enumerate(labels)}
    left = np.full(n_samples, _U16_INVALID, dtype=np.uint16)
    right = np.full(n_samples, _U16_INVALID, dtype=np.uint16)
    for (s, side), lab in hap_to_label.items():
        if s >= n_samples:
            continue
        (left if side == 0 else right)[s] = index[lab]
    return labels, left, right


def wc_fst_from_membership(variants, labels: Sequence[str], left: np.ndarray, right: np.ndarray, region,
                           fst_type: str = "haplotype_groups", per_site: bool = True,
                           per_site_pairs: bool = True) -> WcFstResult:
    """Body of calculate_fst_wc_haplotype_groups / _csv_populations after the label mapping."""
    vs = _parse_variants(variants)
    rs, re = region
    G = len(labels)
    npairs = G * (G - 1) // 2
    pair_keys = [f"{labels[i]}_vs_{labels[j]}" for i in range(G) for j in range(i + 1, G)]
    S = len(left)
    m = _sparse_matrix(vs, max(S, vs.n_samples, 1))
    lft = np.full(m.S, _U16_INVALID, dtype=np.uint16)
    rgt = np.full(m.S, _U16_INVALID, dtype=np.uint16)
    lft[:S], rgt[:S] = left, right
    ph = C.c_void_p()
    check(lib().fm_partition_create(m.handle, _ptr(lft), _ptr(rgt), m.S, G, C.byref(ph)))
    try:
        V = max(vs.n_variants, 1)
        overall = _lib.FstEstimateC()
        pairs = (_lib.FstEstimateC * max(npairs, 1))()
        present = np.zeros(max(npairs, 1), dtype=np.uint8)
        pos = np.zeros(V, dtype=np.int64)
        state = np.zeros(V, dtype=np.int32)
        sa = np.zeros(V, dtype=np.float64)
        sb = np.zeros(V, dtype=np.float64)
        sizes = np.zeros((V, max(G, 1)), dtype=np.uint32)
        want_pairs = per_site and per_site_pairs and npairs > 0
        pa = np.zeros((V, max(npairs, 1)), dtype=np.float64) if want_pairs else None
        pb = np.zeros((V, max(npairs, 1)), dtype=np.float64) if want_pairs else None
        n = C.c_size_t()
        check(lib().fm_wc_fst(ph, rs, re, C.byref(overall), pairs, _ptr(present),
                              _ptr(pos) if per_site else None, _ptr(state) if per_site else None,
                              _ptr(sa) if per_site else None, _ptr(sb) if per_site else None,
                              _ptr(sizes) if per_site else None, _ptr(pa), _ptr(pb), V, C.byref(n)))
    finally:
        lib().fm_partition_release(ph)
    pairwise = {}
    pair_comp = {}
    for i, key in enumerate(pair_keys):
        if present[i]:
            pairwise[key] = FstEstimate._from_c(pairs[i])
            pair_comp[key] = (pairs[i].sum_a, pairs[i].sum_b)
    site_list = []
    if per_site:
        for i in range(n.value):
            st = int(state[i])
            est = FstEstimate(FstEstimate._STATES[st],
                              (sa[i] / (sa[i] + sb[i])) if st == 0 else None, float(sa[i]), float(sb[i]), 1)
            if st == 3:
                est = FstEstimate(FstEstimate._STATES[3], None, 0.0, 0.0, 1)
            has_maps = st != 3
            pw, pc = {}, {}
            if has_maps and want_pairs:
                for p, key in enumerate(pair_keys):
                    a, b = float(pa[i, p]), float(pb[i, p])
                    if math.isnan(a):  # pair without data at this site (stats.rs:2012-2022)
                        pw[key] = FstEstimate(FstEstimate._STATES[3], None, 0.0, 0.0, 1)
                        pc[key] = (0.0, 0.0)
                    else:
                        s2 = _fst_state(a, b)
                        pw[key] = FstEstimate(FstEstimate._STATES[s2], a / (a + b) if s2 == 0 else None, a, b, 1)
                        pc[key] = (a, b)
            popsz = {labels[gi]: int(sizes[i, gi]) for gi in range(G) if sizes[i, gi] > 0} if has_maps else {}
            site_list.append(WcFstSite(int(pos[i]), est, pw, float(sa[i]), float(sb[i]), popsz, pc))
    return WcFstResult(FstEstimate._from_c(overall), pairwise, pair_comp, site_list, fst_type)


def _fst_state(a: float, b: float) -> int:  # stats.rs:1781-1812
    den = a + b
    if den > 1e-12:
        return 0
    if den < -1e-12:
        return 1
    if abs(a) > 1e-12:
        return 0
    return 2


def wc_fst(variants, sample_names, sample_to_group, region) -> WcFstResult:  # lib.rs:1746-1770
    sample_names = list(sample_names)
    if not sample_names:
        raise ValueError("sample_names must contain at least one sample")
    if not isinstance(sample_to_group, dict):
        raise ValueError("sample_to_group must be a dict mapping sample -> (left, right)")
    region = _build_region(region)
    # map_samples_to_haplotype_groups (stats.rs:1036-1052)
    idx = _map_sample_names_to_indices(sample_names)
    hap_to_label: Dict[Tuple[int, int], str] = {}
    for name, grp in sample_to_group.items():
        try:
            lg, rg = int(grp[0]), int(grp[1])
        except Exception:
            raise ValueError("group tuples must contain two entries")
        i = idx.get(_normalize_sample_name(str(name)))
        if i is not None:
            hap_to_label[(i, 0)] = str(lg)
            hap_to_label[(i, 1)] = str(rg)
    labels, left, right = _membership_from_labels(len(sample_names), hap_to_label)
    return wc_fst_from_membership(variants, labels, left, right, region, "haplotype_groups")


def wc_fst_components(estimate: FstEstimate):  # lib.rs:1773-1778
    return estimate.components()


def adjusted_sequence_length(start, end, allow=None, mask=None) -> int:  # lib.rs:2190-2215
    if end < start:
        raise ValueError("end must be greater than or equal to start")

    def ivs(x):
        if x is None:
            return None, 0
        rows = []
        for e in x:
            s, t = int(e[0]), int(e[1])
            if t < s:
                raise ValueError("interval end must be greater than or equal to start")
            rows.append((s, t))
        a = np.asarray(rows, dtype=np.int64).reshape(-1)
        if a.size == 0:
            a = np.zeros(2, dtype=np.int64)
            return a, 0
        return np.ascontiguousarray(a), a.size // 2

    a, na = ivs(allow)
    m, nm = ivs(mask)
    out = C.c_int64()
    check(lib().fm_adjusted_sequence_length(int(start), int(end), _ptr(a), na, _ptr(m), nm, C.byref(out)))
    return out.value


def inversion_allele_frequency(sample_map) -> Optional[float]:  # lib.rs:2218 / stats.rs:3778-3805
    ones = total = 0
    for _, (h1, h2) in sample_map.items():
        for a in (int(h1), int(h2)):
            if a in (0, 1):
                total += 1
                ones += a
    return ones / total if total else None
