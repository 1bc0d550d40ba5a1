"""ctypes binding of libferromic_gpu.so (include/ferromic_gpu.h).

The shared library is the product: if it is missing the import fails loudly -- there is no
Python/CPU fallback on this path."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libferromic_gpu.so")

FM_OK, FM_ERR_INVALID_REGION, FM_ERR_PARSE, FM_ERR_INVALID_ARG = 0, 1, 2, 3
FM_ERR_CUDA, FM_ERR_UNSUPPORTED, FM_ERR_NO_DEVICE = 4, 5, 6
FM_PI_SUMMARY, FM_PI_DENSE, FM_PI_SPARSE = 0, 1, 2
FM_HUDSON_SUMMARIES, FM_HUDSON_DENSE, FM_HUDSON_SPARSE = 0, 1, 2


class HudsonOutcome(C.Structure):
    _fields_ = [("fst", C.c_double), ("d_xy", C.c_double), ("pi_pop1", C.c_double),
                ("pi_pop2", C.c_double), ("pi_xy_avg", C.c_double), ("some", C.c_uint32)]


class HudsonSites(C.Structure):
    _fields_ = [("position", C.c_void_p), ("fst", C.c_void_p), ("d_xy", C.c_void_p),
                ("pi_pop1", C.c_void_p), ("pi_pop2", C.c_void_p), ("num_component", C.c_void_p),
                ("den_component", C.c_void_p), ("n1_called", C.c_void_p), ("n2_called", C.c_void_p),
                ("capacity", C.c_size_t)]


class FstEstimateC(C.Structure):
    _fields_ = [("state", C.c_int32), ("value", C.c_double), ("sum_a", C.c_double),
                ("sum_b", C.c_double), ("sites", C.c_uint64)]


class HudsonSums(C.Structure):
    _fields_ = [("num", C.c_double), ("den", C.c_double), ("dxy", C.c_double), ("pi1", C.c_double),
                ("pi2", C.c_double), ("dxy_uncallable", C.c_uint64), ("unc1", C.c_uint64), ("unc2", C.c_uint64)]


class Timings(C.Structure):
    _fields_ = [("h2d_ms", C.c_float), ("repack_ms", C.c_float), ("stats_ms", C.c_float),
                ("reduce_ms", C.c_float), ("d2h_ms", C.c_float), ("stats_launches", C.c_uint64),
                ("kernel_launches", C.c_uint64), ("stats_bytes", C.c_uint64), ("pack_ms", C.c_float)]


class BenchResult(C.Structure):
    _fields_ = [("step_ms_avg", C.c_float), ("plane_ms_avg", C.c_float), ("plane_launches", C.c_uint64),
                ("other_launches", C.c_uint64), ("plane_bytes_per_step", C.c_uint64),
                ("group_ms_avg", C.c_float * 8), ("group_bytes", C.c_uint64 * 8), ("comm_ms_avg", C.c_float),
                ("last_pi_sum", C.c_double * 8), ("last_seg", C.c_uint64 * 8), ("last_unc", C.c_uint64 * 8),
                ("merged_pi_sum", C.c_double * 8), ("merged_seg", C.c_uint64 * 8), ("merged_unc", C.c_uint64 * 8)]


class VcfInfo(C.Structure):
    _fields_ = [(k, C.c_uint64) for k in (
        "n_lines", "n_variants", "n_errors", "n_samples", "max_ploidy", "total_variants", "filtered_variants",
        "filtered_due_to_mask", "filtered_due_to_allow", "missing_data_variants", "low_gq_variants", "mnp_variants",
        "total_data_points", "missing_data_points", "n_positions_with_missing", "n_filtered_positions")] + [
        ("h2d_ms", C.c_float), ("index_ms", C.c_float), ("parse_ms", C.c_float), ("inflate_ms", C.c_float)]


EXPORTS = [
    "fm_last_error", "fm_version", "fm_device_count", "fm_set_device", "fm_set_devices", "fm_get_devices", "fm_synchronize", "fm_trim_pool",
    "fm_matrix_create", "fm_matrix_create_inband", "fm_matrix_create_device", "fm_matrix_retain", "fm_matrix_release",
    "fm_matrix_info", "fm_ingest_begin", "fm_ingest_add_group", "fm_ingest_add_partition",
    "fm_ingest_rows", "fm_ingest_finish", "fm_ingest_abort", "fm_packed_row_words", "fm_ingest_rows_packed",
    "fm_matrix_create_packed", "fm_pack_rows", "fm_pack_rows_generic", "fm_ingest_rows_pack", "fm_pack_rows_sparse", "fm_ingest_rows_packed_sparse", "fm_ingest_request_tracks",
    "fm_matrix_create_packed_sparse", "fm_group_create", "fm_groups_create", "fm_group_release", "fm_group_capacity", "fm_group_summary", "fm_groups_summary_batch",
    "fm_group_segregating_sites", "fm_group_pi", "fm_harmonic", "fm_watterson_theta",
    "fm_per_site_diversity", "fm_per_site_diversity_multi", "fm_hudson_pair", "fm_hudson_dxy", "fm_partition_create",
    "fm_partition_release", "fm_wc_fst", "fm_wc_window_sums", "fm_fst_estimate_from_sums", "fm_wc_arith_probe", "fm_adjusted_sequence_length", "fm_group_window_sums",
    "fm_hudson_window_sums", "fm_pi_from_sums", "fm_hudson_outcome_from_sums", "fm_comm_create", "fm_comm_export", "fm_comm_connect", "fm_comm_connect_local", "fm_comm_allgather", "fm_comm_set_timeout_ms",
    "fm_comm_destroy", "fm_hudson_pair_sharded", "fm_falsta_track", "fm_falsta_tracks", "fm_falsta_format_value", "fm_vcf_parse", "fm_vcf_parse_device", "fm_vcf_batch_info",
    "fm_vcf_batch_variants", "fm_vcf_batch_genotypes", "fm_vcf_batch_positions", "fm_vcf_batch_errors", "fm_vcf_batch_matrix", "fm_vcf_batch_matrix_packed",
    "fm_vcf_batch_release", "fm_synth_fill", "fm_timings_reset", "fm_timings_get", "fm_bench_diversity",
    "fm_pairwise_differences", "fm_bgzf_inflate", "fm_vcf_parse_bgzf",
]

_lib = None


class FerromicGpuError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(message)
        self.code = code


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise ImportError(
            f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or make -C ferromic_b200/csrc). ferromic_b200 has no CPU fallback.")
    L = C.CDLL(SO_PATH)
    vp, sz, i64, u64, dbl = C.c_void_p, C.c_size_t, C.c_int64, C.c_uint64, C.c_double
    L.fm_last_error.restype = C.c_char_p
    L.fm_version.restype = C.c_char_p
    L.fm_device_count.argtypes = [C.POINTER(C.c_int)]
    L.fm_set_device.argtypes = [C.c_int]
    L.fm_set_devices.argtypes = [vp, sz]
    L.fm_get_devices.argtypes = [vp, sz, C.POINTER(sz)]
    L.fm_matrix_create.argtypes = [vp, vp, sz, sz, sz, C.c_uint8, vp, C.POINTER(vp)]
    L.fm_matrix_create_inband.argtypes = [vp, sz, sz, sz, C.c_uint8, vp, C.POINTER(vp)]
    L.fm_matrix_create_device.argtypes = [vp, vp, sz, sz, sz, C.c_uint8, vp, C.POINTER(vp)]
    L.fm_matrix_retain.argtypes = [vp]
    L.fm_matrix_release.argtypes = [vp]
    L.fm_matrix_info.argtypes = [vp, C.POINTER(sz), C.POINTER(sz), C.POINTER(sz), C.POINTER(C.c_uint8),
                                 C.POINTER(C.c_int)]
    L.fm_ingest_begin.argtypes = [sz, sz, sz, C.c_int, C.c_uint8, vp, sz, C.POINTER(vp)]
    L.fm_ingest_add_group.argtypes = [vp, vp, vp, sz, C.POINTER(sz)]
    L.fm_ingest_add_partition.argtypes = [vp, vp, vp, sz, sz, C.POINTER(sz)]
    L.fm_ingest_rows.argtypes = [vp, vp, vp, sz, sz]
    L.fm_packed_row_words.argtypes = [sz, sz, C.POINTER(sz)]
    L.fm_ingest_rows_packed.argtypes = [vp, vp, vp, sz, sz]
    L.fm_ingest_request_tracks.argtypes = [vp, vp, vp, sz, i64, i64, vp, sz, vp, sz, vp, vp, vp, sz, C.POINTER(sz)]
    L.fm_pack_rows_sparse.argtypes = [vp, vp, C.c_int, sz, sz, sz, sz, vp, vp, vp, sz, C.c_int, C.c_int, C.POINTER(sz)]
    L.fm_ingest_rows_packed_sparse.argtypes = [vp, vp, vp, vp, C.c_int, sz, sz]
    L.fm_matrix_create_packed_sparse.argtypes = [vp, vp, vp, C.c_int, sz, sz, sz, vp, C.POINTER(vp)]
    L.fm_ingest_rows_pack.argtypes = [vp, vp, vp, sz, sz, C.c_int]
    L.fm_matrix_create_packed.argtypes = [vp, vp, sz, sz, sz, vp, C.POINTER(vp)]
    L.fm_pack_rows.argtypes = [vp, vp, C.c_int, sz, sz, sz, sz, vp, vp, C.c_int]
    L.fm_pack_rows_generic.argtypes = [vp, vp, C.c_int, sz, sz, sz, sz, vp, vp]
    L.fm_ingest_finish.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]
    L.fm_ingest_abort.argtypes = [vp]
    L.fm_group_create.argtypes = [vp, vp, vp, sz, C.POINTER(vp)]
    L.fm_groups_create.argtypes = [vp, vp, vp, vp, sz, C.POINTER(vp)]
    L.fm_group_release.argtypes = [vp]
    L.fm_group_capacity.argtypes = [vp, C.POINTER(sz)]
    L.fm_group_summary.argtypes = [vp, vp, vp, C.POINTER(u64), C.POINTER(dbl), C.POINTER(u64)]
    L.fm_groups_summary_batch.argtypes = [C.POINTER(vp), sz, vp, vp, vp]
    L.fm_group_segregating_sites.argtypes = [vp, C.POINTER(u64)]
    L.fm_group_pi.argtypes = [vp, i64, C.c_int, sz, C.POINTER(dbl)]
    L.fm_harmonic.argtypes = [sz, C.POINTER(dbl)]
    L.fm_watterson_theta.argtypes = [sz, sz, i64, C.POINTER(dbl)]
    L.fm_per_site_diversity.argtypes = [vp, sz, i64, i64, vp, sz, vp, sz, vp, vp, vp, sz, C.POINTER(sz)]
    L.fm_per_site_diversity_multi.argtypes = [C.POINTER(vp), vp, sz, i64, i64, vp, sz, vp, sz, vp, vp, vp, sz, C.POINTER(sz)]
    L.fm_hudson_pair.argtypes = [vp, vp, i64, i64, C.c_int, C.c_int, i64, i64, sz, sz,
                                 C.POINTER(HudsonOutcome), C.POINTER(HudsonSites), C.POINTER(sz)]
    L.fm_hudson_dxy.argtypes = [vp, vp, i64, i64, C.c_int, sz, sz, C.POINTER(dbl), C.POINTER(C.c_int)]
    L.fm_partition_create.argtypes = [vp, vp, vp, sz, sz, C.POINTER(vp)]
    L.fm_partition_release.argtypes = [vp]
    L.fm_wc_fst.argtypes = [vp, i64, i64, C.POINTER(FstEstimateC), vp, vp, vp, vp, vp, vp, vp, vp, vp, sz,
                            C.POINTER(sz)]
    L.fm_wc_window_sums.argtypes = [vp, vp, sz, vp, vp, vp, vp, vp, vp, vp]
    L.fm_fst_estimate_from_sums.argtypes = [dbl, dbl, u64, u64, C.POINTER(FstEstimateC)]
    L.fm_wc_arith_probe.argtypes = [vp, vp, vp, vp, vp, sz]
    L.fm_adjusted_sequence_length.argtypes = [i64, i64, vp, sz, vp, sz, C.POINTER(i64)]
    L.fm_group_window_sums.argtypes = [vp, vp, sz, vp, vp, vp, vp]
    L.fm_hudson_window_sums.argtypes = [vp, vp, vp, sz, vp, vp, vp, vp, vp, vp]
    L.fm_pi_from_sums.argtypes = [dbl, u64, i64, sz, C.POINTER(dbl)]
    L.fm_hudson_outcome_from_sums.argtypes = [C.POINTER(HudsonSums), i64, sz, sz, C.POINTER(HudsonOutcome)]
    L.fm_falsta_track.argtypes = [vp, vp, sz, i64, i64, C.c_int, vp, sz, C.POINTER(sz)]
    L.fm_falsta_tracks.argtypes = [vp, vp, sz, sz, i64, i64, C.c_int, vp, sz, vp, C.POINTER(sz)]
    L.fm_falsta_format_value.argtypes = [dbl, C.c_int, vp, sz, C.POINTER(sz)]
    u16 = C.c_uint16
    L.fm_vcf_parse.argtypes = [C.c_char_p, sz, C.c_char_p, vp, sz, vp, sz, u16, C.c_int, vp, sz, C.c_int, vp, sz, sz,
                               C.POINTER(vp)]
    L.fm_vcf_parse_device.argtypes = [vp, sz, C.c_char, C.c_char_p, vp, sz, vp, sz, u16, C.c_int, vp, sz, C.c_int, vp,
                                      sz, sz, C.POINTER(vp)]
    L.fm_bgzf_inflate.argtypes = [vp, sz, vp, sz, C.POINTER(u64)]
    L.fm_vcf_parse_bgzf.argtypes = [vp, sz, u64, C.c_char_p, vp, sz, vp, sz, u16, C.c_int, vp, sz, C.c_int, vp, sz, sz,
                                    C.POINTER(vp)]
    L.fm_vcf_batch_info.argtypes = [vp, C.POINTER(VcfInfo)]
    L.fm_vcf_batch_variants.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    L.fm_vcf_batch_genotypes.argtypes = [vp, vp]
    L.fm_vcf_batch_positions.argtypes = [vp, C.c_int, vp, sz]
    L.fm_vcf_batch_errors.argtypes = [vp, vp, vp, vp, sz]
    L.fm_vcf_batch_matrix.argtypes = [vp, C.c_int, C.POINTER(vp)]
    L.fm_vcf_batch_matrix_packed.argtypes = [vp, C.c_int, C.POINTER(vp)]
    L.fm_vcf_batch_release.argtypes = [vp]
    L.fm_synth_fill.argtypes = [vp, vp, sz, sz, sz, u64, u64, vp, dbl, dbl]
    L.fm_timings_get.argtypes = [C.POINTER(Timings)]
    L.fm_bench_diversity.argtypes = [C.POINTER(vp), sz, C.c_int, vp, sz, C.c_int, vp, C.POINTER(BenchResult), vp,
                                     vp]
    L.fm_comm_create.argtypes = [C.c_int, C.c_int, C.POINTER(vp)]
    L.fm_comm_export.argtypes = [vp, vp]
    L.fm_comm_connect.argtypes = [vp, vp]
    L.fm_comm_connect_local.argtypes = [vp, C.POINTER(vp)]
    L.fm_comm_allgather.argtypes = [vp, vp, sz, sz, vp, vp]
    L.fm_comm_set_timeout_ms.argtypes = [vp, u64]
    L.fm_comm_destroy.argtypes = [vp]
    L.fm_hudson_pair_sharded.argtypes = [vp, vp, i64, sz, sz, vp, C.POINTER(HudsonOutcome), C.POINTER(HudsonSums)]
    L.fm_pairwise_differences.argtypes = [vp, sz, vp, vp, vp, vp, sz, C.POINTER(sz)]
    for name in EXPORTS:
        fn = getattr(L, name)
        if name not in ("fm_last_error", "fm_version"):
            fn.restype = C.c_int
    _lib = L
    return L


def check(status: int) -> None:
    """Map fm_status to the reference's Python error behaviour (lib.rs:1551-1553)."""
    if status == FM_OK:
        return
    msg = lib().fm_last_error().decode("utf-8", "replace")
    if status == FM_ERR_INVALID_REGION:
        raise ValueError(f'VCF error: InvalidRegion("{msg}")')
    if status == FM_ERR_PARSE:
        raise ValueError(f'VCF error: Parse("{msg}")')
    if status == FM_ERR_INVALID_ARG:
        raise ValueError(msg)
    if status == FM_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise FerromicGpuError(status, msg)
