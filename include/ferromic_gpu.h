/*
 * ferromic_gpu.h -- C ABI of the B200 (sm_100a) implementation of ferromic's per-site
 * population-genetics estimators (reference: SauersML/ferromic, src/stats.rs).
 *
 * This is the drop-in boundary: the Rust crate (src/stats.rs entry points, src/lib.rs PyO3
 * wrappers, src/process.rs CLI call sites) binds exactly these symbols through `extern "C"`
 * (see INTEGRATION.md for the build.rs / gpu_ffi.rs stubs).  Plain pointers and sizes only.
 *
 * Conventions
 *  - every function returns an fm_status; fm_last_error() gives the thread-local message.
 *    FM_ERR_INVALID_REGION / FM_ERR_PARSE map to VcfError::InvalidRegion / VcfError::Parse
 *    (process.rs:631-640); nothing ever aborts or throws across the boundary.
 *  - host buffers are owned by the caller and are not retained after the call returns.
 *  - Option<f64> results are returned as a value plus a flag word (bit set = Some); per-site
 *    Option<f64> arrays use NaN for None (no Some value on this path can be NaN).
 *  - positions are 0-based on input; per-site outputs report position+1 (stats.rs:747,3004,4746).
 *  - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *    FM_ERR_NO_DEVICE.
 *  - handles are thread-safe (immutable device buffers; lazily cached summaries are guarded).
 */
#ifndef FERROMIC_GPU_H
#define FERROMIC_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef int fm_status;
#define FM_OK 0
#define FM_ERR_INVALID_REGION 1 /* VcfError::InvalidRegion */
#define FM_ERR_PARSE 2          /* VcfError::Parse */
#define FM_ERR_INVALID_ARG 3
#define FM_ERR_CUDA 4
#define FM_ERR_UNSUPPORTED 5
#define FM_ERR_NO_DEVICE 6

typedef struct fm_matrix fm_matrix; /* device-resident DenseGenotypeMatrix (stats.rs:249-331) */
typedef struct fm_group fm_group;   /* one population's haplotypes repacked into bitplanes      */
typedef struct fm_partition fm_partition; /* G-group partition for Weir & Cockerham (stats.rs:1093-1150) */

/* ---- library / device ---- */
const char *fm_last_error(void);
const char *fm_version(void);
fm_status fm_device_count(int *count);
fm_status fm_set_device(int device); /* device used by handles created afterwards on this thread */
/* Restrict the library to a subset of the visible GPUs (process-wide).  Without a call the environment
 * variable FERROMIC_GPU_DEVICES (comma separated CUDA ordinals, e.g. "0,2,3") is read once; neither:
 * every visible device.  A thread that never called fm_set_device works on the first allowed device;
 * fm_set_device rejects ordinals outside the list.  n == 0 lifts the restriction.  fm_get_devices
 * returns the allowed ordinals (one shard / rank per entry, SURVEY §8e). */
fm_status fm_set_devices(const int *devices, size_t n);
fm_status fm_get_devices(int *devices_out, size_t capacity, size_t *n_out);
fm_status fm_synchronize(void);
/* Device buffers come from a caching allocator inside the library and are kept for reuse when a
 * handle is released; this returns the cached memory of the current device to the driver. */
fm_status fm_trim_pool(void);

/* ---- matrix: replaces DenseGenotypeMatrix::new / ::from_variants (stats.rs:261-296, 339-500) ----
 * data[v*S*ploidy + s*ploidy + side] = allele index; missing = packed bitmap, 1 bit per entry,
 * LSB-first in u64 words (stats.rs:1298-1302), or NULL.  positions may be NULL (then 0..V-1).
 * The u8 matrix is uploaded once and stays resident; groups are repacked from it on device. */
fm_status fm_matrix_create(const uint8_t *data, const uint64_t *missing_or_null, size_t n_variants,
                           size_t n_samples, size_t ploidy, uint8_t max_allele,
                           const int64_t *positions_or_null, fm_matrix **out);
/* Same layout with in-band missingness: cells >= 0x80 (negative int8) are missing, no bitmap --
 * the int8 numpy array of Population.from_numpy as it is (lib.rs:1168-1199); see FM_MISSING_IN_BAND. */
fm_status fm_matrix_create_inband(const uint8_t *data, size_t n_variants, size_t n_samples, size_t ploidy,
                                  uint8_t max_allele, const int64_t *positions_or_null, fm_matrix **out);
/* Same, but data/missing already live in device memory of the current device (not copied, not
 * freed; must outlive the handle; d_data 16-byte aligned).  positions is a host pointer. */
fm_status fm_matrix_create_device(const uint8_t *d_data, const uint64_t *d_missing_or_null,
                                  size_t n_variants, size_t n_samples, size_t ploidy,
                                  uint8_t max_allele, const int64_t *positions_or_null,
                                  fm_matrix **out);
fm_status fm_matrix_retain(fm_matrix *m);
fm_status fm_matrix_release(fm_matrix *m);
fm_status fm_matrix_info(const fm_matrix *m, size_t *n_variants, size_t *n_samples, size_t *ploidy,
                         uint8_t *max_allele, int *has_missing);

/* ---- streaming ingest (SURVEY §8 f1: direct-to-bitplane ingestion) ----
 * For callers that can hand the matrix over in row chunks (process.rs:2602-2660 builds it row by
 * row; lib.rs:1135-1227 converts numpy row by row).  Declare every group / partition first, then
 * push rows; each chunk is staged in one of two device buffers and repacked into the declared
 * groups' bitplanes while the next chunk is copied, so upload and repack overlap and the u8
 * matrix is never resident.  The resulting matrix handle has no u8 data: fm_group_create /
 * fm_partition_create on it fail with FM_ERR_UNSUPPORTED.
 *   rows          -> u8 of row `first_row` (n_rows * n_samples * ploidy bytes, reference layout)
 *   missing_whole -> base of the WHOLE matrix's packed bitmap (stats.rs:1298-1302) or NULL when the
 *                    matrix was begun with has_missing == 0; only the words of the rows are read.
 * Host buffers are free again when fm_ingest_rows returns.  fm_ingest_finish hands out the
 * handles (groups in declaration order) and destroys the ingest handle.
 *
 * has_missing: FM_MISSING_NONE, FM_MISSING_BITMAP (the reference's packed bitmap) or
 * FM_MISSING_IN_BAND: cells >= 0x80 are missing and no bitmap exists -- exactly the int8 numpy
 * array Population.from_numpy receives (negative = missing, lib.rs:1168-1199), so the host hands
 * the caller's buffer over as it is: no convert_numeric_array pass, no bitmap packing, 11 % fewer
 * bytes over PCIe. */
#define FM_MISSING_NONE 0
#define FM_MISSING_BITMAP 1
#define FM_MISSING_IN_BAND 2
typedef struct fm_ingest fm_ingest;
fm_status fm_ingest_begin(size_t n_variants, size_t n_samples, size_t ploidy, int has_missing,
                          uint8_t max_allele, const int64_t *positions_or_null, size_t chunk_rows_or_0,
                          fm_ingest **out);
fm_status fm_ingest_add_group(fm_ingest *h, const uint64_t *sample_idx, const uint8_t *side, size_t n,
                              size_t *group_index);
fm_status fm_ingest_add_partition(fm_ingest *h, const uint16_t *left, const uint16_t *right,
                                  size_t n_samples, size_t n_groups, size_t *partition_index);
fm_status fm_ingest_rows(fm_ingest *h, const uint8_t *rows, const uint64_t *missing_whole_or_null,
                         size_t first_row, size_t n_rows);
/* Per-site tracks WHILE the rows arrive (calculate_per_site_diversity, stats.rs:4628-4806, for groups declared
 * with fm_ingest_add_group): same arguments, output layout and NaN rules as fm_per_site_diversity_multi, with
 * group_index[] naming declared groups.  Must be called after the groups are declared and before the first
 * rows call; *n_out (the number of sites in the region) is known at once, the arrays are complete when
 * fm_ingest_finish returns.  Every chunk's tracks are computed right after its repack on the ingest's compute
 * stream; page-locked output arrays receive them over PCIe while the following chunks are still being uploaded
 * (the two directions of the link do not compete), pageable ones are copied out in fm_ingest_finish.  The
 * caller's arrays must stay valid until then.  Biallelic bitplane groups only. */
fm_status fm_ingest_request_tracks(fm_ingest *h, const size_t *group_index, const size_t *raw_haplotype_counts,
                                   size_t n_groups, int64_t region_start, int64_t region_end,
                                   const int64_t *mask_intervals_or_null, size_t n_mask,
                                   const int64_t *filtered_positions_or_null, size_t n_filtered,
                                   int64_t *pos_out_or_null, double *pi_out, double *theta_out, size_t capacity,
                                   size_t *n_out);
/* ---- packed rows: 2 bits per genotype instead of 9 over PCIe (SURVEY §8 f1, "skip the u8 matrix") ----
 * Row v of the cohort as row_words = ceil(n_samples * ploidy / 32) u32 words of ALLELE bits followed
 * (in a second array) by row_words words of CALLED bits: bit (c & 31) of word (c >> 5) describes cell
 * c = sample * ploidy + side of the reference layout (stats.rs:249-331); allele bit = the cell is called
 * and carries a non-zero allele index, called bit = the cell is not missing; bits past the last cell are
 * zero.  Biallelic matrices only (max_allele <= 1).  This is what a parser can emit directly while it
 * reads genotypes (process.rs:2602-2660 / from_variants, stats.rs:339-500, build the u8 matrix AND the
 * bitmap today), and what fm_pack_rows produces from an existing u8 / int8 matrix (lib.rs:1135-1227).
 *
 * fm_ingest_rows_packed is the packed twin of fm_ingest_rows: rows go straight into the resident
 * packed matrix (0.25 B per genotype of HBM) and the declared groups / partitions are compressed out
 * of them chunk by chunk while the next chunk is on the bus.  Because the packed rows stay resident,
 * fm_group_create / fm_groups_create / fm_partition_create keep working on the finished matrix
 * (Population.with_haplotypes, lib.rs:622).  called_bits must be NULL iff the ingest was begun with
 * FM_MISSING_NONE; FM_MISSING_IN_BAND is a u8 notion and is rejected here.  An ingest takes either u8
 * rows or packed rows, not both. */
fm_status fm_packed_row_words(size_t n_samples, size_t ploidy, size_t *row_words);
fm_status fm_ingest_rows_packed(fm_ingest *h, const uint32_t *allele_bits, const uint32_t *called_bits_or_null,
                                size_t first_row, size_t n_rows);
/* Packed rows with a SPARSE MISSING LIST: the allele bit words as above and, instead of a called plane,
 * the columns c = sample * ploidy + side of the missing cells of every row in ascending order, as a CSR
 * list -- row_missing_start[r] .. row_missing_start[r + 1] (n_rows + 1 entries, relative to the call,
 * [0] == 0) index missing_cols, whose elements are col_bytes = 2 (row stride <= 65536) or 4 bytes wide.
 * col_bytes = 1 is the GAP CODE of the same list: the position starts at -1 in every row; a byte b < 255
 * moves it b + 1 columns on and names the cell it lands on, the byte 255 moves it 255 columns on without
 * naming a cell (row_missing_start then counts bytes).  With 1 % missing cells the list costs 0.16 bits
 * per genotype as u16 columns and 0.09 as gap codes -- 1.1 bits per genotype over PCIe in all instead of 2
 * (and 9 for u8 + bitmap); the called words are rebuilt on the device.  A parser sees the missing calls as it reads them ("./."),
 * so this is the natural output of process.rs:2602-2660; fm_pack_rows_sparse derives it from an existing
 * u8 / int8 matrix (*needed = number of list entries; FM_ERR_INVALID_ARG when capacity is too small, with
 * *needed and row_missing_start filled in so the caller can retry). */
fm_status fm_pack_rows_sparse(const uint8_t *rows, const uint64_t *missing_whole_or_null, int missing_mode,
                              size_t first_row, size_t n_rows, size_t n_total_rows, size_t stride,
                              uint32_t *allele_bits, uint64_t *row_missing_start, void *missing_cols,
                              size_t capacity, int col_bytes, int n_threads, size_t *needed);
fm_status fm_ingest_rows_packed_sparse(fm_ingest *h, const uint32_t *allele_bits, const uint64_t *row_missing_start,
                                       const void *missing_cols, int col_bytes, size_t first_row, size_t n_rows);
fm_status fm_matrix_create_packed_sparse(const uint32_t *allele_bits, const uint64_t *row_missing_start,
                                         const void *missing_cols, int col_bytes, size_t n_variants,
                                         size_t n_samples, size_t ploidy, const int64_t *positions_or_null,
                                         fm_matrix **out);
/* fm_ingest_rows with the packer inside: same arguments (u8 rows + whole-matrix bitmap, or in-band
 * cells), but the library packs chunk i+1 on the host with n_threads threads (<= 0: all) while chunk i
 * crosses PCIe as bit words -- the drop-in for callers that hold the reference's u8 / int8 matrix
 * (lib.rs:1135-1227) and cannot emit bits themselves.  Pageable sources are read in place. */
fm_status fm_ingest_rows_pack(fm_ingest *h, const uint8_t *rows, const uint64_t *missing_whole_or_null,
                              size_t first_row, size_t n_rows, int n_threads);
/* One-shot form: upload a whole packed matrix (replaces DenseGenotypeMatrix::new, stats.rs:261-296,
 * for hosts that pack); groups are created afterwards with fm_group_create & co. */
fm_status fm_matrix_create_packed(const uint32_t *allele_bits, const uint32_t *called_bits_or_null,
                                  size_t n_variants, size_t n_samples, size_t ploidy,
                                  const int64_t *positions_or_null, fm_matrix **out);
/* Host packer (no GPU involved; usable before any device call): rows -> first of n_rows u8 rows of
 * `stride` = n_samples * ploidy cells (row first_row of a matrix of n_total_rows rows);
 * missing_mode FM_MISSING_NONE / FM_MISSING_BITMAP (missing_whole = the WHOLE matrix's LSB-first
 * bitmap, stats.rs:1298-1302) / FM_MISSING_IN_BAND (cells >= 0x80 are missing).  Writes
 * allele_bits[n_rows][row_words] and, unless missing_mode is FM_MISSING_NONE, called_bits likewise.
 * n_threads <= 0: one thread per hardware thread.  AVX2 when the CPU has it (runtime check). */
fm_status fm_pack_rows(const uint8_t *rows, const uint64_t *missing_whole_or_null, int missing_mode,
                       size_t first_row, size_t n_rows, size_t n_total_rows, size_t stride,
                       uint32_t *allele_bits, uint32_t *called_bits_or_null, int n_threads);
/* the portable (non-AVX2) code path of the packer, single-threaded; exported for the parity tests */
fm_status fm_pack_rows_generic(const uint8_t *rows, const uint64_t *missing_whole_or_null, int missing_mode,
                               size_t first_row, size_t n_rows, size_t n_total_rows, size_t stride,
                               uint32_t *allele_bits, uint32_t *called_bits_or_null);

fm_status fm_ingest_finish(fm_ingest *h, fm_matrix **matrix_out, fm_group **groups_out,
                           fm_partition **partitions_out);
fm_status fm_ingest_abort(fm_ingest *h);

/* ---- group: replaces DenseMembership::build (stats.rs:1251-1284) + the per-group gather ----
 * haplotypes are (sample index, side 0=Left/1=Right); duplicates are counted once, out-of-range
 * samples are dropped, Right is dropped when ploidy <= 1 -- exactly as the reference.  The
 * group's columns are repacked on device into an allele bitplane and (when the matrix has a
 * missing bitmap) a called bitplane. */
fm_status fm_group_create(fm_matrix *m, const uint64_t *sample_idx, const uint8_t *side, size_t n,
                          fm_group **out);
/* Several groups of one matrix at once (e.g. the two haplotype groups of a config entry,
 * process.rs:3191-3208): the haplotype lists are concatenated, group g takes group_sizes[g] of them.
 * The u8 rows are read ONCE for all groups (fm_group_create reads them once per group). */
fm_status fm_groups_create(fm_matrix *m, const uint64_t *sample_idx, const uint8_t *side,
                           const size_t *group_sizes, size_t n_groups, fm_group **out);
fm_status fm_group_release(fm_group *g);
fm_status fm_group_capacity(const fm_group *g, size_t *haplotype_capacity);

/* build_dense_population_summary (stats.rs:1367-1470): alt/called may be NULL.  The summary is
 * computed once per group (the reference caches it in a OnceLock, lib.rs:738,777-789).
 * uncallable_lt2 = #{sites with called < 2} (used by stats.rs:1512-1517). */
fm_status fm_group_summary(fm_group *g, uint32_t *alt_out_or_null, uint32_t *called_out_or_null,
                           uint64_t *segregating_sites, double *pi_sum, uint64_t *uncallable_lt2);

/* The same for MANY groups in ONE persistent launch -- normally one group per region-sized matrix, the
 * shape of the CLI's serial loop over config entries (process.rs:2169: every entry builds its own
 * DenseGenotypeMatrix and summary).  Groups whose summaries are not cached yet are streamed by a single
 * pass over a segment table (any matrices of one device), so 64 regions of 100k sites run at the HBM
 * rate of one 6.4M-site matrix instead of 64 latency-sized launches.  Outputs [n_groups], any may be
 * NULL; afterwards every group is in the state fm_group_summary leaves it in (bit-identical scalars). */
fm_status fm_groups_summary_batch(fm_group *const *groups, size_t n_groups, uint64_t *segregating_sites,
                                  double *pi_sum, uint64_t *uncallable_lt2);

/* count_segregating_sites_for_population (stats.rs:3831-3851) for a dense ploidy-2 context. */
fm_status fm_group_segregating_sites(fm_group *g, uint64_t *out);

/* calculate_pi_for_population (stats.rs:4599-4614).  path: FM_PI_SUMMARY follows
 * calculate_pi_from_summary (:1480-1542); FM_PI_DENSE follows calculate_pi_dense(_biallelic)
 * (:4434-4597); FM_PI_SPARSE follows calculate_pi (:4317-4432, per-site form :2723-2733) and is
 * meant for matrices built with from_variants semantics. */
#define FM_PI_SUMMARY 0
#define FM_PI_DENSE 1
#define FM_PI_SPARSE 2
fm_status fm_group_pi(fm_group *g, int64_t sequence_length, int path, size_t raw_haplotype_count,
                      double *out);

/* harmonic (stats.rs:4234-4240) / calculate_watterson_theta (stats.rs:4243-4307); host scalars. */
fm_status fm_harmonic(size_t n, double *out);
fm_status fm_watterson_theta(size_t seg_sites, size_t n, int64_t sequence_length, double *out);

/* calculate_per_site_diversity (stats.rs:4628-4806) on the group's matrix (from_variants
 * missingness == the reference's sparse semantics).  region is 0-based inclusive; mask intervals
 * are 0-based half-open pairs [s,e) (mask_iv_or_null == NULL <=> None); filtered positions are
 * 0-based.  Outputs are caller-allocated with room for `capacity` sites; *n_out receives the
 * number of variants inside the region (in variant order).  raw_haplotype_count is
 * haplotypes_in_group.len() before de-duplication (the <2 guard at :4675 uses it).  pos_out may be
 * NULL when the caller already holds the positions (they are the input positions + 1).
 * Output arrays in page-locked host memory (cudaHostAlloc / cudaHostRegister, the whole row inside one
 * allocation) are written by the kernels themselves over PCIe; pageable arrays are filled by copies
 * from device buffers.  Same values either way. */
fm_status fm_per_site_diversity(fm_group *g, size_t raw_haplotype_count, int64_t region_start,
                                int64_t region_end, const int64_t *mask_iv_or_null, size_t n_mask,
                                const int64_t *filtered_pos, size_t n_filtered, int64_t *pos_out,
                                double *pi_out, double *theta_out, size_t capacity, size_t *n_out);

/* The same for several groups of one matrix over one region (the inversion-orientation groups
 * of a config entry, process.rs:1158): groups whose counts are not cached yet share ONE plane-pass
 * launch that streams their planes one after the other.  pi_out / theta_out are
 * [n_groups][capacity]; a group with fewer than two listed haplotypes (empty result in the
 * reference, stats.rs:4675-4681) gets NaN rows.  Values are bit-identical to per-group calls. */
fm_status fm_per_site_diversity_multi(fm_group *const *groups, const size_t *raw_haplotype_counts,
                                      size_t n_groups, int64_t region_start, int64_t region_end,
                                      const int64_t *mask_iv_or_null, size_t n_mask,
                                      const int64_t *filtered_pos, size_t n_filtered, int64_t *pos_out,
                                      double *pi_out, double *theta_out, size_t capacity, size_t *n_out);

/* ---- Hudson FST / Dxy (stats.rs:2403-2611, 2969-3278, 3435-3641) ---- */
typedef struct {
    double fst, d_xy, pi_pop1, pi_pop2, pi_xy_avg;
    uint32_t some; /* bit0 fst, bit1 d_xy, bit2 pi_pop1, bit3 pi_pop2, bit4 pi_xy_avg */
} fm_hudson_outcome;

/* SoA per-site outputs (any pointer may be NULL); Option<f64> => NaN for None. */
typedef struct {
    int64_t *position; /* 1-based */
    double *fst, *d_xy, *pi_pop1, *pi_pop2, *num_component, *den_component;
    uint32_t *n1_called, *n2_called;
    size_t capacity;
} fm_hudson_sites;

/* Which reference code path the call mirrors (stats.rs:3473-3503): */
#define FM_HUDSON_SUMMARIES 0 /* both contexts carry dense summaries (Python Population path) */
#define FM_HUDSON_DENSE 1     /* shared dense matrix, no summaries (CLI contexts)             */
#define FM_HUDSON_SPARSE 2    /* sparse per-site path (always taken when a region is given)   */

/* calculate_hudson_fst_for_pair_core (stats.rs:3435-3599).  g1 and g2 must share one matrix.
 * has_region != 0 selects calculate_hudson_fst_for_pair_with_sites (per-site values for variants
 * inside [region_start, region_end], FST from the sparse per-site form); the auxiliary pi/Dxy of
 * the outcome follow aux_path (FM_HUDSON_SUMMARIES / _DENSE / _SPARSE).  raw_n1/raw_n2 are the
 * un-deduplicated haplotype list lengths.  sites_or_null->capacity bounds the per-site outputs. */
fm_status fm_hudson_pair(fm_group *g1, fm_group *g2, int64_t sequence_length1,
                         int64_t sequence_length2, int path, int has_region, int64_t region_start,
                         int64_t region_end, size_t raw_n1, size_t raw_n2, fm_hudson_outcome *out,
                         fm_hudson_sites *sites_or_null, size_t *n_sites);

/* calculate_d_xy_hudson (stats.rs:2403-2524) */
fm_status fm_hudson_dxy(fm_group *g1, fm_group *g2, int64_t sequence_length1,
                        int64_t sequence_length2, int path, size_t raw_n1, size_t raw_n2,
                        double *d_xy, int *is_some);

/* ---- Weir & Cockerham (stats.rs:675-934, 1814-2374) ----
 * left/right[n_samples] give the group index (0..G-1) of each sample's Left/Right haplotype or
 * 0xFFFF (SubpopulationMembership, stats.rs:1093-1150); labels/pair keys stay on the host side.
 * The matrix must carry from_variants missingness (the reference's W&C path is sparse-only). */
typedef struct {
    int32_t state; /* 0 Calculable, 1 ComponentsYieldIndeterminateRatio,
                      2 NoInterPopulationVariance, 3 InsufficientDataForEstimation */
    double value;  /* FST when state == 0 (may be +-inf), NaN otherwise */
    double sum_a, sum_b;
    uint64_t sites;
} fm_fst_estimate;

fm_status fm_partition_create(fm_matrix *m, const uint16_t *left, const uint16_t *right,
                              size_t n_samples, size_t n_groups, fm_partition **out);
fm_status fm_partition_release(fm_partition *p);

/* Region W&C: overall estimate, per-pair estimates (pair order i<j, n_groups*(n_groups-1)/2
 * entries; pair_present[i]=0 when the key never appears in the reference's maps), and optional
 * per-site outputs for the variants inside the region (capacity entries each):
 *   site_pos (1-based), site_state, site_a, site_b, site_pop_sizes [capacity * n_groups],
 *   pair_a / pair_b [capacity * n_pairs] (per-site pairwise components). */
fm_status fm_wc_fst(fm_partition *p, int64_t region_start, int64_t region_end,
                    fm_fst_estimate *overall, fm_fst_estimate *pairs, uint8_t *pair_present,
                    int64_t *site_pos, int32_t *site_state, double *site_a, double *site_b,
                    uint32_t *site_pop_sizes, double *pair_a, double *pair_b, size_t capacity,
                    size_t *n_sites);

/* Shard-mergeable W&C window totals (sums and counts add across site shards; pair order i<j):
 * per window #variants, overall sum a / sum b / #sites with an estimate, and per pair
 * [n_windows * n_pairs] sum a / sum b / #informative sites.  Windows are 0-based inclusive
 * [start,end] position pairs.  Any output pointer may be NULL. */
fm_status fm_wc_window_sums(fm_partition *p, const int64_t *windows, size_t n_windows,
                            uint64_t *n_variants, double *overall_a, double *overall_b,
                            uint64_t *overall_sites, double *pair_a, double *pair_b,
                            uint64_t *pair_sites);
/* Region estimate from (merged) totals: the threshold ladder of calculate_overall_fst_wc
 * (stats.rs:2231-2270, 2290-2356).  informative_sites == 0 -> InsufficientDataForEstimation with
 * sites = sites_attempted. */
fm_status fm_fst_estimate_from_sums(double sum_a, double sum_b, uint64_t informative_sites,
                                    uint64_t sites_attempted, fm_fst_estimate *out);

/* Test hook: the two FP64 building blocks of the W&C kernels evaluated on the device over host arrays --
 * y[i] = the branch-free correctly rounded reciprocal of b[i] (b normal, away from the exponent limits),
 * q[i] = a[i] / b[i] computed from RN(1 / b[i]) with two residual corrections.  Both must equal IEEE
 * division bit for bit (tests/test_gpu_wc_arith.py); that is what lets K4 replace the per-pair divisions
 * of stats.rs:2034-2127 by table reciprocals without changing a single rounding. */
fm_status fm_wc_arith_probe(const double *a, const double *b, double *y, double *q, double *q_int_or_null,
                            size_t n); /* q_int: the one-correction form used for integer-like divisors */

/* ---- calculate_adjusted_sequence_length (stats.rs:3644-3736); host integer arithmetic ----
 * region is 1-based inclusive; allow/mask are 0-based half-open pairs; NULL <=> None. */
fm_status fm_adjusted_sequence_length(int64_t region_start, int64_t region_end,
                                      const int64_t *allow_or_null, size_t n_allow,
                                      const int64_t *mask_or_null, size_t n_mask, int64_t *out);

/* ---- windowed region summaries (K5: segmented reductions over site ranges) ----
 * windows are 0-based inclusive [start,end] pairs over positions (must be sorted ascending in the
 * matrix).  Per window: #variants, segregating sites, sum of per-site pi, #sites with called<2. */
fm_status fm_group_window_sums(fm_group *g, const int64_t *windows, size_t n_windows,
                               uint64_t *n_variants, uint64_t *seg_sites, double *pi_sum,
                               uint64_t *uncallable_lt2);
/* Per window Hudson component sums (from the two groups' cached summaries):
 * sum num, sum den, sum dxy (all callable), #uncallable, sum pi1, sum pi2. */
fm_status fm_hudson_window_sums(fm_group *g1, fm_group *g2, const int64_t *windows, size_t n_windows,
                                double *num_sum, double *den_sum, double *dxy_sum,
                                uint64_t *dxy_uncallable, double *pi1_sum, double *pi2_sum);

/* ---- finishing merged totals (host scalars; what every rank does after the gather) ----
 * calculate_pi_from_summary_with_precomputed (stats.rs:1480-1542): pi = pi_sum / (L - uncallable)
 * with the reference's guard order (haplotype_capacity <= 1 -> NaN; L < 0 -> 0; L == 0 -> +inf;
 * effective length 0 -> NaN). */
fm_status fm_pi_from_sums(double pi_sum, uint64_t uncallable_lt2, int64_t sequence_length,
                          size_t haplotype_capacity, double *out);
typedef struct {
    double num, den, dxy, pi1, pi2;       /* sums over the sites of the window / shard          */
    uint64_t dxy_uncallable, unc1, unc2;  /* #sites with n1==0||n2==0; #sites with n1<2; n2<2   */
} fm_hudson_sums;
/* Outcome of calculate_hudson_fst_for_pair_core on the summaries path (stats.rs:3476-3488,
 * 3505-3566) from merged totals. */
fm_status fm_hudson_outcome_from_sums(const fm_hudson_sums *sums, int64_t sequence_length,
                                      size_t haplotype_capacity1, size_t haplotype_capacity2,
                                      fm_hudson_outcome *out);

/* ---- region-total exchange over NVLink peer memory (the path's only exchange step) ----
 * One process (or host thread) per GPU creates a communicator on its device; the 64-byte handles
 * are swapped through whatever the host already has (torch.distributed, MPI, a pipe) and every
 * rank maps every peer's mailbox (cudaIpc).  fm_comm_allgather then runs ONE small kernel that
 * stores this rank's words into every peer's mailbox with P2P stores, publishes a step flag,
 * waits for all peers' flags and returns the gathered words plus their rank-ordered sum (the
 * first n_double words are summed as FP64, the rest as u64) -- bit-identical on every rank.
 * Ranks must issue the same sequence of exchanges.  Like a collective, an exchange waits for the slowest
 * rank; a peer that has not arrived after the timeout (default 120 s, fm_comm_set_timeout_ms; 0 = wait
 * for ever) makes the call fail with FM_ERR_CUDA on the waiting rank instead of hanging the GPU -- the
 * error is reported once, the communicator stays usable.  fm_comm_destroy runs a closing handshake with
 * all peers before it frees the mailbox, so it must be called by every rank (it is collective). */
typedef struct fm_comm fm_comm;
#define FM_COMM_HANDLE_BYTES 64
#define FM_COMM_MAX_WORDS 2048
fm_status fm_comm_create(int rank, int world, fm_comm **out);
fm_status fm_comm_export(fm_comm *c, uint8_t *handle_out /* [FM_COMM_HANDLE_BYTES] */);
fm_status fm_comm_connect(fm_comm *c, const uint8_t *handles /* [world][FM_COMM_HANDLE_BYTES] */);
/* Same-process variant (one host thread per GPU, or tests): all[r] is rank r's communicator. */
fm_status fm_comm_connect_local(fm_comm *c, fm_comm *const *all);
fm_status fm_comm_allgather(fm_comm *c, const void *local_words, size_t n_words, size_t n_double,
                            void *gathered_out_or_null /* [world][n_words] */,
                            void *merged_out_or_null /* [n_words] */);
fm_status fm_comm_set_timeout_ms(fm_comm *c, uint64_t milliseconds); /* default 120000; 0 = none */
fm_status fm_comm_destroy(fm_comm *c);

/* One Hudson FST / Dxy call over a cohort that is sharded by site range across the ranks of a
 * communicator (SURVEY §8e, BASELINE config 3): g1 / g2 are THIS rank's shard of the two populations
 * (built from the shard's rows), sequence_length is the whole region's.  Collective: every rank calls it
 * (also with an empty shard) and every rank receives the same outcome, bit for bit -- summaries path of
 * calculate_hudson_fst_for_pair_core (stats.rs:3476-3566) over the rank-ordered merged component sums.
 * Per rank: one sweep of the shard's planes (fused two-group pass, nothing cached), one fold kernel, one
 * fused fold + NVLink mailbox exchange kernel, one small copy.  comm == NULL computes the single shard.
 * merged_sums_or_null receives the merged totals (for window-wise post-processing). */
fm_status fm_hudson_pair_sharded(fm_group *g1, fm_group *g2, int64_t sequence_length, size_t raw_n1,
                                 size_t raw_n2, fm_comm *comm_or_null, fm_hudson_outcome *out,
                                 fm_hudson_sums *merged_sums_or_null);

/* ---- FALSTA per-site track bodies (process.rs:3740-4041; SURVEY 8f rank 3) ----
 * A track body is ONE comma-joined line of region_len tokens (region is 1-based inclusive, clamped
 * like ZeroBasedHalfOpen::from_1based_inclusive, process.rs:193-206): positions without a record
 * get the default token, a record's value prints as NaN -> "NA", 0.0 -> "0", otherwise Rust's
 * `{:.6}` (exactly, incl. round-half-even on the binary value); the last record at a position
 * wins (process.rs:3782-3795 overwrites line[idx] in record order).
 *   FM_FALSTA_DIVERSITY  default "0"   (append_diversity_falsta: pi / theta tracks, :3777-3793)
 *   FM_FALSTA_FST        default "NA", +-inf -> "Infinity" / "-Infinity"  (append_fst_falsta, :3842-3856)
 * pos1 are 1-based positions as in the per-site outputs.  fm_falsta_tracks renders n_tracks lines
 * that share the record positions (values[t*n + i] is record i of track t; e.g. pi and theta of one
 * group, or FST / numerator / denominator), separated by '\n'; line_len[t] (may be NULL) receives
 * each line's length.  out == NULL only queries the lengths; there is no trailing newline and no
 * terminating NUL.  The lines are rendered by the GPU (scatter -> token lengths -> scan -> write);
 * fm_falsta_format_value is the host instance of the same token routine (buf >= 56 bytes). */
#define FM_FALSTA_DIVERSITY 0
#define FM_FALSTA_FST 1
#define FM_FALSTA_TSV 2 /* fm_falsta_format_value only: format_optional_float (process.rs:3702-3713): NaN -> "NA",
                           everything else `{:.6}` (0.0 -> "0.000000", infinities -> "inf" / "-inf") */
fm_status fm_falsta_track(const int64_t *pos1, const double *values, size_t n, int64_t region_start,
                          int64_t region_end, int mode, char *out, size_t capacity, size_t *len_out);
fm_status fm_falsta_tracks(const int64_t *pos1, const double *values, size_t n, size_t n_tracks,
                           int64_t region_start, int64_t region_end, int mode, char *out, size_t capacity,
                           size_t *line_len, size_t *len_out);
fm_status fm_falsta_format_value(double value, int mode, char *buf, size_t capacity, size_t *len_out);

/* ---- VCF parse/filter stage (SURVEY 8f rank 4): process_variant over a chunk of raw text ----
 * Replaces the per-line work of process_vcf (process.rs:4262-4400) + process_variant (:4471-4768):
 * `text` holds VCF DATA lines (header already consumed by the host, :4181-4215), each terminated by
 * '\n' as BufRead::read_line frames them (a final unterminated line is a line).  Every line goes
 * through the reference's checks in the reference's order: field counts, chromosome match
 * (chr/Chr/CHR prefix stripped), POS, regions (ZeroBasedHalfOpen pairs, sorted as process_vcf passes
 * them), allow / mask flags, the REF/ALT length guard (MNP counter), the GQ key in FORMAT, genotypes
 * of the kept columns (None for ".", "./.", ".|." and anything u8 parsing rejects), GQ < min_gq,
 * missing data.  Line-local statistics are merged only for lines that returned Ok, a line that
 * returned Err is reported (fm_vcf_batch_errors) and skipped, and the surviving variants are sorted
 * by (position, compressed genotype bytes) exactly like process.rs:4377-4386.
 *   allow_mode / mask_mode: FM_VCF_NONE (Option is None), FM_VCF_INTERVALS (the map's (start, end)
 *   pairs of this chromosome), FM_VCF_CHR_ABSENT (a map was given but lacks this chromosome).
 *   max_ploidy: longest genotype the batch can hold (1..8); a longer one fails its line with
 *   FM_VCF_E_PLOIDY.  n_bytes < 2^31 per call (chunk on line boundaries; statistics are additive).
 * Genotypes stay on the device: gt[n_variants][n_kept][max_ploidy] u8 with the CompressedGenotypes
 * sentinel (0xFF in slot 0 = None, a later 0xFF ends the genotype, process.rs:430-478). */
typedef struct fm_vcf_batch fm_vcf_batch;
#define FM_VCF_NONE 0
#define FM_VCF_INTERVALS 1
#define FM_VCF_CHR_ABSENT 2
#define FM_VCF_E_FEW_FIELDS 10     /* "Invalid VCF line format: expected at least 9 fixed fields, found {aux}" */
#define FM_VCF_E_MISSING_COLUMN 11 /* "... expected genotype field at column {max+1}, found {aux} columns"     */
#define FM_VCF_E_INVALID_POS 12    /* "Invalid position"                                                       */
#define FM_VCF_E_POS_LT1 13        /* "Invalid 1-based pos: {aux}"                                             */
#define FM_VCF_E_NO_GQ_FORMAT 14   /* "GQ field not found in FORMAT"                                           */
#define FM_VCF_E_GQ_MISSING 15     /* "GQ value missing in sample genotype field at chr{chr}:{aux}"            */
#define FM_VCF_E_PLOIDY 16         /* unsupported: genotype longer than max_ploidy (aux = 1-based POS)         */
#define FM_VCF_E_TOO_MANY_ALTS 17  /* unsupported: more than 7 single-base ALT alleles (aux = 1-based POS)     */
typedef struct {
    uint64_t n_lines, n_variants, n_errors, n_samples, max_ploidy;
    /* FilteringStats (process.rs:406-416) and MissingDataInfo (:543-548) */
    uint64_t total_variants, filtered_variants, filtered_due_to_mask, filtered_due_to_allow,
        missing_data_variants, low_gq_variants, mnp_variants, total_data_points, missing_data_points,
        n_positions_with_missing, n_filtered_positions;
    float h2d_ms, index_ms, parse_ms; /* device time of the upload, line index and the two parse kernels */
} fm_vcf_info;
fm_status fm_vcf_parse(const char *text, size_t n_bytes, const char *chr, const int64_t *regions,
                       size_t n_regions, const uint32_t *kept_col_indices, size_t n_kept, uint16_t min_gq,
                       int allow_mode, const int64_t *allow, size_t n_allow, int mask_mode,
                       const int64_t *mask, size_t n_mask, size_t max_ploidy, fm_vcf_batch **out);
/* Same over text that already lives in device memory of the current device (16-byte aligned, at
 * least 32 readable bytes after n_bytes, zero up to the next 16-byte boundary; host_last_byte =
 * text[n_bytes-1]). */
fm_status fm_vcf_parse_device(const char *d_text, size_t n_bytes, char host_last_byte, const char *chr,
                              const int64_t *regions, size_t n_regions, const uint32_t *kept_col_indices,
                              size_t n_kept, uint16_t min_gq, int allow_mode, const int64_t *allow,
                              size_t n_allow, int mask_mode, const int64_t *mask, size_t n_mask,
                              size_t max_ploidy, fm_vcf_batch **out);
fm_status fm_vcf_batch_info(const fm_vcf_batch *b, fm_vcf_info *out);
/* per-variant arrays in output order (any pointer may be NULL): 0-based position, flags
 * (1 mask | 2 allow | 4 low GQ | 8 missing, process.rs:785-789), the variant's own genotype stride,
 * allele info (ref, number of ALT alleles, alts[n][7]) */
fm_status fm_vcf_batch_variants(const fm_vcf_batch *b, int64_t *pos0, uint8_t *flags, uint8_t *stride,
                                uint8_t *ref, uint8_t *n_alt, uint8_t *alts);
fm_status fm_vcf_batch_genotypes(const fm_vcf_batch *b, uint8_t *gt); /* [n_variants][n_samples][max_ploidy] */
/* sorted, de-duplicated members of MissingDataInfo::positions_with_missing / FilteringStats::filtered_positions */
fm_status fm_vcf_batch_positions(const fm_vcf_batch *b, int which /*0 missing, 1 filtered*/, int64_t *out,
                                 size_t capacity);
fm_status fm_vcf_batch_errors(const fm_vcf_batch *b, uint64_t *line_index, int32_t *code, int64_t *aux,
                              size_t capacity);
/* DenseGenotypeMatrix::from_variants (stats.rs:339-500) over the batch's variants (pass_only != 0:
 * only those with flags == 0, the CLI's "filtered" set) without leaving the device.  *out is NULL
 * when from_variants would return None (no variants / no genotype data). */
fm_status fm_vcf_batch_matrix(const fm_vcf_batch *b, int pass_only, fm_matrix **out);
/* The same matrix as resident PACKED rows (2 bits per genotype): genotypes go from the parser's output
 * straight to full-row bit words, the u8 matrix is never materialised (SURVEY §8 f1).  Biallelic batches
 * only -- FM_ERR_UNSUPPORTED when an allele index above 1 occurs (then use fm_vcf_batch_matrix). */
fm_status fm_vcf_batch_matrix_packed(const fm_vcf_batch *b, int pass_only, fm_matrix **out);
fm_status fm_vcf_batch_release(fm_vcf_batch *b);

/* ---- pairwise genotype differences (calculate_pairwise_differences, stats.rs:4106-4231) ----
 * For every pair of the first n_samples samples (n_samples <= the matrix's sample count), i < j in the order
 * (0,1), (0,2), ..., (1,2), ... (scipy.spatial.distance.pdist order, n_pairs = n_samples (n_samples - 1) / 2):
 *   comparable[p]  = #variants where neither genotype is None,
 *   differences[p] = #of those where the genotypes differ as whole ordered vectors (phase and length count),
 *   positions      = the 0-based positions of those variants, pair after pair, each pair's in site order;
 *                    pair p's run is positions[pair_start[p] .. pair_start[p + 1]).
 * A sample's genotype is the run of its leading called cells (side 0, side 1); it is None when cell 0 is missing --
 * the inverse of from_variants, so every matrix form has an answer (u8 with bitmap / in-band / no missingness, rank
 * LUT, resident packed rows).  Ploidy 1 or 2.  Outputs are host arrays: differences [n_pairs] (required),
 * comparable [n_pairs], pair_start [n_pairs + 1] and positions [positions_capacity] may be NULL; *n_positions_out
 * (may be NULL) receives the total number of differences.  Positions are requested by positions != NULL; when
 * positions_capacity is too small the counts, pair_start and *n_positions_out are written and the call returns
 * FM_ERR_INVALID_ARG so that the caller can retry.  The output grows with the number of differences: positions are
 * meant for small inputs.  FM_ERR_UNSUPPORTED for a matrix streamed as u8 rows (no resident rows) and ploidy > 2. */
fm_status fm_pairwise_differences(fm_matrix *m, size_t n_samples, uint32_t *differences, uint32_t *comparable_or_null,
                                  uint64_t *pair_start_or_null /* [n_pairs+1] */, int64_t *positions_or_null,
                                  size_t positions_capacity, size_t *n_positions_out);

/* ---- synthetic cohorts for benchmarks and full-size parity tests ----
 * Fills a device-resident u8 matrix (reference layout) and, when d_missing != NULL, its packed
 * missing bitmap with a counter-based generator: entry (site, column) is a pure integer function
 * of (seed, first_variant + site, column), so any slice can be re-evaluated on the CPU
 * (tests/synth.py::synth_rows) and shards generated with the right first_variant tile one cohort.
 * pop_of_sample (host, [n_samples] or NULL) selects the population whose frequency offset
 * (uniform in +-sigma around the U-shaped site frequency) applies to a sample. */
fm_status fm_synth_fill(uint8_t *d_data, uint64_t *d_missing_or_null, size_t n_variants, size_t n_samples,
                        size_t ploidy, uint64_t first_variant, uint64_t seed,
                        const uint16_t *pop_of_sample_or_null, double sigma, double missing_rate);

/* ---- instrumentation for bench.py (device timings of the last call, milliseconds) ---- */
typedef struct {
    float h2d_ms, repack_ms, stats_ms, reduce_ms, d2h_ms;
    uint64_t stats_launches;   /* launches of the plane-streaming kernels */
    uint64_t kernel_launches;  /* all kernel launches since the counters were reset */
    uint64_t stats_bytes;      /* algorithmic plane bytes streamed by the last stats kernel */
    float pack_ms;             /* host time inside the packer of fm_ingest_rows_pack (overlaps h2d) */
} fm_timings;
fm_status fm_timings_reset(void);
fm_status fm_timings_get(fm_timings *out);

/* Device-resident benchmark of the hot kernels (no host transfer inside the timed region).
 * One "step" streams the planes of every listed group once with the fused diversity epilogue
 * (mode 0: counts + summary partials; mode 1: + per-site pi/theta tracks with the mask applied)
 * and folds the per-batch partials on device.  Timing uses CUDA events on the launching stream:
 * step_ms_avg brackets all `iterations` steps, plane_ms_avg is the mean duration of one
 * plane-pass launch (events around every launch).  With a communicator every step ends with the
 * fused fold + peer exchange of the groups' region totals (S, sum pi, uncallable sites).
 * Mode 1 only: non-null last_pi / last_theta (host or device memory, [n_groups][V] doubles)
 * receive the per-site tracks of the last timed step, copied after the timed region. */
typedef struct {
    float step_ms_avg;
    float plane_ms_avg;
    uint64_t plane_launches;       /* plane-pass launches inside the timed region */
    uint64_t other_launches;       /* partial-reduction launches inside the timed region */
    uint64_t plane_bytes_per_step; /* bytes a step moves: per group and site the allele plane row (16-byte words +
                                    * tail words) and, with missing data, the 4-byte called count read, plus the
                                    * 16 B of pi / theta tracks written (mode 1) */
    float group_ms_avg[8];         /* mean duration of each plane-pass launch of a step (first 8): one launch for
                                    * the groups whose rows fit the row pass, then one per group with wider rows */
    uint64_t group_bytes[8];       /* the same bytes for each listed group */
    float comm_ms_avg;             /* mean duration of the fused fold + peer exchange kernel (incl. waiting) */
    /* region totals of the last timed step, per listed group (first 8): this rank's, and -- with a
     * communicator -- the exchanged rank-ordered sums (parity check of the run) */
    double last_pi_sum[8];
    uint64_t last_seg[8], last_unc[8];
    double merged_pi_sum[8];
    uint64_t merged_seg[8], merged_unc[8];
} fm_bench_result;
fm_status fm_bench_diversity(fm_group *const *groups, size_t n_groups, int mode,
                             const int64_t *mask_iv_or_null, size_t n_mask, int iterations,
                             fm_comm *comm_or_null, fm_bench_result *out, double *last_pi_or_null,
                             double *last_theta_or_null);

#ifdef __cplusplus
}
#endif
#endif /* FERROMIC_GPU_H */
