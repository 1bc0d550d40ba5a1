// Materialised from INTEGRATION.md section 2 (+ the round-2 additions at the end).  Not compiled in the authoring
// image: there is no rustc / cargo.  include/ferromic_gpu.h is the authority for every signature.
#![allow(non_camel_case_types)]
use std::{ffi::CStr, os::raw::{c_char, c_int}, ptr, sync::Arc};
use crate::process::VcfError;

#[repr(C)] pub struct fm_matrix { _p: [u8; 0] }
#[repr(C)] pub struct fm_group { _p: [u8; 0] }
#[repr(C)] pub struct fm_partition { _p: [u8; 0] }
#[repr(C)] pub struct fm_ingest { _p: [u8; 0] }
#[repr(C)] pub struct fm_comm { _p: [u8; 0] }
#[repr(C)] pub struct fm_vcf_batch { _p: [u8; 0] }

#[repr(C)] #[derive(Default, Clone, Copy)]
pub struct fm_hudson_outcome { pub fst: f64, pub d_xy: f64, pub pi_pop1: f64, pub pi_pop2: f64,
                               pub pi_xy_avg: f64, pub some: u32 }
#[repr(C)]
pub struct fm_hudson_sites { pub position: *mut i64, pub fst: *mut f64, pub d_xy: *mut f64,
    pub pi_pop1: *mut f64, pub pi_pop2: *mut f64, pub num_component: *mut f64,
    pub den_component: *mut f64, pub n1_called: *mut u32, pub n2_called: *mut u32, pub capacity: usize }
#[repr(C)] #[derive(Clone, Copy)]
pub struct fm_fst_estimate { pub state: i32, pub value: f64, pub sum_a: f64, pub sum_b: f64, pub sites: u64 }
#[repr(C)] #[derive(Default, Clone, Copy)]
pub struct fm_hudson_sums { pub num: f64, pub den: f64, pub dxy: f64, pub pi1: f64, pub pi2: f64,
                            pub dxy_uncallable: u64, pub unc1: u64, pub unc2: u64 }

extern "C" {
    pub fn fm_last_error() -> *const c_char;
    pub fn fm_device_count(count: *mut c_int) -> c_int;
    pub fn fm_set_device(device: c_int) -> c_int;
    // DenseGenotypeMatrix::new / ::from_variants            (stats.rs:261-296, 339-500)
    pub fn fm_matrix_create(data: *const u8, missing: *const u64, n_variants: usize, n_samples: usize,
        ploidy: usize, max_allele: u8, positions: *const i64, out: *mut *mut fm_matrix) -> c_int;
    pub fn fm_matrix_create_inband(data: *const u8, n_variants: usize, n_samples: usize, ploidy: usize,
        max_allele: u8, positions: *const i64, out: *mut *mut fm_matrix) -> c_int;   // int8 cells < 0 = missing
    pub fn fm_matrix_retain(m: *mut fm_matrix) -> c_int;
    pub fn fm_matrix_release(m: *mut fm_matrix) -> c_int;
    // streaming variant for process.rs:2602-2660 / lib.rs:1135-1227 (row-by-row producers)
    pub fn fm_ingest_begin(n_variants: usize, n_samples: usize, ploidy: usize, has_missing: c_int,
        max_allele: u8, positions: *const i64, chunk_rows: usize, out: *mut *mut fm_ingest) -> c_int;
    pub fn fm_ingest_add_group(h: *mut fm_ingest, sample_idx: *const u64, side: *const u8, n: usize,
        group_index: *mut usize) -> c_int;
    pub fn fm_ingest_add_partition(h: *mut fm_ingest, left: *const u16, right: *const u16,
        n_samples: usize, n_groups: usize, partition_index: *mut usize) -> c_int;
    pub fn fm_ingest_rows(h: *mut fm_ingest, rows: *const u8, missing_whole: *const u64,
        first_row: usize, n_rows: usize) -> c_int;
    pub fn fm_ingest_finish(h: *mut fm_ingest, matrix_out: *mut *mut fm_matrix,
        groups_out: *mut *mut fm_group, partitions_out: *mut *mut fm_partition) -> c_int;
    pub fn fm_ingest_abort(h: *mut fm_ingest) -> c_int;
    // DenseMembership::build + build_dense_population_summary (stats.rs:1251-1284, 1367-1470)
    pub fn fm_group_create(m: *mut fm_matrix, sample_idx: *const u64, side: *const u8, n: usize,
        out: *mut *mut fm_group) -> c_int;
    pub fn fm_group_release(g: *mut fm_group) -> c_int;
    pub fn fm_group_summary(g: *mut fm_group, alt_out: *mut u32, called_out: *mut u32,
        segregating_sites: *mut u64, pi_sum: *mut f64, uncallable_lt2: *mut u64) -> c_int;
    pub fn fm_group_segregating_sites(g: *mut fm_group, out: *mut u64) -> c_int;   // stats.rs:3831
    pub fn fm_group_pi(g: *mut fm_group, sequence_length: i64, path: c_int, raw_haplotype_count: usize,
        out: *mut f64) -> c_int;                                                   // stats.rs:4599
    pub fn fm_watterson_theta(seg_sites: usize, n: usize, sequence_length: i64, out: *mut f64) -> c_int;
    pub fn fm_per_site_diversity(g: *mut fm_group, raw_haplotype_count: usize, region_start: i64,
        region_end: i64, mask_iv: *const i64, n_mask: usize, filtered_pos: *const i64, n_filtered: usize,
        pos_out: *mut i64, pi_out: *mut f64, theta_out: *mut f64, capacity: usize, n_out: *mut usize) -> c_int;
    pub fn fm_hudson_pair(g1: *mut fm_group, g2: *mut fm_group, l1: i64, l2: i64, path: c_int,
        has_region: c_int, region_start: i64, region_end: i64, raw_n1: usize, raw_n2: usize,
        out: *mut fm_hudson_outcome, sites: *mut fm_hudson_sites, n_sites: *mut usize) -> c_int;
    pub fn fm_hudson_dxy(g1: *mut fm_group, g2: *mut fm_group, l1: i64, l2: i64, path: c_int,
        raw_n1: usize, raw_n2: usize, d_xy: *mut f64, is_some: *mut c_int) -> c_int;
    pub fn fm_partition_create(m: *mut fm_matrix, left: *const u16, right: *const u16, n_samples: usize,
        n_groups: usize, out: *mut *mut fm_partition) -> c_int;
    pub fn fm_partition_release(p: *mut fm_partition) -> c_int;
    pub fn fm_wc_fst(p: *mut fm_partition, region_start: i64, region_end: i64,
        overall: *mut fm_fst_estimate, pairs: *mut fm_fst_estimate, pair_present: *mut u8,
        site_pos: *mut i64, site_state: *mut i32, site_a: *mut f64, site_b: *mut f64,
        site_pop_sizes: *mut u32, pair_a: *mut f64, pair_b: *mut f64, capacity: usize,
        n_sites: *mut usize) -> c_int;
    pub fn fm_adjusted_sequence_length(region_start: i64, region_end: i64, allow: *const i64,
        n_allow: usize, mask: *const i64, n_mask: usize, out: *mut i64) -> c_int;
    // calculate_pairwise_differences (stats.rs:4106-4231): condensed pair order (0,1), (0,2), ..., (1,2), ...;
    // positions != NULL requests the differing positions (FM_ERR_INVALID_ARG + *n_positions_out when the capacity
    // is too small)
    pub fn fm_pairwise_differences(m: *mut fm_matrix, n_samples: usize, differences: *mut u32,
        comparable: *mut u32, pair_start: *mut u64, positions: *mut i64, positions_capacity: usize,
        n_positions_out: *mut usize) -> c_int;
    // shard-mergeable window totals + finishers (multi-GPU, windows)
    pub fn fm_group_window_sums(g: *mut fm_group, windows: *const i64, n_windows: usize,
        n_variants: *mut u64, seg_sites: *mut u64, pi_sum: *mut f64, uncallable_lt2: *mut u64) -> c_int;
    pub fn fm_hudson_window_sums(g1: *mut fm_group, g2: *mut fm_group, windows: *const i64,
        n_windows: usize, num: *mut f64, den: *mut f64, dxy: *mut f64, dxy_uncallable: *mut u64,
        pi1: *mut f64, pi2: *mut f64) -> c_int;
    pub fn fm_wc_window_sums(p: *mut fm_partition, windows: *const i64, n_windows: usize,
        n_variants: *mut u64, overall_a: *mut f64, overall_b: *mut f64, overall_sites: *mut u64,
        pair_a: *mut f64, pair_b: *mut f64, pair_sites: *mut u64) -> c_int;
    pub fn fm_pi_from_sums(pi_sum: f64, uncallable: u64, l: i64, cap: usize, out: *mut f64) -> c_int;
    pub fn fm_hudson_outcome_from_sums(s: *const fm_hudson_sums, l: i64, cap1: usize, cap2: usize,
        out: *mut fm_hudson_outcome) -> c_int;
    pub fn fm_fst_estimate_from_sums(sum_a: f64, sum_b: f64, informative: u64, attempted: u64,
        out: *mut fm_fst_estimate) -> c_int;
    // region-total exchange over NVLink peer memory (one process per GPU; 64-byte handles are
    // swapped by the host: MPI, a pipe, or any existing control channel)
    pub fn fm_comm_create(rank: c_int, world: c_int, out: *mut *mut fm_comm) -> c_int;
    pub fn fm_comm_export(c: *mut fm_comm, handle_out: *mut u8) -> c_int;          // [64]
    pub fn fm_comm_connect(c: *mut fm_comm, handles: *const u8) -> c_int;          // [world][64]
    pub fn fm_comm_allgather(c: *mut fm_comm, local_words: *const u64, n_words: usize, n_double: usize,
        gathered_out: *mut u64, merged_out: *mut u64) -> c_int;
    pub fn fm_comm_destroy(c: *mut fm_comm) -> c_int;
}

/// fm_status -> the crate's error type (process.rs:631-640). Precondition failures are `Err`,
/// data insufficiency stays `None`/NaN in the outputs, nothing panics or aborts.
pub fn check(status: c_int) -> Result<(), VcfError> {
    if status == 0 { return Ok(()); }
    let msg = unsafe { CStr::from_ptr(fm_last_error()) }.to_string_lossy().into_owned();
    Err(match status {
        1 => VcfError::InvalidRegion(msg),
        2 => VcfError::Parse(msg),
        _ => VcfError::Parse(format!("GPU backend: {msg}")),   // or a new VcfError::Gpu(String)
    })
}

/// Device twin of `DenseGenotypeMatrix`; lives inside it as `gpu: OnceLock<Arc<GpuMatrix>>`.
pub struct GpuMatrix(pub *mut fm_matrix);
unsafe impl Send for GpuMatrix {}
unsafe impl Sync for GpuMatrix {}   // handles are thread-safe (immutable device buffers)
impl Drop for GpuMatrix { fn drop(&mut self) { unsafe { fm_matrix_release(self.0); } } }

pub struct GpuGroup(pub *mut fm_group, pub Arc<GpuMatrix>);
unsafe impl Send for GpuGroup {}
unsafe impl Sync for GpuGroup {}
impl Drop for GpuGroup { fn drop(&mut self) { unsafe { fm_group_release(self.0); } } }

impl GpuMatrix {
    pub fn upload(data: &[u8], missing: Option<&[u64]>, variants: usize, samples: usize, ploidy: usize,
                  max_allele: u8, positions: &[i64]) -> Result<Arc<Self>, VcfError> {
        let mut h = ptr::null_mut();
        check(unsafe { fm_matrix_create(data.as_ptr(), missing.map_or(ptr::null(), |m| m.as_ptr()),
                                        variants, samples, ploidy, max_allele, positions.as_ptr(), &mut h) })?;
        Ok(Arc::new(GpuMatrix(h)))
    }
    pub fn group(self: &Arc<Self>, haps: &[(usize, crate::stats::HaplotypeSide)]) -> Result<GpuGroup, VcfError> {
        let idx: Vec<u64> = haps.iter().map(|h| h.0 as u64).collect();
        let side: Vec<u8> = haps.iter().map(|h| matches!(h.1, crate::stats::HaplotypeSide::Right) as u8).collect();
        let mut g = ptr::null_mut();
        check(unsafe { fm_group_create(self.0, idx.as_ptr(), side.as_ptr(), haps.len(), &mut g) })?;
        Ok(GpuGroup(g, self.clone()))
    }
}

// ---- round 2: packed ingest (2 bits, or 1 bit + sparse missing list, per genotype over PCIe), batched summaries,
//      sharded Hudson call, device selection.  include/ferromic_gpu.h is the authority for every signature.
#[repr(C)] pub struct fm_ingest { _p: [u8; 0] }
#[repr(C)] #[derive(Default, Clone, Copy)]
pub struct fm_hudson_sums { pub num: f64, pub den: f64, pub dxy: f64, pub pi1: f64, pub pi2: f64,
                            pub dxy_uncallable: u64, pub unc1: u64, pub unc2: u64 }
pub const FM_MISSING_NONE: c_int = 0;
pub const FM_MISSING_BITMAP: c_int = 1;
pub const FM_MISSING_IN_BAND: c_int = 2;
extern "C" {
    pub fn fm_set_devices(devices: *const c_int, n: usize) -> c_int;            // or env FERROMIC_GPU_DEVICES
    pub fn fm_get_devices(out: *mut c_int, capacity: usize, n_out: *mut usize) -> c_int;
    pub fn fm_packed_row_words(n_samples: usize, ploidy: usize, row_words: *mut usize) -> c_int;
    pub fn fm_pack_rows(rows: *const u8, missing_whole: *const u64, missing_mode: c_int, first_row: usize, n_rows: usize,
                        n_total_rows: usize, stride: usize, allele_bits: *mut u32, called_bits: *mut u32,
                        n_threads: c_int) -> c_int;
    pub fn fm_pack_rows_sparse(rows: *const u8, missing_whole: *const u64, missing_mode: c_int, first_row: usize,
                               n_rows: usize, n_total_rows: usize, stride: usize, allele_bits: *mut u32,
                               row_missing_start: *mut u64, missing_cols: *mut core::ffi::c_void, capacity: usize,
                               col_bytes: c_int, n_threads: c_int, needed: *mut usize) -> c_int;
    pub fn fm_ingest_begin(v: usize, s: usize, ploidy: usize, has_missing: c_int, max_allele: u8, positions: *const i64,
                           chunk_rows_or_0: usize, out: *mut *mut fm_ingest) -> c_int;
    pub fn fm_ingest_add_group(h: *mut fm_ingest, sample_idx: *const u64, side: *const u8, n: usize,
                               group_index: *mut usize) -> c_int;
    pub fn fm_ingest_add_partition(h: *mut fm_ingest, left: *const u16, right: *const u16, n_samples: usize,
                                   n_groups: usize, partition_index: *mut usize) -> c_int;
    pub fn fm_ingest_rows(h: *mut fm_ingest, rows: *const u8, missing_whole: *const u64, first_row: usize,
                          n_rows: usize) -> c_int;
    pub fn fm_ingest_rows_pack(h: *mut fm_ingest, rows: *const u8, missing_whole: *const u64, first_row: usize,
                               n_rows: usize, n_threads: c_int) -> c_int;
    pub fn fm_ingest_rows_packed(h: *mut fm_ingest, allele_bits: *const u32, called_bits: *const u32, first_row: usize,
                                 n_rows: usize) -> c_int;
    pub fn fm_ingest_request_tracks(h: *mut fm_ingest, group_index: *const usize, raw_haplotype_counts: *const usize,
                                    n_groups: usize, region_start: i64, region_end: i64, mask_intervals: *const i64,
                                    n_mask: usize, filtered_positions: *const i64, n_filtered: usize,
                                    pos_out: *mut i64, pi_out: *mut f64, theta_out: *mut f64, capacity: usize,
                                    n_out: *mut usize) -> c_int;
    pub fn fm_ingest_rows_packed_sparse(h: *mut fm_ingest, allele_bits: *const u32, row_missing_start: *const u64,
                                        missing_cols: *const core::ffi::c_void, col_bytes: c_int, first_row: usize,
                                        n_rows: usize) -> c_int;
    pub fn fm_ingest_finish(h: *mut fm_ingest, matrix_out: *mut *mut fm_matrix, groups_out: *mut *mut fm_group,
                            partitions_out: *mut *mut fm_partition) -> c_int;
    pub fn fm_ingest_abort(h: *mut fm_ingest) -> c_int;
    pub fn fm_matrix_create_packed(allele_bits: *const u32, called_bits: *const u32, v: usize, s: usize, ploidy: usize,
                                   positions: *const i64, out: *mut *mut fm_matrix) -> c_int;
    pub fn fm_matrix_create_packed_sparse(allele_bits: *const u32, row_missing_start: *const u64,
                                          missing_cols: *const core::ffi::c_void, col_bytes: c_int, v: usize, s: usize,
                                          ploidy: usize, positions: *const i64, out: *mut *mut fm_matrix) -> c_int;
    pub fn fm_groups_summary_batch(groups: *const *mut fm_group, n_groups: usize, seg: *mut u64, pi_sum: *mut f64,
                                   unc: *mut u64) -> c_int;
    pub fn fm_hudson_pair_sharded(g1: *mut fm_group, g2: *mut fm_group, sequence_length: i64, raw_n1: usize,
                                  raw_n2: usize, comm: *mut fm_comm, out: *mut fm_hudson_outcome,
                                  merged: *mut fm_hudson_sums) -> c_int;
}

/// `DenseGenotypeMatrix::from_variants` (stats.rs:339-500) for the GPU path: instead of the u8 matrix + bitmap the
/// row loop writes one allele bit per cell and the columns of the missing cells, and hands them over in row blocks.
/// `rows()` yields (allele_bits, row_missing_start, missing_cols) blocks; 1.2 bits per genotype cross PCIe.
pub struct PackedIngest { h: *mut fm_ingest, n_groups: usize }
impl PackedIngest {
    pub fn begin(variants: usize, samples: usize, ploidy: usize, positions: &[i64]) -> Result<Self, VcfError> {
        let mut h = ptr::null_mut();
        check(unsafe { fm_ingest_begin(variants, samples, ploidy, FM_MISSING_BITMAP, 1, positions.as_ptr(), 0, &mut h) })?;
        Ok(PackedIngest { h, n_groups: 0 })
    }
    pub fn add_group(&mut self, haps: &[(usize, crate::stats::HaplotypeSide)]) -> Result<usize, VcfError> {
        let idx: Vec<u64> = haps.iter().map(|h| h.0 as u64).collect();
        let side: Vec<u8> = haps.iter().map(|h| matches!(h.1, crate::stats::HaplotypeSide::Right) as u8).collect();
        let mut gi = 0usize;
        check(unsafe { fm_ingest_add_group(self.h, idx.as_ptr(), side.as_ptr(), haps.len(), &mut gi) })?;
        self.n_groups += 1;
        Ok(gi)
    }
    /// Per-site pi / theta of declared groups, produced chunk by chunk while the rows upload (call between
    /// `add_group` and the first `push_*`).  The output slices must stay alive and unmoved until `finish()`; page-locked
    /// ones (cudaHostAlloc / cudaHostRegister) receive the values straight from the kernels.  Returns the number of sites.
    pub fn request_tracks(&mut self, groups: &[usize], raw_counts: &[usize], region: (i64, i64), mask: &[(i64, i64)],
                          pos_out: &mut [i64], pi_out: &mut [f64], theta_out: &mut [f64], capacity: usize)
                          -> Result<usize, VcfError> {
        assert!(pi_out.len() >= groups.len() * capacity && theta_out.len() >= groups.len() * capacity);
        let mut n = 0usize;
        check(unsafe { fm_ingest_request_tracks(self.h, groups.as_ptr(), raw_counts.as_ptr(), groups.len(), region.0,
                                                region.1, mask.as_ptr() as *const i64, mask.len(), ptr::null(), 0,
                                                pos_out.as_mut_ptr(), pi_out.as_mut_ptr(), theta_out.as_mut_ptr(),
                                                capacity, &mut n) })?;
        Ok(n)
    }
    pub fn push_sparse(&mut self, first_row: usize, n_rows: usize, allele_bits: &[u32], row_start: &[u64],
                       missing_cols: &[u16]) -> Result<(), VcfError> {
        check(unsafe { fm_ingest_rows_packed_sparse(self.h, allele_bits.as_ptr(), row_start.as_ptr(),
                                                    missing_cols.as_ptr() as *const _, 2, first_row, n_rows) })
    }
    /// The same list as one-byte gap codes (col_bytes = 1, include/ferromic_gpu.h): per row the position starts at
    /// -1; a byte b < 255 moves it b + 1 columns on and names that cell, 255 moves it 255 columns on without a cell.
    /// `row_start` counts bytes.
    pub fn push_gaps(&mut self, first_row: usize, n_rows: usize, allele_bits: &[u32], row_start: &[u64],
                     gap_codes: &[u8]) -> Result<(), VcfError> {
        check(unsafe { fm_ingest_rows_packed_sparse(self.h, allele_bits.as_ptr(), row_start.as_ptr(),
                                                    gap_codes.as_ptr() as *const _, 1, first_row, n_rows) })
    }
    pub fn finish(self) -> Result<(Arc<GpuMatrix>, Vec<GpuGroup>), VcfError> {
        let mut m = ptr::null_mut();
        let mut gs = vec![ptr::null_mut(); self.n_groups.max(1)];
        check(unsafe { fm_ingest_finish(self.h, &mut m, gs.as_mut_ptr(), ptr::null_mut()) })?;
        let m = Arc::new(GpuMatrix(m));
        let groups = gs.into_iter().take(self.n_groups).map(|g| GpuGroup(g, m.clone())).collect();
        std::mem::forget(self);
        Ok((m, groups))
    }
}
impl Drop for PackedIngest { fn drop(&mut self) { unsafe { fm_ingest_abort(self.h); } } }
