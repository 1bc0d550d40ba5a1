// fm_haplotypes.cuh -- the cells of a haplotype set and the site filter shared by haplotype PCA and haplotype LD
// (DESIGN.md §4 "Haplotype PCA" and "Haplotype LD"; filters in include/ferromic_gpu.h).
#pragma once
#include "fm_device.cuh"

namespace fm {

// One cell of a resident matrix, in any of its forms: u8 rows (bitmap, in-band or no missingness) or packed rows.
// `alt` is the RAW allele value 1 (never a rank of the LUT), `other` a called value other than 0 and 1.
struct HapCells {
    const uint8_t *data;
    const uint64_t *missing;
    uint32_t miss_mode;  // 0 none, 1 bitmap, 2 in band (cells >= 0x80)
    uint64_t stride;
    const uint32_t *abits, *cbits;  // packed rows (abits != nullptr); cbits may be null
    uint32_t rw;
    __device__ __forceinline__ void read(uint32_t v, uint32_t col, bool &called, bool &alt, bool &other) const {
        if (abits) {
            const size_t w = (size_t)v * rw + (col >> 5);
            alt = (__ldg(abits + w) >> (col & 31)) & 1u;
            called = cbits ? ((__ldg(cbits + w) >> (col & 31)) & 1u) : true;
            other = false;
            return;
        }
        const uint64_t e = (uint64_t)v * stride + col;
        const uint8_t x = __ldg(data + e);
        called = miss_mode == 1 ? ((__ldg(missing + (e >> 6)) >> (e & 63)) & 1ull) == 0 : (miss_mode == 2 ? x < 0x80 : true);
        alt = called && x == 1;
        other = called && x > 1;
    }
};

// Site statistics: one warp per site of [v_lo, v_lo + n_sites); counts over the n selected cells and the keep flag.
// *incomplete |= 1 when a kept site has a missing cell among the n (the callers then build a called plane).  `allow`
// (nullable, one flag per site of the range) limits the kept sites to a caller's site list.
__global__ void __launch_bounds__(256)
fm_k_hap_site_stats(HapCells cells, const uint32_t *__restrict__ off, uint32_t n, uint32_t v_lo, uint32_t n_sites,
                    double min_maf, double max_missing, const uint8_t *__restrict__ allow, uint32_t *__restrict__ alt_out,
                    uint32_t *__restrict__ called_out, uint8_t *__restrict__ keep_out, uint32_t *__restrict__ incomplete) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= n_sites) return;
    const uint32_t v = v_lo + r;
    uint32_t called = 0, alt = 0, other = 0;
    for (uint32_t i = lane; i < n; i += 32) {
        bool c, a, o;
        cells.read(v, __ldg(off + i), c, a, o);
        called += c;
        alt += a;
        other += o;
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) {
        called += __shfl_xor_sync(0xffffffffu, called, d);
        alt += __shfl_xor_sync(0xffffffffu, alt, d);
        other += __shfl_xor_sync(0xffffffffu, other, d);
    }
    if (lane) return;
    const uint32_t minor = min(alt, called - alt);
    const bool keep = other == 0 && alt > 0 && alt < called && (double)(n - called) <= max_missing * (double)n &&
                      (double)minor >= min_maf * (double)called && (!allow || allow[r]);
    alt_out[r] = alt;
    called_out[r] = called;
    keep_out[r] = keep;
    if (keep && called < n) atomicOr(incomplete, 1u);
}

// allow[list[i] - v_lo] = 1 for the entries of a site list that fall in [v_lo, v_lo + n_sites) (allow cleared first).
__global__ void __launch_bounds__(256)
fm_k_hap_allow(const uint64_t *__restrict__ list, uint64_t len, uint32_t v_lo, uint32_t n_sites,
               uint8_t *__restrict__ allow) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= len) return;
    const uint64_t v = list[i];
    if (v >= v_lo && v - v_lo < n_sites) allow[v - v_lo] = 1;
}

}  // namespace fm
