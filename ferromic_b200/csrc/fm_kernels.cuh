// fm_kernels.cuh -- sm_100a kernels of the per-site estimator path.
//
//   K1  fm_k_repack              u8 matrix (+ missing bitmap)  ->  per-group bitplanes
//   K2  fm_k_plane_pass_seq      a list of (group, site range) segments, one group or a Hudson pair per unit
//                                -> alt/called counts, pi/theta tracks, S, sum pi (+ fused Hudson components)
//   K2c fm_k_plane_pass_chunked  one group with rows wider than a warp's ring, streamed in column chunks
//   K2'/K3' light kernels evaluating estimators from cached count arrays
//   K5  fm_k_window_*            segmented (window) reductions
//   fm_k_reduce_partials         deterministic second-level reduction of per-batch partials
//
// The plane pass is a persistent kernel: every warp owns a private ring of shared-memory
// stages filled by 1-D TMA bulk copies (cp.async.bulk + mbarrier) and consumes them with
// 128-bit LDS + __popc; per-site counts are transposed with warp shuffles so that the FP64
// epilogue runs with one site per lane (32 sites = one "batch").  All reductions have a fixed
// shape keyed by the global batch index, so results do not depend on grid size or GPU count.
#pragma once
#include "fm_device.cuh"

namespace fm {

constexpr int kWarpsPerCta = 16;
constexpr uint32_t kWarpSmemBytes = 14 * 1024;  // private staging ring of one warp (16 x 14 KB = 224 KB)
constexpr int kMaxStages = 6;
constexpr uint32_t kStepBytesTarget = 7 * 1024;  // preferred bytes per pipeline step (two stages per warp)
// Dynamic scheduler: same-address atomics serialise in L2 (~3.6 ns each on B200, which capped the
// pass at one batch per 3.6 ns), so the batch range is split over kSchedCounters counters that
// live in separate 128-byte lines; a CTA starts on its home range and steals from the others.
constexpr uint32_t kSchedCounters = 16;
constexpr uint32_t kSchedStrideWords = 32;
constexpr uint32_t kSuperBatches = 256;          // batches folded by fm_k_reduce_partials
constexpr int kBatchRing = 8;                    // claimed-batch ring per warp (> kMaxStages)

__device__ __forceinline__ double fm_warp_sum(double v) {
    // fixed-shape butterfly: identical association for every batch
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ uint32_t fm_warp_sum_u(uint32_t v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ------------------------------------------------------------------------------ K1 repack
// One warp builds 32-bit words with __ballot_sync: lane j handles haplotype k = 32*w + j of
// the group (offset table `off`, sorted/de-duplicated exactly like DenseMembership::build,
// stats.rs:1251-1284).  allele bit = (byte != 0) & called, called bit = !missing (or k < n
// when the matrix has no bitmap).  Words are written 32 at a time (one per lane, 128 B).
// Plane row = wq uint4 = 4*wq words; padding bits are zero.  `data` starts at row v_base and
// `missing` at bitmap word word_base, so a staged chunk of rows can be repacked in place.
// Biallelic groups of a matrix with missing data keep no called plane (called == nullptr): the
// row's called count is added to cnt[v] instead (zeroed by the caller; a row spans several warps).
__global__ void __launch_bounds__(256)
fm_k_repack(const uint8_t *__restrict__ data, const uint64_t *__restrict__ missing, size_t stride,
            const uint32_t *__restrict__ off, uint32_t n, uint32_t wq, uint32_t v_base, uint64_t word_base,
            uint32_t v_lo, uint32_t v_hi, uint32_t *__restrict__ allele, uint32_t *__restrict__ called,
            uint32_t *__restrict__ cnt, uint32_t n_bits, size_t plane_stride_words, uint32_t in_band,
            const uint8_t *__restrict__ lut) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t nwarps = (gridDim.x * blockDim.x) >> 5;
    const uint32_t words = wq * 4;
    const uint32_t wgroups = (words + 31) / 32;  // groups of 32 words (1024 haplotypes)
    const uint64_t total = (uint64_t)(v_hi - v_lo) * wgroups;
    for (uint64_t item = warp; item < total; item += nwarps) {
        const uint32_t v = v_lo + (uint32_t)(item / wgroups);
        const uint32_t wg = (uint32_t)(item % wgroups);
        const size_t base = (size_t)(v - v_base) * stride;  // offset inside `data` (row v_base first)
        const size_t bit_base = (size_t)v * stride;          // bit index in the whole-matrix bitmap
        uint32_t my_a[4] = {0, 0, 0, 0}, my_c = 0;
#pragma unroll 4
        for (uint32_t i = 0; i < 32; ++i) {
            const uint32_t w = wg * 32 + i;
            if (w >= words) break;  // warp-uniform
            const uint32_t k = w * 32 + lane;
            uint32_t byte = 0;
            bool c = false;
            if (k < n) {
                const uint32_t o = off[k];
                c = true;
                if (missing) {
                    const size_t bit = bit_base + o;
                    c = !((missing[(bit >> 6) - word_base] >> (bit & 63)) & 1ull);
                }
                byte = data[base + o];
                if (in_band) c = byte < 0x80u;  // in-band missingness: a negative int8 cell
                if (!c) byte = 0u;
                else if (lut) byte = __ldg(lut + byte);  // allele values above 15: order-preserving dense ranks
            }
            const uint32_t wc = __ballot_sync(0xffffffffu, c);
            if (n_bits == 1) {  // biallelic: any non-zero allele index is the alternate allele
                const uint32_t wa = __ballot_sync(0xffffffffu, byte != 0);
                if (i == lane) my_a[0] = wa;
            } else {            // bit b of the allele index goes to plane b
#pragma unroll
                for (uint32_t b = 0; b < 4; ++b) {  // compile-time indices keep my_a in registers
                    if (b < n_bits) {
                        const uint32_t wa = __ballot_sync(0xffffffffu, (byte >> b) & 1u);
                        if (i == lane) my_a[b] = wa;
                    }
                }
            }
            if (i == lane) my_c = wc;
        }
        const uint32_t w = wg * 32 + lane;
        if (w < words) {
#pragma unroll
            for (uint32_t b = 0; b < 4; ++b)
                if (b < n_bits) allele[b * plane_stride_words + (size_t)v * words + w] = my_a[b];
            if (called) called[(size_t)v * words + w] = my_c;
        }
        if (cnt) {  // warp-uniform
            const uint32_t c = fm_warp_sum_u(w < words ? __popc(my_c) : 0u);
            if (lane == 0 && c) atomicAdd(cnt + v, c);
        }
    }
}

// ------------------------------------------------------------------------------ K1 v2 repack
// Row-staged, multi-group repack: one warp owns one matrix row at a time.  It pulls the row's
// u8 cells (128-bit loads) and the row's slice of the missing bitmap into its shared-memory
// slice once, then builds the bitplane words of EVERY listed group from shared memory with
// __ballot_sync -- the u8 matrix is read exactly once however many groups (a 27-group W&C
// partition, the two orientation groups of a per-site call) are repacked, and the per-lane byte
// gathers hit shared memory instead of paying an L2 round trip each (K1 v1 ran at ~0.4 TB/s).
struct RepackGroup {
    const uint32_t *off;       // sorted, de-duplicated column offsets (DenseMembership, stats.rs:1251-1284)
    uint32_t n, wq, n_bits;
    uint32_t *allele, *called; // called plane: multi-allelic groups of a matrix with missing data only
    size_t plane_stride_words; // distance between allele bit planes (multi-allelic groups)
    // count-only groups (the subpopulations of a W&C partition): no bitplanes are kept, the
    // per-site alt / called counts -- all K4 ever reads -- are produced straight from the staged row
    uint32_t *alt_out, *cnt_out;
    // biallelic plane groups: the group's plane row is a bit COMPRESS of the full-row bit words by the
    // membership mask (offsets are sorted).  One plan entry (two uint4) per row word the group touches:
    // {row word, member mask, first output bit, mv0} {mv1, mv2, mv3, mv4} -- mv = the precomputed move masks
    // of the parallel-suffix compress (Hacker's Delight 7-4), so a lane extracts its word's members in
    // 5 x 4 logic ops instead of one ballot per 32 haplotypes.
    const uint4 *plan;
    uint32_t n_ent;
    // tail layout (plan path only): the plane row holds the wq FULL 16-byte words of the group; the remaining
    // n % 128 haplotypes go to tw = ceil((n % 128) / 32) u32 words per row in a separate array (tw == 0: padded rows)
    uint32_t *tail_a;
    uint32_t tw;
    // biallelic groups of a matrix with missing data: the called count of every row (u32 [V]) in place of a
    // called plane -- every consumer only ever reduces the group's called bits of a row to this one number
    uint32_t *cnt;
};

__device__ __forceinline__ uint32_t fm_compress32(uint32_t x, const uint4 p0, const uint4 p1) {
    uint32_t t;
    x &= p0.y;
    t = x & p0.w; x = (x ^ t) | (t >> 1);
    t = x & p1.x; x = (x ^ t) | (t >> 2);
    t = x & p1.y; x = (x ^ t) | (t >> 4);
    t = x & p1.z; x = (x ^ t) | (t >> 8);
    t = x & p1.w; x = (x ^ t) | (t >> 16);
    return x;
}

// Count-only groups (W&C subpopulations): the row is packed ONCE into full-row allele / called
// bit words in matrix column order (4 cells per lane and step, no gather); group g then owns a
// sparse list of (row word, membership mask) entries, lane = group, and its alt / called counts
// are masked popcounts -- the cost follows the number of row words a group touches (7 for a
// contiguous 190-haplotype population), not the number of haplotypes.
struct CountTable {
    const uint32_t *ent_start;  // [n_groups + 1]
    const uint32_t *ent_word;   // [n_entries] row word index (column >> 5)
    const uint32_t *ent_mask;   // [n_entries] member columns inside that word
    uint32_t *const *alt_out;   // [n_groups] -> [V]
    uint32_t *const *cnt_out;   // [n_groups] -> [V]
    uint32_t n_groups;
};

// Packed rows (SURVEY 8 f1, the 2-bit ingest format): row v of the cohort as rw = ceil(stride / 32) u32 words of
// allele bits (bit c & 31 of word c >> 5: cell c carries a non-zero allele and is called) and, when the matrix
// has missing data, rw words of called bits.  In this mode the kernel never sees u8 cells: the full-row bit
// words are loaded as they are (coalesced 4-byte loads) and every group is served from them.
struct PackedRows {
    const uint32_t *a;  // [rows][rw] allele bits, row v_base first; nullptr = u8 mode
    const uint32_t *c;  // [rows][rw] called bits or nullptr (every cell called)
    uint32_t rw;
};

// MODE: 0 = general (staged row, every group kind), 1 = direct rows (whole 16-byte rows read straight from global
// memory; groups are served from the full-row bit words only), 2 = packed rows.  Modes 1 and 2 compile without
// the ballot-gather paths (fewer registers, more resident warps).  BIAL: every cell is 0, 1 or (in band) missing,
// so the allele bit of a byte is its bit 0 -- three operations per four cells instead of seven.
template <int MODE, bool BIAL>
__global__ void __launch_bounds__(256, MODE == 0 ? 4 : 6)
fm_k_repack_rows(const uint8_t *__restrict__ data, size_t data_bytes, const uint64_t *__restrict__ missing,
                 size_t stride, uint32_t v_base, uint64_t word_base, uint32_t v_lo, uint32_t v_hi,
                 const RepackGroup *__restrict__ groups, uint32_t n_groups, uint32_t warp_smem_bytes,
                 uint32_t row_buf_bytes, uint32_t bit_buf_bytes, CountTable ct, uint32_t in_band,
                 uint32_t need_row_bits, uint32_t direct_rows_arg, PackedRows pk_arg, const uint8_t *__restrict__ lut) {
    constexpr uint32_t direct_rows = MODE == 1 ? 1u : 0u;
    PackedRows pk = pk_arg;
    if (MODE != 2) pk.a = nullptr;  // lets the compiler drop the packed path
    (void)direct_rows_arg;
    // direct_rows: every group is served from the full-row bit words (compress plans / count tables) and rows are
    // whole 16-byte words, so the u8 row is packed straight from global memory (coalesced 16-byte loads) and is
    // never staged: row_buf_bytes == 0, three times the resident warps per SM
    extern __shared__ __align__(16) uint8_t rp_smem[];
    constexpr uint32_t FULL = 0xffffffffu;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint8_t *rowb = rp_smem + (size_t)warp * warp_smem_bytes;                       // staged row bytes
    uint64_t *bits = reinterpret_cast<uint64_t *>(rowb + row_buf_bytes);             // staged bitmap words
    const uint32_t gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t GW = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t v = v_lo + gw; v < v_hi; v += GW) {
        // ---- stage the row: aligned 16-byte loads over [a0, a1) covering [row0, row0 + stride)
        const size_t row0 = (size_t)(v - v_base) * stride;
        const size_t a0 = row0 & ~(size_t)15;
        const uint32_t delta = (uint32_t)(row0 - a0);
        const size_t a1 = (row0 + stride + 15) & ~(size_t)15;
        const uint32_t nq = (uint32_t)((a1 - a0) >> 4);
        __syncwarp();
        // asynchronous 16-byte copies straight into shared memory: every chunk of the row is in
        // flight at once (no register staging, no per-iteration load latency)
        for (uint32_t q = lane; !direct_rows && !pk.a && q < nq; q += 32) {
            const size_t at = a0 + ((size_t)q << 4);
            if (at + 16 <= data_bytes) {
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(fm_smem_u32(rowb + ((size_t)q << 4))),
                             "l"(data + at)
                             : "memory");
            } else {  // last bytes of the buffer: never read past its end
                uint32_t w[4] = {0, 0, 0, 0};
                for (uint32_t b = 0; b < 16 && at + b < data_bytes; ++b) w[b >> 2] |= (uint32_t)data[at + b] << ((b & 3) * 8);
                *reinterpret_cast<uint4 *>(rowb + ((size_t)q << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
            }
        }
        const size_t bit0 = (size_t)v * stride;
        const uint64_t w0 = bit0 >> 6;
        if (missing) {
            const uint32_t nw = (uint32_t)(((bit0 + stride + 63) >> 6) - w0);
            for (uint32_t q = lane; q < nw; q += 32)
                asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(fm_smem_u32(bits + q)),
                             "l"(missing + (w0 - word_base + q))
                             : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncwarp();
        // 32-bit views for the inner loops: bit (brel + o) of the staged bitmap slice, byte rb[o]
        const uint32_t brel = (uint32_t)(bit0 - (w0 << 6));
        const uint32_t *bits32 = reinterpret_cast<const uint32_t *>(bits);
        const uint8_t *rb = rowb + delta;
        // ---- full-row bit words (allele != 0, called) in matrix column order; count-only groups take
        //      masked popcounts of them, biallelic plane groups compress them by their membership masks
        const uint32_t rw = (uint32_t)((stride + 31) >> 5);
        uint32_t *arow = reinterpret_cast<uint32_t *>(rowb + row_buf_bytes + bit_buf_bytes);
        uint32_t *crow = arow + rw + 1;
        uint32_t *outb = crow + rw + 1;  // one group's allele plane row while it is assembled
        if (pk.a) {  // packed rows: the full-row bit words arrive ready-made
            const size_t r0 = (size_t)(v - v_base) * pk.rw;
            const uint32_t tail = (uint32_t)stride & 31u;
            for (uint32_t w = lane; w < rw; w += 32) {
                uint32_t c = pk.c ? __ldg(pk.c + r0 + w) : FULL;
                if (tail && w == rw - 1) c &= (1u << tail) - 1u;  // bits past the last cell never count
                crow[w] = c;
                arow[w] = __ldg(pk.a + r0 + w) & c;
            }
            __syncwarp();
            for (uint32_t g = lane; g < ct.n_groups; g += 32) {  // count-only groups
                uint32_t a = 0, c = 0;
                const uint32_t e1 = __ldg(ct.ent_start + g + 1);
                for (uint32_t e = __ldg(ct.ent_start + g); e < e1; ++e) {
                    const uint32_t w = __ldg(ct.ent_word + e);
                    const uint32_t cw = crow[w] & __ldg(ct.ent_mask + e);
                    c += __popc(cw);
                    a += __popc(arow[w] & cw);
                }
                ct.alt_out[g][v] = a;
                ct.cnt_out[g][v] = c;
            }
        } else if (need_row_bits) {
            const uint32_t *row32 = reinterpret_cast<const uint32_t *>(rowb + (delta & ~3u));
            const uint32_t sh8 = (delta & 3u) * 8u;
            // rows that start on a 16-byte boundary (stride % 16 == 0, e.g. 5008 or 200000 haplotypes): 16 cells per
            // lane and step (one LDS.128, four nibbles), two lanes per row word; otherwise 4 cells per lane
            const bool wide = direct_rows || (delta & 15u) == 0u;
            if (wide) {
                const uint4 *row128 = direct_rows ? reinterpret_cast<const uint4 *>(data + row0)
                                                  : reinterpret_cast<const uint4 *>(rowb + delta);
                const uint32_t nq16 = ((uint32_t)stride + 15u) >> 4;
                // bit 7 of every non-zero byte (the add only sees 7-bit fields: no carry crosses bytes), gathered by one multiply
                auto nib = [](uint32_t w) {
                    if (BIAL) return ((w & 0x01010101u) * 0x01020408u) >> 24;  // cells are 0 / 1 (missing ones are masked later)
                    return (((((w & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | w) >> 7 & 0x01010101u) * 0x01020408u) >> 24;
                };
                auto cnib = [](uint32_t w) { return (((~w >> 7) & 0x01010101u) * 0x01020408u >> 24) & 0xFu; };
                // four 16-byte loads per lane are issued before the first is consumed (direct mode reads global memory)
                for (uint32_t base = 0; base < nq16; base += 128) {
                    uint4 xq[4];
#pragma unroll
                    for (uint32_t u = 0; u < 4; ++u) {
                        const uint32_t q = base + u * 32u + lane;
                        xq[u] = make_uint4(0, 0, 0, 0);
                        if (q < nq16) xq[u] = direct_rows ? __ldg(row128 + q) : row128[q];
                    }
#pragma unroll
                    for (uint32_t u = 0; u < 4; ++u) {
                        const uint32_t q = base + u * 32u + lane;
                        if (base + u * 32u >= nq16) break;  // warp-uniform
                        uint4 x = xq[u];
                        if (q < nq16) {
                            const uint32_t left = (uint32_t)stride - q * 16u;  // cells that exist in this group
                            if (left < 16u) {
                                uint32_t xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
                                for (uint32_t k = 0; k < 4; ++k) {
                                    const uint32_t have = left > 4u * k ? min(4u, left - 4u * k) : 0u;
                                    xs[k] = have >= 4u ? xs[k] : (have ? xs[k] & ((1u << (8u * have)) - 1u) : 0u);
                                }
                                x = make_uint4(xs[0], xs[1], xs[2], xs[3]);
                            }
                        }
                        const uint32_t a16 = nib(x.x) | (nib(x.y) << 4) | (nib(x.z) << 8) | (nib(x.w) << 12);
                        const uint32_t ao = __shfl_xor_sync(FULL, a16, 1);
                        const uint32_t w = q >> 1;
                        if (!(lane & 1u) && w < rw) arow[w] = a16 | (ao << 16);
                        if (in_band) {  // called = cell < 0x80 (a non-negative int8); absent cells read 0 and are masked below
                            const uint32_t c16 = cnib(x.x) | (cnib(x.y) << 4) | (cnib(x.z) << 8) | (cnib(x.w) << 12);
                            const uint32_t co = __shfl_xor_sync(FULL, c16, 1);
                            if (!(lane & 1u) && w < rw) crow[w] = c16 | (co << 16);
                        }
                    }
                }
            }
            for (uint32_t i = 0; !wide && i * 128u < (uint32_t)stride; ++i) {
                const uint32_t col = (i * 32u + lane) * 4u;  // first of this lane's 4 columns
                uint32_t x = 0;
                if (col < (uint32_t)stride) {
                    const uint32_t q = i * 32u + lane;
                    x = __funnelshift_r(row32[q], row32[q + 1], sh8);
                    const uint32_t left = (uint32_t)stride - col;  // columns that exist
                    if (left < 4u) x &= (1u << (8u * left)) - 1u;
                }
                const uint32_t y = __vcmpne4(x, 0u) & 0x01010101u;
                uint32_t wv = (((y * 0x01020408u) >> 24) & 0xFu) << (4u * (lane & 7u));
                wv |= __shfl_xor_sync(FULL, wv, 1);
                wv |= __shfl_xor_sync(FULL, wv, 2);
                wv |= __shfl_xor_sync(FULL, wv, 4);
                const uint32_t w = i * 4u + (lane >> 3);
                if ((lane & 7u) == 0 && w < rw) arow[w] = wv;
                if (in_band) {  // called = cell < 0x80 (a non-negative int8)
                    const uint32_t z = (~x >> 7) & 0x01010101u;
                    uint32_t cv = (((z * 0x01020408u) >> 24) & 0xFu) << (4u * (lane & 7u));
                    cv |= __shfl_xor_sync(FULL, cv, 1);
                    cv |= __shfl_xor_sync(FULL, cv, 2);
                    cv |= __shfl_xor_sync(FULL, cv, 4);
                    if ((lane & 7u) == 0 && w < rw) crow[w] = cv;
                }
            }
            const uint32_t qb = brel >> 5, sb = brel & 31u;
            if (!in_band)
                for (uint32_t w = lane; w < rw; w += 32)
                    crow[w] = missing ? ~__funnelshift_r(bits32[w + qb], bits32[w + qb + 1], sb) : FULL;
            __syncwarp();
            for (uint32_t g = lane; g < ct.n_groups; g += 32) {  // count-only groups
                uint32_t a = 0, c = 0;
                const uint32_t e1 = __ldg(ct.ent_start + g + 1);
                for (uint32_t e = __ldg(ct.ent_start + g); e < e1; ++e) {
                    const uint32_t w = __ldg(ct.ent_word + e);
                    const uint32_t cw = crow[w] & __ldg(ct.ent_mask + e);
                    c += __popc(cw);
                    a += __popc(arow[w] & cw);
                }
                ct.alt_out[g][v] = a;  // dense_sum_alt_with_missing / _no_missing (stats.rs:1665-1697)
                ct.cnt_out[g][v] = c;
            }
        }
        // ---- every plane group's words from the staged row
        for (uint32_t gi = 0; gi < n_groups; ++gi) {
            const RepackGroup G = groups[gi];
            const uint32_t words = G.wq * 4 + G.tw;  // tw != 0 only on the plan path
            if (G.n_bits == 1 && G.plan) {
                uint32_t *oa = outb;
                for (uint32_t i = lane; i < words; i += 32) oa[i] = 0;
                __syncwarp();
                uint32_t nc = 0;  // called members of this lane's entries
                for (uint32_t e = lane; e < G.n_ent; e += 32) {
                    const uint4 p0 = __ldg(G.plan + 2 * e), p1 = __ldg(G.plan + 2 * e + 1);
                    const uint32_t cw = crow[p0.x];
                    nc += __popc(cw & p0.y);
                    const uint32_t xa = fm_compress32(arow[p0.x] & cw, p0, p1);
                    const uint32_t sh = p0.z & 31u, wi = p0.z >> 5;
                    // straight-line: the fragment's low part and the part that spills into the next word (zero when
                    // sh == 0: the funnel shift yields the high word of (0 : x) << sh).  Nearly every fragment is
                    // non-empty and spills, so the four tests this replaces only cost issue slots and reconvergence
                    // barriers (ncu: 9 % BRA + 7 % BSSY / BSYNC of the kernel's instructions); or-ing a zero is free.
                    // The word after the row's last one is padding (repack_warp_smem).
                    atomicOr(oa + wi, xa << sh);
                    atomicOr(oa + wi + 1, __funnelshift_l(xa, 0u, sh));
                }
                if (G.cnt) {  // warp-uniform
                    nc = fm_warp_sum_u(nc);
                    if (lane == 0) G.cnt[v] = nc;
                }
                __syncwarp();
                const uint32_t fw = G.wq * 4;
                for (uint32_t i = lane; i < fw; i += 32) G.allele[(size_t)v * fw + i] = oa[i];
                if (lane < G.tw) G.tail_a[(size_t)v * G.tw + lane] = oa[fw + lane];  // the row's last n % 128 haplotypes
                __syncwarp();
                continue;
            }
            if (MODE != 0) continue;  // direct / packed launches only carry plan groups (checked on the host)
            if (G.n_bits == 1) continue;  // every biallelic group of a staged row takes its compress plan
            for (uint32_t wb = 0; wb < words; wb += 32) {  // multi-allelic: bit b of the allele index -> plane b
                uint32_t my_a[4] = {0, 0, 0, 0}, my_c = 0;
                const uint32_t lim = min(32u, words - wb);
                for (uint32_t i = 0; i < lim; ++i) {
                    const uint32_t k = (wb + i) * 32 + lane;
                    uint32_t byte = 0;
                    bool c = false;
                    if (k < G.n) {
                        const uint32_t o = __ldg(G.off + k);
                        c = true;
                        byte = rb[o];
                        if (missing) {
                            const uint32_t r = brel + o;
                            c = !((bits32[r >> 5] >> (r & 31u)) & 1u);
                        } else if (in_band) {
                            c = byte < 0x80u;
                        }
                        if (!c) byte = 0u;
                        else if (lut) byte = __ldg(lut + byte);  // allele values above 15: dense ranks
                    }
                    const uint32_t wc = __ballot_sync(FULL, c);
#pragma unroll
                    for (uint32_t b = 0; b < 4; ++b) {  // compile-time indices keep my_a in registers
                        if (b < G.n_bits) {
                            const uint32_t wa = __ballot_sync(FULL, (byte >> b) & 1u);
                            if (i == lane) my_a[b] = wa;
                        }
                    }
                    if (i == lane) my_c = wc;
                }
                if (lane < lim) {
                    const size_t o = (size_t)v * words + wb + lane;
#pragma unroll
                    for (uint32_t b = 0; b < 4; ++b)
                        if (b < G.n_bits) G.allele[b * G.plane_stride_words + o] = my_a[b];
                    if (G.called) G.called[o] = my_c;
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------ sparse missing list -> called plane
// Packed rows may arrive with a sparse list of missing cells instead of a called plane (0.15 instead of 1 bit per
// genotype over PCIe at 1 % missing; 0.09 with the one-byte gap code, ColT = uint8_t).  One warp per row rebuilds the row's called words in shared memory -- all
// ones, the listed cells cleared -- and writes them to the resident packed matrix with coalesced stores.
//   start[r - r_base] .. start[r - r_base + 1]: the row's slice of `cols` (indices relative to cols_base)
template <typename ColT>
__global__ void __launch_bounds__(256)
fm_k_expand_called(const uint64_t *__restrict__ start, const ColT *__restrict__ cols, uint64_t cols_base, uint32_t r_base,
                   uint32_t v_lo, uint32_t v_hi, uint32_t rw, uint32_t stride, uint32_t *__restrict__ cbits) {
    extern __shared__ uint32_t ex_smem[];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t *crow = ex_smem + (size_t)warp * rw;
    const uint32_t gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t GW = (gridDim.x * blockDim.x) >> 5;
    const uint32_t tail = stride & 31u;
    for (uint32_t v = v_lo + gw; v < v_hi; v += GW) {
        for (uint32_t w = lane; w < rw; w += 32) crow[w] = (tail && w == rw - 1) ? ((1u << tail) - 1u) : 0xffffffffu;
        __syncwarp();
        const uint64_t s0 = start[v - r_base], s1 = start[v - r_base + 1];
        if (sizeof(ColT) == 1) {
            // gap code: byte b < 255 = the missing cell b + 1 columns after the previous position, 255 = move on 255
            // columns without a cell; positions start at -1.  Warp-wide inclusive scan of the steps, 32 bytes at a time.
            uint32_t at = 0;  // position + 1 reached so far
            for (uint64_t i0 = s0; i0 < s1; i0 += 32) {
                const uint64_t i = i0 + lane;
                const uint32_t b = i < s1 ? (uint32_t)cols[i - cols_base] : 255u;
                uint32_t step = i < s1 ? (b == 255u ? 255u : b + 1u) : 0u;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t up = __shfl_up_sync(0xffffffffu, step, o);
                    if ((int)lane >= o) step += up;
                }
                const uint32_t c = at + step - 1u;  // at + step >= 1 whenever this lane holds a cell
                if (i < s1 && b != 255u && c < stride) atomicAnd(crow + (c >> 5), ~(1u << (c & 31u)));
                at += __shfl_sync(0xffffffffu, step, 31);
            }
        } else {
            for (uint64_t i = s0 + lane; i < s1; i += 32) {
                const uint32_t c = (uint32_t)cols[i - cols_base];
                if (c < stride) atomicAnd(crow + (c >> 5), ~(1u << (c & 31u)));
            }
        }
        __syncwarp();
        uint32_t *dst = cbits + (size_t)v * rw;
        for (uint32_t w = lane; w < rw; w += 32) dst[w] = crow[w];
        __syncwarp();
    }
}

// Which allele values occur in a u8 matrix (called cells only)?  256-bit presence set, for the order-preserving
// remap of matrices whose max_allele exceeds 15 (the bitplanes hold at most 4 bits per cell).
__global__ void __launch_bounds__(256)
fm_k_allele_presence(const uint8_t *__restrict__ data, const uint64_t *__restrict__ missing, uint64_t total,
                     uint32_t in_band, uint32_t *__restrict__ present /*[8]*/) {
    __shared__ uint32_t sp[8];
    if (threadIdx.x < 8) sp[threadIdx.x] = 0;
    __syncthreads();
    uint32_t mine[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t b = data[i];
        bool called = true;
        if (missing) called = !((missing[i >> 6] >> (i & 63)) & 1ull);
        else if (in_band) called = b < 0x80u;
        if (called) {
#pragma unroll
            for (int k = 0; k < 8; ++k)
                if ((b >> 5) == (uint32_t)k) mine[k] |= 1u << (b & 31u);
        }
    }
#pragma unroll
    for (int k = 0; k < 8; ++k)
        if (mine[k]) atomicOr(&sp[k], mine[k]);
    __syncthreads();
    if (threadIdx.x < 8 && sp[threadIdx.x]) atomicOr(&present[threadIdx.x], sp[threadIdx.x]);
}

// ------------------------------------------------------------------------------ synthetic cohorts
// Counter-based generator for benchmarks and full-size parity tests: every matrix entry is a pure
// integer function of (seed, site, column), so any slice can be re-evaluated on the CPU
// (tests/synth.py::synth_rows) without moving the matrix.  Site base frequency is U-shaped
// (x^2 mirrored), each population gets a uniform offset scaled by sigma_q, alleles are Bernoulli.
__host__ __device__ __forceinline__ uint64_t fm_splitmix64(uint64_t x) {
    uint64_t z = x + 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__host__ __device__ __forceinline__ uint64_t fm_mix(uint64_t seed, uint64_t a, uint64_t b) {
    return fm_splitmix64(fm_splitmix64(seed + a) + b);
}
__host__ __device__ __forceinline__ uint32_t fm_synth_threshold(uint64_t seed, uint64_t v, uint32_t pop,
                                                                uint32_t sigma_q) {
    const uint64_t hs = fm_mix(seed, v, 0);
    const uint32_t x = (uint32_t)(hs & 0xFFFFu);
    uint32_t y = (x * x) >> 16;
    if ((hs >> 16) & 1u) y = 65535u - y;
    const uint64_t hp = fm_mix(seed, v, 1u + pop);
    const int32_t d = ((int32_t)(hp & 0x1FFFu) - 4096) * (int32_t)sigma_q / 4096;
    int32_t t = (int32_t)y + d;
    t = t < 66 ? 66 : (t > 65470 ? 65470 : t);
    return (uint32_t)t;
}

// One thread per bitmap word = 64 consecutive entries of the linear layout.
__global__ void __launch_bounds__(256)
fm_k_synth(uint8_t *__restrict__ data, uint64_t *__restrict__ missing, uint64_t total, uint32_t stride,
           uint32_t ploidy, uint64_t first_variant, uint64_t seed, const uint16_t *__restrict__ pop_of_sample,
           uint32_t sigma_q, uint32_t miss_q) {
    const uint64_t n_words = (total + 63) / 64;
    for (uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < n_words;
         w += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t e0 = w * 64;
        uint64_t v = e0 / stride;
        uint32_t col = (uint32_t)(e0 - v * stride);
        uint64_t bits = 0;
        uint32_t packed[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) packed[i] = 0;
        uint32_t cur_pop = 0xFFFFFFFFu, thr = 0;
        uint64_t cur_v = ~0ull;
#pragma unroll 4
        for (uint32_t i = 0; i < 64; ++i) {
            if (e0 + i < total) {
                const uint32_t pop = pop_of_sample ? pop_of_sample[col / ploidy] : 0u;
                if (pop != cur_pop || v != cur_v) {
                    thr = fm_synth_threshold(seed, first_variant + v, pop, sigma_q);
                    cur_pop = pop;
                    cur_v = v;
                }
                const uint64_t he = fm_mix(seed, first_variant + v, 0x10000ull + col);
                const bool miss = (uint32_t)((he >> 32) & 0xFFFFu) < miss_q;
                const bool allele = (uint32_t)(he & 0xFFFFu) < thr;
                if (miss) bits |= 1ull << i;
                if (allele && !miss) packed[i >> 2] |= 1u << ((i & 3) * 8);
            }
            if (++col == stride) {
                col = 0;
                ++v;
            }
        }
        if (e0 + 64 <= total) {
            uint4 *dst = reinterpret_cast<uint4 *>(data + e0);
#pragma unroll
            for (int q = 0; q < 4; ++q)
                dst[q] = make_uint4(packed[4 * q], packed[4 * q + 1], packed[4 * q + 2], packed[4 * q + 3]);
        } else {
            for (uint32_t i = 0; e0 + i < total; ++i) data[e0 + i] = (uint8_t)((packed[i >> 2] >> ((i & 3) * 8)) & 0xFFu);
        }
        if (missing) missing[w] = bits;
    }
}

// ------------------------------------------------------------------------------ plane pass
// A biallelic group's plane pass input.  The allele plane is masked with "called" (allele bit = non-zero allele and
// called), so alt = popc(allele row); the called count n comes from `cnt`, filled by K1 when the rows are repacked.
struct GroupPlanes {
    const uint4 *allele;
    const uint32_t *cnt;  // [V] called members per site; nullptr => every member haplotype is called (n = cap)
    uint32_t wq;          // uint4 per row
    uint32_t cap;         // haplotype capacity (offsets.len())
    // tail layout: the last cap % 128 haplotypes of every row live in tw u32 words per row (tail_a [V][tw]) instead
    // of a padded 16-byte word; the streaming pass reads them in the batch epilogue (lane = site).
    // Cuts the padding of a 3463 + 1545 haplotype pair from 4.8 % of the plane bytes to 1 %.
    const uint32_t *tail_a;
    uint32_t tw;
};

// tail words and called count of this lane's site, requested at the start of a batch (one coalesced load per
// array and warp) and consumed in its epilogue
struct TailRegs {
    uint32_t a[3], n;
};
__device__ __forceinline__ void fm_tail_load(const GroupPlanes &g, uint32_t v, uint32_t n_sites_total, TailRegs &t) {
#pragma unroll
    for (uint32_t k = 0; k < 3; ++k) t.a[k] = 0;
    t.n = g.cap;
    if (v < n_sites_total) {
        if (g.cnt) t.n = __ldg(g.cnt + v);
#pragma unroll
        for (uint32_t k = 0; k < 3; ++k)
            if (k < g.tw) t.a[k] = __ldg(g.tail_a + (size_t)v * g.tw + k);
    }
}
__device__ __forceinline__ void fm_tail_add(const TailRegs &t, uint32_t &alt, uint32_t &cnt) {
    alt += __popc(t.a[0]) + __popc(t.a[1]) + __popc(t.a[2]);
    cnt = t.n;
}

struct PassGeom {
    uint32_t n_chunks;    // column chunks per row (chunked pass)
    uint32_t cq;          // chunk width in uint4 (chunked pass)
    uint32_t n_stages;    // pipeline depth of the per-warp ring (2..kMaxStages)
    uint32_t stage_bytes; // bytes reserved per stage (multiple of 128)
    uint32_t warp_smem_bytes;  // private staging ring of one warp (n_stages * stage_bytes <= this)
    uint32_t warps;            // warps per CTA (<= kWarpsPerCta); warps * warp_smem_bytes <= 224 KB
    uint32_t v_lo, v_hi;
    uint32_t b_lo, n_batches;  // global batch range (batch b = sites [32b, 32b+32))
    uint32_t n_sites_total;    // V (rows available in the planes)
    uint32_t *batch_counter;   // dynamic scheduler counters (zeroed before launch)
};

// Diversity epilogue: build_dense_population_summary (stats.rs:1367-1470) +
// calculate_per_site_diversity (stats.rs:4693-4750) fused.
struct DivEpilogue {
    uint32_t *alt_out, *called_out;  // [V] or nullptr
    double *pi_out, *theta_out;      // [v_hi - v_lo] or nullptr   (tracks)
    const uint32_t *site_flags;      // [n_batches] bit i of word b-b_lo: site 32b+i is masked or
                                     // filtered (fm_k_site_flags); nullptr when nothing is dropped
    // per-group lookup tables indexed by the called count n = 0..cap.  They hold exactly the
    // values the reference computes per site (IEEE division is correctly rounded on host and
    // device alike): inv_n = 1/n, scale = n/(n-1), theta = 1/H_{n-1} with H by forward summation
    // (stats.rs:4234-4240, 4716-4722).
    const double *tab_inv_n, *tab_scale, *tab_theta;
    int pi_form;                     // formula used for the sum-of-pi partial
    double *part_pi;                 // [n_batches]
    uint32_t *part_u;                // [n_batches][2]: segregating sites, sites with called < 2
};

// Hudson epilogue of a pair of groups.
struct HudsonEpilogue {
    int variant;                           // FM_HV_* (per-site form) or -1 for the summaries form
    double *fst, *dxy, *pi1, *pi2, *num, *den;  // per-site [v_hi - v_lo] or nullptr
    uint32_t *n1_out, *n2_out;
    // per batch: 0 num, 1 den, 2 dxy_sum, 3 pi1_sum, 4 pi2_sum
    double *part_d;   // [n_batches][5]
    uint32_t *part_u; // [n_batches][3]: dxy_skipped, unc1 (n1<2), unc2 (n2<2)
};

__device__ __forceinline__ bool fm_in_intervals(const int64_t *iv, uint32_t n, int64_t pos) {
    // merged + sorted half-open intervals: find last start <= pos
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        uint32_t mid = (lo + hi) >> 1;
        if (iv[2 * mid] <= pos)
            lo = mid + 1;
        else
            hi = mid;
    }
    return lo > 0 && pos < iv[2 * (lo - 1) + 1];
}
__device__ __forceinline__ bool fm_in_sorted(const int64_t *a, uint32_t n, int64_t x) {
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        uint32_t mid = (lo + hi) >> 1;
        if (a[mid] < x)
            lo = mid + 1;
        else
            hi = mid;
    }
    return lo < n && a[lo] == x;
}

// Mask / filtered-position lookup hoisted out of the streaming kernel: one bit per site
// (stats.rs:4731-4743: position in filtered_positions or inside any mask interval [s,e)).
// One warp per batch; the result is a 32-bit word per batch.  Positions are ascending, so the
// warp locates the batch's first position among the merged, sorted intervals with a 32-ary
// search (3 dependent loads for 2,000 intervals instead of 11) and every lane then only walks
// forward over the few intervals that start inside the batch.
__global__ void __launch_bounds__(256)
fm_k_site_flags(const int64_t *__restrict__ pos, uint32_t v_lo, uint32_t v_hi, uint32_t b_lo,
                uint32_t n_batches, const int64_t *__restrict__ mask, uint32_t n_mask,
                const int64_t *__restrict__ filt, uint32_t n_filt, uint32_t *__restrict__ flags) {
    constexpr uint32_t FULL = 0xffffffffu;
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t GW = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t bi = gw; bi < n_batches; bi += GW) {
        const uint32_t vb = (b_lo + bi) * 32;
        const uint32_t v = vb + lane;
        const bool valid = v >= v_lo && v < v_hi;
        const int64_t p = valid ? pos[v] : 0;
        bool drop = false;
        if (valid && filt) drop = fm_in_sorted(filt, n_filt, p);
        if (mask && n_mask) {
            const uint32_t first = v_lo > vb ? v_lo - vb : 0u;  // first valid lane of the batch
            const int64_t p0 = __shfl_sync(FULL, p, first & 31u);
            // last interval with start <= p0, or -1: invariant start[lo] <= p0 < start[hi]
            int lo = -1, hi = (int)n_mask;
            while (hi - lo > 1) {
                const int step = (hi - lo - 1 + 31) / 32;
                const int idx = lo + 1 + (int)lane * step;
                const bool le = idx < hi && mask[2 * (size_t)idx] <= p0;
                const int k = __popc(__ballot_sync(FULL, le));  // probes are ascending: a prefix of ones
                const int nlo = k > 0 ? lo + 1 + (k - 1) * step : lo;
                const int nhi = min(hi, lo + 1 + k * step);
                lo = nlo;
                hi = nhi;
            }
            if (valid && !drop) {
                int j = lo;
                while (j + 1 < (int)n_mask && mask[2 * (size_t)(j + 1)] <= p) ++j;
                drop = j >= 0 && p < mask[2 * (size_t)j + 1];
            }
        }
        const uint32_t w = __ballot_sync(FULL, drop);
        if (lane == 0) flags[bi] = w;
    }
}

// Per-site diversity values (shared by the fused epilogue and the light kernel).
__device__ __forceinline__ void fm_div_site(const DivEpilogue &e, uint32_t v, uint32_t v_lo,
                                            uint32_t n, uint32_t alt, bool dropped, double &pi_part,
                                            uint32_t &seg, uint32_t &unc) {
    const bool poly = (n >= 2 && alt > 0 && alt < n);
    seg = poly ? 1u : 0u;       // stats.rs:1389 / 1406
    unc = (n < 2) ? 1u : 0u;    // stats.rs:1512-1516
    double pi_comp = 0.0;       // pi_from_components (stats.rs:2723-2733) via the tables
    if (n >= 2 && (e.pi_out || e.pi_form == FM_PIFORM_COMPONENTS)) {
        const double r = (double)(n - alt), a = (double)alt;
        const double sum_counts_sq = r * r + a * a;
        const double inv_n = __ldg(e.tab_inv_n + n);
        const double sum_p2 = sum_counts_sq * inv_n * inv_n;
        pi_comp = __ldg(e.tab_scale + n) * (1.0 - sum_p2);
    }
    if (e.pi_form == FM_PIFORM_COMPONENTS) {
        pi_part = pi_comp;
    } else {
        double val;
        pi_part = fm_pi_form(e.pi_form, n, alt, val) ? val : 0.0;
    }
    if (e.alt_out) e.alt_out[v] = alt;
    if (e.called_out) e.called_out[v] = n;
    if (e.pi_out) {
        // calculate_per_site_diversity, stats.rs:4710-4743
        double pi_value, theta_value;
        if (n < 2 || dropped) {
            pi_value = fm_nan();
            theta_value = fm_nan();
        } else {
            theta_value = poly ? __ldg(e.tab_theta + n) : 0.0;  // distinct_alleles > 1
            pi_value = pi_comp;
        }
        e.pi_out[v - v_lo] = pi_value;
        e.theta_out[v - v_lo] = theta_value;
    }
}

struct HudsonAcc {
    double num, den, dxy, pi1, pi2;
    uint32_t skipped, unc1, unc2;
};

// Per-site Hudson contributions. variant >= 0: per-site form (FM_HV_*), sums follow
// hudson_component_sums (stats.rs:1625-1635) + calculate_pi_dense / calculate_dxy_dense;
// variant < 0: aggregate_hudson_components_from_summaries (stats.rs:1554-1623).
__device__ __forceinline__ void fm_hudson_contrib(const HudsonEpilogue &e, uint32_t v, uint32_t v_lo,
                                                  uint32_t n1, uint32_t a1, uint32_t n2, uint32_t a2,
                                                  HudsonAcc &acc) {
    acc = HudsonAcc{0.0, 0.0, 0.0, 0.0, 0.0, 0u, 0u, 0u};
    acc.unc1 = n1 < 2;
    acc.unc2 = n2 < 2;
    if (e.variant < 0) {
        double dxy;
        if (!fm_dxy_summaries(n1, a1, n2, a2, dxy)) {
            acc.skipped = 1;
            return;
        }
        acc.dxy = dxy;
        if (n1 < 2 || n2 < 2) return;
        double p1 = fm_pi_summaries(n1, a1), p2 = fm_pi_summaries(n2, a2);
        acc.pi1 = p1;
        acc.pi2 = p2;
        if (dxy > FM_FST_EPSILON) {
            acc.num = dxy - 0.5 * (p1 + p2);
            acc.den = dxy;
        }
        return;
    }
    fm_hudson_vals o;
    fm_hudson_site(e.variant, n1, a1, n2, a2, o);
    if (o.num == o.num && o.den == o.den) {  // both Some
        acc.num = o.num;
        acc.den = o.den;
    }
    // regional Dxy via calculate_dxy_dense / sparse fold (dot form), skipped when a pop is empty
    double d;
    if (fm_dxy_dot(n1, a1, n2, a2, d))
        acc.dxy = d;
    else
        acc.skipped = 1;
    // regional pi via calculate_pi_dense(_biallelic) or calculate_pi (same form as the site pi)
    if (o.pi1 == o.pi1) acc.pi1 = o.pi1;
    if (o.pi2 == o.pi2) acc.pi2 = o.pi2;
    if (e.fst) {
        const uint32_t i = v - v_lo;
        e.fst[i] = o.fst;
        e.dxy[i] = o.dxy;
        e.pi1[i] = o.pi1;
        e.pi2[i] = o.pi2;
        e.num[i] = o.num;
        e.den[i] = o.den;
        e.n1_out[i] = n1;
        e.n2_out[i] = n2;
    }
}

// ------------------------------------------------------------------------------ plane pass: shared pieces
// Both plane-pass kernels are persistent: every warp owns a private ring of n_stages shared-memory stages with one
// mbarrier each.  Lane 0 fills a stage with one TMA bulk copy and the whole warp waits on its barrier phase.
__device__ __forceinline__ void fm_ring_init(uint32_t bar_base, uint32_t n_stages, uint32_t lane) {
    if (lane == 0) {
        for (uint32_t s = 0; s < n_stages; ++s)
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_base + 8u * s));
        fm_fence_mbar_init();
    }
    __syncwarp();
}

// lane 0: copy `bytes` from global memory into the stage at `dst`, completing on the stage's barrier `bar`;
// bytes == 0 (a step past the last row) completes the phase with a plain arrive
__device__ __forceinline__ void fm_ring_fill(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    if (bytes == 0) {
        asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
        return;
    }
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}

__device__ __forceinline__ void fm_ring_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    } while (!ok);
}

// Dynamic batch scheduler of one warp.  The batch range [0, n_batches) is split over kSchedCounters counters; a
// warp starts on its CTA's home range and steals from the others.  The issue side claims batches and the consume
// side replays the same sequence from a small per-warp ring.  Partials are keyed by the batch index, so the
// result does not depend on which warp processed which batch.  The atomic is fired one batch ahead so its round
// trip never sits on the critical path.
struct BatchScheduler {
    uint32_t *counters;
    uint32_t n_batches, j, tried, prefetched;
    __device__ __forceinline__ BatchScheduler(uint32_t *c, uint32_t nb, uint32_t lane)
        : counters(c), n_batches(nb), j(blockIdx.x % kSchedCounters), tried(0), prefetched(0) {
        if (lane == 0) prefetched = atomicAdd(counters + j * kSchedStrideWords, 1u);
    }
    __device__ __forceinline__ uint32_t range_lo(uint32_t k) const {
        return (uint32_t)(((uint64_t)n_batches * k) / kSchedCounters);
    }
    // next batch of the launch (warp-uniform), or 0xffffffff once every range is drained
    __device__ __forceinline__ uint32_t claim(uint32_t lane) {
        for (;;) {
            const uint32_t idx = __shfl_sync(0xffffffffu, prefetched, 0);
            const uint32_t lo = range_lo(j), hi = range_lo(j + 1);
            if (idx < hi - lo) {  // fire the next claim on the same range, one batch ahead
                if (lane == 0) prefetched = atomicAdd(counters + j * kSchedStrideWords, 1u);
                return lo + idx;
            }
            if (++tried == kSchedCounters) return 0xffffffffu;
            j = (j + 1 == kSchedCounters) ? 0 : j + 1;
            if (lane == 0) prefetched = atomicAdd(counters + j * kSchedStrideWords, 1u);
        }
    }
};

// Diversity epilogue of one batch, lane i <-> site v = 32b + i (all 32 lanes active): the per-site values of the
// sites in [v_lo, v_hi), then the batch's partials at index bl.
__device__ __forceinline__ void fm_div_batch(const DivEpilogue &e, uint32_t v, uint32_t v_lo, uint32_t v_hi,
                                             uint32_t bl, uint32_t lane, uint32_t n, uint32_t alt) {
    double pi_part = 0.0;
    uint32_t seg = 0, unc = 0;
    const uint32_t flags = e.site_flags ? __ldg(e.site_flags + bl) : 0u;
    if (v >= v_lo && v < v_hi) fm_div_site(e, v, v_lo, n, alt, (flags >> lane) & 1u, pi_part, seg, unc);
    const double s_pi = fm_warp_sum(pi_part);
    const uint32_t s_u = fm_warp_sum_u(seg | (unc << 16));
    if (lane == 0) {
        e.part_pi[bl] = s_pi;
        e.part_u[2 * bl] = s_u & 0xffffu;
        e.part_u[2 * bl + 1] = s_u >> 16;
    }
}

// ------------------------------------------------------------------------------ plane pass, rows
// fm_k_plane_pass_seq: one persistent launch streams a LIST of plane segments.  A unit is one segment or, in the PAIR
// instances, two segments over the same sites:
//   * one segment per unit: independent (group, site range) units share one launch -- the groups of one per-site call, the
//     per-region matrices the CLI builds one after the other (process.rs:2169), each with its own population --
//     so many small passes stream at the rate of one large one, and the launch ramp-up and the end-of-kernel
//     quantisation are paid once;
//   * PAIR: a warp streams the batch of group 1, keeps its counts in registers, streams the same batch of
//     group 2 and evaluates the Hudson components of the 32 sites in place (stats.rs:3179-3278 / 1554-1623) --
//     both groups' counts and summary partials AND the Hudson partials from one sweep of the planes.
// The batch index space is the concatenation of the units' batch ranges.  A step holds `rounds` x SPS consecutive
// sites of one segment (SPS = 32/LPS sites per round); in every round LPS consecutive lanes read consecutive uint4
// of one row, so a quarter-warp always touches one contiguous 128-byte span (bank-conflict free without padding).
constexpr int kMaxSeq = 4;  // segments carried in the kernel parameters (no descriptor upload)

struct RowSeg {
    GroupPlanes g;
    DivEpilogue div;          // div.part_pi == nullptr: no diversity epilogue
    uint32_t rounds;          // rounds of (32/lps) sites per pipeline step for this segment's row width
    uint32_t v_lo, v_hi;      // site range analysed
    uint32_t b_lo;            // first batch of the range (v_lo / 32)
    uint32_t n_sites_total;   // rows available in this segment's planes
    uint32_t pad;
};

struct RowParams {
    const RowSeg *segs;            // [n_units] (one segment per unit; the PAIR instances use the inline table only)
    const uint32_t *unit_prefix;   // [n_units + 1]: batches of the units before u (unit u has prefix[u+1]-prefix[u])
    uint32_t n_units;
    PassGeom geom;                 // n_stages, stage_bytes, warp_smem_bytes, n_batches (whole launch), counters
    // up to kMaxSeq segments travel in the kernel parameters themselves: a descriptor upload is three small H2D
    // copies (~20 us of a 250 us sharded step).  The INLINE instances read these instead of the pointers above.
    RowSeg inline_segs[kMaxSeq];
    HudsonEpilogue inline_hud[kMaxSeq / 2];  // PAIR: one Hudson epilogue per unit
    uint32_t inline_prefix[kMaxSeq + 1];
};
static_assert(sizeof(RowParams) <= 4096, "the row-pass parameters must fit the 4 KB kernel parameter space");

// INLINE: the table is read from the kernel parameters.  Those reads compile to constant-bank loads, which keep
// the per-batch segment lookups off the critical path; a pointer that may address either the parameters or global
// memory makes every one of them a generic load (that form took 10 % longer per bench step on a B200:
// profiles/r04_ab_one_table_variant.txt).  PAIR: two segments per unit and the Hudson epilogue; the one-segment
// instances compile without them (the bench step and single groups run the smaller kernel).
template <int LG, bool INLINE, bool PAIR>
__global__ void __launch_bounds__(kWarpsPerCta * 32, 1)
fm_k_plane_pass_seq(const __grid_constant__ RowParams P) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bars[kWarpsPerCta * kMaxStages];
    __shared__ uint32_t batch_ring[kWarpsPerCta * kBatchRing];
    static_assert(LG < 5, "column-chunked rows take fm_k_plane_pass_chunked");
    static_assert(INLINE || !PAIR, "pair units travel in the kernel parameters");
    constexpr uint32_t LPS = 1u << LG;
    constexpr uint32_t SPS = 32u >> LG;
    constexpr uint32_t FULL = 0xffffffffu;

    const uint32_t lane = threadIdx.x & 31;
    // broadcast through a shuffle so the compiler knows the warp index (and everything derived
    // from it: staging addresses, barrier addresses) is warp-uniform
    const uint32_t warp = __shfl_sync(FULL, threadIdx.x >> 5, 0);
    const PassGeom &G = P.geom;
    const uint32_t n_stages = G.n_stages;
    const uint32_t stage_bytes = G.stage_bytes;
    const uint32_t n_batches = G.n_batches;  // whole launch
    constexpr uint32_t gpu = PAIR ? 2u : 1u;  // segments per unit
    auto seg = [&](uint32_t i) -> const RowSeg & {
        if constexpr (INLINE) return P.inline_segs[i]; else return P.segs[i];
    };
    auto prefix = [&](uint32_t u) -> uint32_t {
        if constexpr (INLINE) return P.inline_prefix[u]; else return P.unit_prefix[u];
    };

    const uint32_t smem_base = fm_smem_u32(smem_raw) + warp * G.warp_smem_bytes;
    const uint32_t bar_base = fm_smem_u32(bars + warp * kMaxStages);
    uint32_t *my_ring = batch_ring + warp * kBatchRing;
    fm_ring_init(bar_base, n_stages, lane);
    BatchScheduler sched(G.batch_counter, n_batches, lane);
    // unit of a launch-wide batch index: last u with prefix[u] <= gb (warp-uniform)
    auto unit_of = [&](uint32_t gb) -> uint32_t {
        uint32_t lo = 0, hi = P.n_units;
        while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if (prefix(mid) <= gb) lo = mid; else hi = mid;
        }
        return lo;
    };

    // ---- issue side: context of the (unit batch, group) whose steps are being issued
    uint32_t iss_ring = 0, iss_k = 0, iss_spb = 0, iss_stage = 0, iss_batch = 0;
    uint32_t iss_w16 = 0, iss_step_sites = 1, iss_g = 0, iss_unit = 0, iss_b = 0, iss_nst = 0;
    const uint4 *iss_allele = nullptr;
    bool iss_live = false;
    auto load_iss_seg = [&]() {
        const RowSeg &S = seg(iss_unit * gpu + iss_g);
        iss_w16 = S.g.wq * 16u;
        iss_step_sites = SPS * S.rounds;
        iss_spb = LPS / S.rounds;
        iss_nst = S.n_sites_total;
        iss_allele = S.g.allele;
    };
    auto issue = [&](uint32_t stage) {  // lane 0 only
        const uint32_t v0 = iss_b * 32 + iss_k * iss_step_sites;
        const uint32_t nsites = (v0 < iss_nst) ? min(iss_step_sites, iss_nst - v0) : 0u;
        fm_ring_fill(smem_base + stage * stage_bytes, reinterpret_cast<const uint8_t *>(iss_allele) + (size_t)v0 * iss_w16,
                     nsites * iss_w16, bar_base + 8u * stage);
    };
    auto issue_next = [&]() {
        if (iss_k == iss_spb) {
            if (iss_live && iss_g + 1 < gpu) {  // next group of the same unit batch
                ++iss_g;
                iss_k = 0;
                load_iss_seg();
            } else {
                if (iss_ring != 0 && iss_batch >= n_batches) return;  // scheduler drained
                iss_batch = sched.claim(lane);
                iss_k = 0;
                if (lane == 0) my_ring[iss_ring & (kBatchRing - 1)] = iss_batch;
                ++iss_ring;
                if (iss_batch >= n_batches) {
                    iss_spb = 0;
                    iss_live = false;
                    return;
                }
                iss_live = true;
                iss_unit = unit_of(iss_batch);
                iss_g = 0;
                load_iss_seg();
                iss_b = seg(iss_unit * gpu).b_lo + (iss_batch - prefix(iss_unit));
            }
        }
        if (lane == 0) issue(iss_stage);
        ++iss_k;
        iss_stage = (iss_stage + 1 == n_stages) ? 0 : iss_stage + 1;
    };
    for (uint32_t s = 0; s < n_stages; ++s) issue_next();
    __syncwarp();

    const uint32_t slot_in_round = lane >> LG;
    const uint32_t phase = lane & (LPS - 1);
    const uint32_t xfer_from = (lane & (SPS - 1)) << LG;  // source lane of the transpose
    const uint32_t xfer_round = lane >> (5 - LG);         // round whose sites land here

    uint32_t con_ring = 0, stage = 0, parity = 0;
    for (;;) {
        const uint32_t gb = my_ring[con_ring & (kBatchRing - 1)];
        ++con_ring;
        if (gb >= n_batches) break;
        const uint32_t unit = unit_of(gb);
        const uint32_t bl = gb - prefix(unit);  // batch inside the unit's range
        uint32_t alt_g0 = 0, cnt_g0 = 0, alt_g1 = 0, cnt_g1 = 0;
        uint32_t b = 0, u_vlo = 0, u_vhi = 0;
        for (uint32_t g = 0; g < gpu; ++g) {
            const RowSeg &S = seg(unit * gpu + g);
            const uint32_t w = S.g.wq, w16 = w * 16u, rounds = S.rounds;
            const uint32_t step_sites = SPS * rounds, spb = LPS / rounds;
            // columns phase, phase+LPS, ...: the first nit-1 are inside the row for every lane, only the last one
            // needs a bound check
            const uint32_t nit = (w + LPS - 1) / LPS;
            const uint32_t nfull = nit - 1, last_cols = w - nfull * LPS;
            const uint32_t nst = S.n_sites_total;
            b = S.b_lo + bl;
            u_vlo = S.v_lo;
            u_vhi = S.v_hi;
            uint32_t site_a = 0;  // alt count of this lane's batch site
            TailRegs tails;
            fm_tail_load(S.g, b * 32 + lane, nst, tails);
            for (uint32_t k = 0; k < spb; ++k) {
                fm_ring_wait(bar_base + 8u * stage, parity);
                const uint32_t sbase = smem_base + stage * stage_bytes;
                const uint32_t v0 = b * 32 + k * step_sites;
                auto round_body = [&](uint32_t r) {
                    const uint32_t site_local = r * SPS + slot_in_round;
                    const bool live = (v0 + site_local) < nst;
                    const uint32_t ra = sbase + site_local * w16;
                    uint32_t a = 0;
                    if (live) {
                        uint32_t p = ra + phase * 16u;
#pragma unroll 2
                        for (uint32_t j = 0; j < nfull; ++j) {
                            a += fm_popc4(fm_lds128(p));
                            p += LPS * 16u;
                        }
                        if (phase < last_cols) a += fm_popc4(fm_lds128(p));
                    }
#pragma unroll
                    for (uint32_t o = LPS >> 1; o > 0; o >>= 1) a += __shfl_xor_sync(FULL, a, o);
                    const uint32_t t = __shfl_sync(FULL, a, xfer_from);
                    if (xfer_round == k * rounds + r) site_a = t;
                };
                if (rounds == 1) {
                    round_body(0);
                } else {
                    for (uint32_t r = 0; r < rounds; r += 2) {  // rounds is a power of two
                        round_body(r);
                        round_body(r + 1);
                    }
                }
                __syncwarp();   // every lane is done reading this stage
                issue_next();   // refill it with the step n_stages ahead
                stage = (stage + 1 == n_stages) ? 0 : stage + 1;
                parity ^= (stage == 0);
            }
            // ---- group epilogue: lane i <-> site 32b + i (counts, summary partials, optional tracks)
            uint32_t alt = site_a, cnt;
            fm_tail_add(tails, alt, cnt);
            if (g == 0) {
                alt_g0 = alt;
                cnt_g0 = cnt;
            } else {
                alt_g1 = alt;
                cnt_g1 = cnt;
            }
            if (S.div.part_pi) fm_div_batch(S.div, b * 32 + lane, S.v_lo, S.v_hi, bl, lane, cnt, alt);
        }
        if constexpr (PAIR) {  // ---- Hudson components of the batch from both groups' counts
            const HudsonEpilogue &H = P.inline_hud[unit];
            const uint32_t v = b * 32 + lane;
            HudsonAcc acc{0.0, 0.0, 0.0, 0.0, 0.0, 0u, 0u, 0u};
            if (v >= u_vlo && v < u_vhi) fm_hudson_contrib(H, v, u_vlo, cnt_g0, alt_g0, cnt_g1, alt_g1, acc);
            const double r0 = fm_warp_sum(acc.num), r1 = fm_warp_sum(acc.den), r2 = fm_warp_sum(acc.dxy),
                         r3 = fm_warp_sum(acc.pi1), r4 = fm_warp_sum(acc.pi2);
            const uint32_t u01 = fm_warp_sum_u(acc.skipped | (acc.unc1 << 8) | (acc.unc2 << 16));
            if (lane == 0) {
                double *pd = H.part_d + (size_t)bl * 5;
                pd[0] = r0; pd[1] = r1; pd[2] = r2; pd[3] = r3; pd[4] = r4;
                uint32_t *pu = H.part_u + (size_t)bl * 3;
                pu[0] = u01 & 0xffu; pu[1] = (u01 >> 8) & 0xffu; pu[2] = u01 >> 16;
            }
        }
    }
}

// ------------------------------------------------------------------------------ plane pass, column chunks
// fm_k_plane_pass_chunked: one group whose rows are too wide for two sites per warp ring (biobank cohorts).  A
// pipeline step holds one column chunk of cq uint4 of one site's row (the whole row when it fits a stage: n_chunks
// == 1); every lane popcounts its 16-byte columns of the chunk and the warp sums the row when its last chunk is in.
struct ChunkParams {
    GroupPlanes g;
    PassGeom geom;
    DivEpilogue div;
};

__global__ void __launch_bounds__(kWarpsPerCta * 32, 1)
fm_k_plane_pass_chunked(const __grid_constant__ ChunkParams P) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bars[kWarpsPerCta * kMaxStages];
    __shared__ uint32_t batch_ring[kWarpsPerCta * kBatchRing];
    constexpr uint32_t FULL = 0xffffffffu;

    const uint32_t lane = threadIdx.x & 31;
    const uint32_t warp = __shfl_sync(FULL, threadIdx.x >> 5, 0);
    const PassGeom &G = P.geom;
    const uint32_t n_stages = G.n_stages;
    const uint32_t stage_bytes = G.stage_bytes;
    const uint32_t n_sites_total = G.n_sites_total;
    const uint32_t n_batches = G.n_batches;
    const uint32_t n_chunks = G.n_chunks;
    const uint32_t cq = G.cq;
    const uint32_t spb = 32u * n_chunks;  // steps per batch
    const uint32_t w = P.g.wq;

    const uint32_t smem_base = fm_smem_u32(smem_raw) + warp * G.warp_smem_bytes;
    const uint32_t bar_base = fm_smem_u32(bars + warp * kMaxStages);
    uint32_t *my_ring = batch_ring + warp * kBatchRing;
    fm_ring_init(bar_base, n_stages, lane);
    BatchScheduler sched(G.batch_counter, n_batches, lane);

    // issue the bulk copy of step k of local batch `bl` into `stage` (lane 0 only)
    auto issue = [&](uint32_t bl, uint32_t k, uint32_t stage) {
        const uint32_t v0 = (G.b_lo + bl) * 32 + k / n_chunks;
        const uint32_t c0 = (k % n_chunks) * cq;
        const uint32_t bytes = (v0 < n_sites_total && c0 < w) ? min(cq, w - c0) * 16u : 0u;
        fm_ring_fill(smem_base + stage * stage_bytes, P.g.allele + ((size_t)v0 * w + c0), bytes, bar_base + 8u * stage);
    };

    // issue cursor (uniform across the warp)
    uint32_t iss_ring = 0, iss_k = spb, iss_stage = 0, iss_batch = 0;
    auto issue_next = [&]() {
        if (iss_k == spb) {
            if (iss_ring != 0 && iss_batch >= n_batches) return;  // scheduler drained
            iss_batch = sched.claim(lane);
            iss_k = 0;
            if (lane == 0) my_ring[iss_ring & (kBatchRing - 1)] = iss_batch;
            ++iss_ring;
            if (iss_batch >= n_batches) {
                iss_k = spb;
                return;
            }
        }
        if (lane == 0) issue(iss_batch, iss_k, iss_stage);
        ++iss_k;
        iss_stage = (iss_stage + 1 == n_stages) ? 0 : iss_stage + 1;
    };
    for (uint32_t s = 0; s < n_stages; ++s) issue_next();
    __syncwarp();

    uint32_t site_a = 0, acc_a = 0;  // alt count of this lane's batch site, running row sum of this lane's columns
    uint32_t con_ring = 0, stage = 0, parity = 0;
    for (;;) {
        const uint32_t bl = my_ring[con_ring & (kBatchRing - 1)];
        ++con_ring;
        if (bl >= n_batches) break;
        const uint32_t b = G.b_lo + bl;
        TailRegs tails;
        fm_tail_load(P.g, b * 32 + lane, n_sites_total, tails);
        for (uint32_t k = 0; k < spb; ++k) {
            fm_ring_wait(bar_base + 8u * stage, parity);
            const uint32_t sbase = smem_base + stage * stage_bytes;
            const uint32_t site_in_batch = k / n_chunks;
            const uint32_t ck = k - site_in_batch * n_chunks;
            const uint32_t c0 = ck * cq;
            const bool live = (b * 32 + site_in_batch) < n_sites_total;
            const uint32_t cols16 = (c0 < w) ? min(cq, w - c0) * 16u : 0u;
            if (live) {
#pragma unroll 2
                for (uint32_t u = lane * 16u; u < cols16; u += 512u) acc_a += fm_popc4(fm_lds128(sbase + u));
            }
            if (ck == n_chunks - 1) {
                const uint32_t ta = fm_warp_sum_u(acc_a);
                if (lane == site_in_batch) site_a = ta;
                acc_a = 0;
            }
            __syncwarp();   // every lane is done reading this stage
            issue_next();   // refill it with the step n_stages ahead
            stage = (stage + 1 == n_stages) ? 0 : stage + 1;
            parity ^= (stage == 0);
        }
        // ---- batch epilogue: lane i <-> site 32b + i
        uint32_t alt = site_a, cnt;
        fm_tail_add(tails, alt, cnt);
        fm_div_batch(P.div, b * 32 + lane, G.v_lo, G.v_hi, bl, lane, cnt, alt);
    }
}

// ------------------------------------------------------------------------------ light kernels
// Same per-site functions evaluated from cached count arrays (8 B per site and group).
// One warp per batch of 32 sites so that the per-batch partials are bit-identical to the
// fused pass.
__global__ void __launch_bounds__(256)
fm_k_div_from_counts(const uint32_t *__restrict__ alt, const uint32_t *__restrict__ called,
                     DivEpilogue e, uint32_t v_lo, uint32_t v_hi, uint32_t b_lo, uint32_t n_batches) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t GW = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t bi = gw; bi < n_batches; bi += GW) {
        const uint32_t v = (b_lo + bi) * 32 + lane;
        const bool valid = v >= v_lo && v < v_hi;
        double pi_part = 0.0;
        uint32_t seg = 0, unc = 0;
        const uint32_t flags = e.site_flags ? e.site_flags[bi] : 0u;
        if (valid) fm_div_site(e, v, v_lo, called[v], alt[v], (flags >> lane) & 1u, pi_part, seg, unc);
        const double s_pi = fm_warp_sum(pi_part);
        const uint32_t s_seg = fm_warp_sum_u(seg), s_unc = fm_warp_sum_u(unc);
        if (lane == 0) {
            e.part_pi[bi] = s_pi;
            e.part_u[2 * bi] = s_seg;
            e.part_u[2 * bi + 1] = s_unc;
        }
    }
}

__global__ void __launch_bounds__(256)
fm_k_hudson_from_counts(const uint32_t *__restrict__ alt1, const uint32_t *__restrict__ n1,
                        const uint32_t *__restrict__ alt2, const uint32_t *__restrict__ n2,
                        HudsonEpilogue e, uint32_t v_lo, uint32_t v_hi, uint32_t b_lo,
                        uint32_t n_batches) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t GW = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t bi = gw; bi < n_batches; bi += GW) {
        const uint32_t v = (b_lo + bi) * 32 + lane;
        const bool valid = v >= v_lo && v < v_hi;
        HudsonAcc acc{0.0, 0.0, 0.0, 0.0, 0.0, 0u, 0u, 0u};
        if (valid) fm_hudson_contrib(e, v, v_lo, n1[v], alt1[v], n2[v], alt2[v], acc);
        const double r0 = fm_warp_sum(acc.num), r1 = fm_warp_sum(acc.den), r2 = fm_warp_sum(acc.dxy),
                     r3 = fm_warp_sum(acc.pi1), r4 = fm_warp_sum(acc.pi2);
        const uint32_t u0 = fm_warp_sum_u(acc.skipped), u1 = fm_warp_sum_u(acc.unc1),
                       u2 = fm_warp_sum_u(acc.unc2);
        if (lane == 0) {
            double *pd = e.part_d + (size_t)bi * 5;
            pd[0] = r0; pd[1] = r1; pd[2] = r2; pd[3] = r3; pd[4] = r4;
            uint32_t *pu = e.part_u + (size_t)bi * 3;
            pu[0] = u0; pu[1] = u1; pu[2] = u2;
        }
    }
}

// Second-level reduction: super-batch s folds batches [s*256, s*256+256) of the GLOBAL batch
// grid with a fixed shape -- lane l sums its 8 consecutive batches in order, then a butterfly
// over lanes -- for `nd` double columns and `nu` u32 columns.  One warp per super-batch.
__global__ void __launch_bounds__(128)
fm_k_reduce_partials(const double *__restrict__ pd, int nd, const uint32_t *__restrict__ pu, int nu,
                     uint32_t b_lo, uint32_t n_batches, uint32_t s_lo, uint32_t n_super,
                     double *__restrict__ out_d, uint64_t *__restrict__ out_u) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (s >= n_super) return;
    constexpr uint32_t per_lane = kSuperBatches / 32;
    const uint64_t g0 = (uint64_t)(s_lo + s) * kSuperBatches + (uint64_t)lane * per_lane;
    const uint64_t b_hi = (uint64_t)b_lo + n_batches;
    for (int col = 0; col < nd; ++col) {
        double acc = 0.0;
#pragma unroll
        for (uint32_t i = 0; i < per_lane; ++i) {
            const uint64_t b = g0 + i;
            if (b >= b_lo && b < b_hi) acc += pd[(b - b_lo) * nd + col];
        }
        acc = fm_warp_sum(acc);
        if (lane == 0) out_d[(size_t)s * nd + col] = acc;
    }
    for (int col = 0; col < nu; ++col) {
        uint32_t acc = 0;
#pragma unroll
        for (uint32_t i = 0; i < per_lane; ++i) {
            const uint64_t b = g0 + i;
            if (b >= b_lo && b < b_hi) acc += pu[(b - b_lo) * nu + col];
        }
        acc = fm_warp_sum_u(acc);
        if (lane == 0) out_u[(size_t)s * nu + col] = acc;
    }
}

// The same fold for many units at once (fm_k_plane_pass_seq launches): entry e = (first partial of the unit in
// the shared partial arrays, the unit's first global batch, its batch count, the global super-batch index); one
// warp per entry, the association of fm_k_reduce_partials -- a unit reduced here gives the bits it would give alone.
__global__ void __launch_bounds__(128)
fm_k_reduce_partials_tab(const double *__restrict__ pd, int nd, const uint32_t *__restrict__ pu, int nu,
                         const uint4 *__restrict__ ents, uint32_t n_ent, double *__restrict__ out_d,
                         uint64_t *__restrict__ out_u) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (e >= n_ent) return;
    const uint4 E = ents[e];
    constexpr uint32_t per_lane = kSuperBatches / 32;
    const uint64_t g0 = (uint64_t)E.w * kSuperBatches + (uint64_t)lane * per_lane;
    const uint64_t b_lo = E.y, b_hi = (uint64_t)E.y + E.z;
    for (int col = 0; col < nd; ++col) {
        double acc = 0.0;
#pragma unroll
        for (uint32_t i = 0; i < per_lane; ++i) {
            const uint64_t b = g0 + i;
            if (b >= b_lo && b < b_hi) acc += pd[((size_t)E.x + (b - b_lo)) * nd + col];
        }
        acc = fm_warp_sum(acc);
        if (lane == 0) out_d[(size_t)e * nd + col] = acc;
    }
    for (int col = 0; col < nu; ++col) {
        uint32_t acc = 0;
#pragma unroll
        for (uint32_t i = 0; i < per_lane; ++i) {
            const uint64_t b = g0 + i;
            if (b >= b_lo && b < b_hi) acc += pu[((size_t)E.x + (b - b_lo)) * nu + col];
        }
        acc = fm_warp_sum_u(acc);
        if (lane == 0) out_u[(size_t)e * nu + col] = acc;
    }
}

// ------------------------------------------------------------------------------ K5 windows
// One warp per window [lo, hi) of site indices: lanes stride the window, then a fixed-shape
// butterfly.  Values are evaluated from cached counts.
__global__ void __launch_bounds__(256)
fm_k_window_div(const uint32_t *__restrict__ alt, const uint32_t *__restrict__ called,
                const uint32_t *__restrict__ win_lo, const uint32_t *__restrict__ win_hi,
                uint32_t n_windows, int pi_form, uint64_t *__restrict__ seg_out,
                double *__restrict__ pi_out, uint64_t *__restrict__ unc_out) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t GW = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t w = gw; w < n_windows; w += GW) {
        double pi = 0.0;
        uint32_t seg = 0, unc = 0;
        for (uint32_t v = win_lo[w] + lane; v < win_hi[w]; v += 32) {
            const uint32_t n = called[v], a = alt[v];
            seg += (n >= 2 && a > 0 && a < n);
            unc += (n < 2);
            double val;
            if (fm_pi_form(pi_form, n, a, val)) pi += val;
        }
        pi = fm_warp_sum(pi);
        seg = fm_warp_sum_u(seg);
        unc = fm_warp_sum_u(unc);
        if (lane == 0) {
            seg_out[w] = seg;
            pi_out[w] = pi;
            unc_out[w] = unc;
        }
    }
}

__global__ void __launch_bounds__(256)
fm_k_window_hudson(const uint32_t *__restrict__ alt1, const uint32_t *__restrict__ n1,
                   const uint32_t *__restrict__ alt2, const uint32_t *__restrict__ n2,
                   const uint32_t *__restrict__ win_lo, const uint32_t *__restrict__ win_hi,
                   uint32_t n_windows, double *__restrict__ out_d /*[n][5]*/,
                   uint64_t *__restrict__ out_skipped) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t GW = (gridDim.x * blockDim.x) >> 5;
    HudsonEpilogue e{};
    e.variant = -1;
    for (uint32_t w = gw; w < n_windows; w += GW) {
        double s[5] = {0, 0, 0, 0, 0};
        uint32_t skipped = 0;
        for (uint32_t v = win_lo[w] + lane; v < win_hi[w]; v += 32) {
            HudsonAcc acc;
            fm_hudson_contrib(e, v, 0, n1[v], alt1[v], n2[v], alt2[v], acc);
            s[0] += acc.num; s[1] += acc.den; s[2] += acc.dxy; s[3] += acc.pi1; s[4] += acc.pi2;
            skipped += acc.skipped;
        }
#pragma unroll
        for (int i = 0; i < 5; ++i) s[i] = fm_warp_sum(s[i]);
        skipped = fm_warp_sum_u(skipped);
        if (lane == 0) {
            for (int i = 0; i < 5; ++i) out_d[(size_t)w * 5 + i] = s[i];
            out_skipped[w] = skipped;
        }
    }
}

}  // namespace fm
