// fm_pairwise.cuh -- per-sample-pair genotype difference counts (calculate_pairwise_differences,
// stats.rs:4106-4231; definition and parity status in DESIGN.md §3 and §4 "Pairwise differences").
//
// A sample's genotype at a site is the run of its leading called cells (side 0, side 1); it is None when cell 0 is
// missing.  Per sample and site the transpose builds bit planes over sites:
//   pc_p      cells 0..p are all called                         (only when the matrix carries missingness)
//   a_{p,k}   bit k of the allele rank of cell p, masked by pc_p
// and a pair (i, j) compares
//   comparable = pc_0[i] & pc_0[j]
//   differ     = comparable & (OR_{p>=1} (pc_p[i] ^ pc_p[j]) | OR_{p,k} (a_{p,k}[i] ^ a_{p,k}[j]))
// Plane 0 is pc_0 when the matrix has missingness (the "comparability plane"); every other plane is an "identity
// plane" that only enters through XOR.  Without missingness every genotype is the full vector, comparable = V and
// only the allele planes exist.
//
// Layout (K-tiled, sample-major inside a tile): for K-chunk c (kPwKT site words), sample block b (kPwBlk samples),
// plane p, word k of the chunk and sample sl of the block, the word sits at
//   ((((c * n_blk + b) * planes + p) * kPwKT + k) * kPwBlk + sl
// so the chunk of one sample block is ONE contiguous run of planes * kPwKT * kPwBlk words -- a single 1-D bulk copy
// -- and inside it the 64 samples of a (plane, word) are consecutive, which lets a thread fetch 4 samples with one
// 128-bit shared-memory load without bank conflicts.  Padded samples and words are zero in every plane, so they add
// nothing to either count.
#pragma once
#include "fm_device.cuh"
#include "fm_wc.cuh"  // fm_mbar_wait / fm_mbar_arrive on shared-memory addresses

namespace fm {

constexpr uint32_t kPwBlk = 64;          // samples per tile side
constexpr uint32_t kPwKT = 8;            // site words (256 sites) per K-chunk
constexpr uint32_t kPwStages = 4;        // shared-memory ring depth
constexpr uint32_t kPwConsumerWarps = 4; // 128 threads x (4 x 8) pairs = one 64 x 64 tile

struct PwLayout {
    uint32_t n_blk;   // sample blocks
    uint32_t planes;  // planes per sample
    __host__ __device__ __forceinline__ size_t word(uint32_t w, uint32_t s, uint32_t p) const {
        const uint32_t c = w / kPwKT, k = w % kPwKT, b = s / kPwBlk, sl = s % kPwBlk;
        return ((((size_t)c * n_blk + b) * planes + p) * kPwKT + k) * kPwBlk + sl;
    }
    __host__ __device__ __forceinline__ uint32_t tile_words() const { return planes * kPwKT * kPwBlk; }
};

// ---------------------------------------------------------------------------------------------- transposes
// Resident u8 matrix (bitmap, in-band or no missingness; rank LUT for allele values above 15).  One warp per
// (site word, 32 consecutive samples), lane = sample: each of the 32 site rows is read as one coalesced run of the
// warp's cells and the lane shifts its bits into its own plane words.
template <int PL, int NB>
__global__ void __launch_bounds__(256)
fm_k_sample_planes(const uint8_t *__restrict__ data, const uint64_t *__restrict__ missing, uint32_t miss_mode,
                   const uint8_t *__restrict__ lut, uint32_t V, uint32_t n_samples, uint64_t stride, uint32_t n_words,
                   PwLayout L, uint32_t *__restrict__ planes) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t groups = (n_samples + 31) / 32;
    const uint64_t n_tasks = (uint64_t)n_words * groups;
    const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t task = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; task < n_tasks; task += n_warps) {
        const uint32_t w = (uint32_t)(task / groups), s = (uint32_t)(task % groups) * 32 + lane;
        if (s >= n_samples) continue;
        uint32_t pc[PL], al[PL][NB];
#pragma unroll
        for (int p = 0; p < PL; ++p) {
            pc[p] = 0;
#pragma unroll
            for (int k = 0; k < NB; ++k) al[p][k] = 0;
        }
        const uint32_t n_t = min(32u, V - w * 32u);
        for (uint32_t t = 0; t < n_t; ++t) {
            const uint64_t e0 = ((uint64_t)w * 32 + t) * stride + (uint64_t)s * PL;
            bool run = true;
#pragma unroll
            for (int p = 0; p < PL; ++p) {
                const uint8_t x = __ldg(data + e0 + p);
                bool called = true;
                if (miss_mode == 1) called = ((__ldg(missing + ((e0 + p) >> 6)) >> ((e0 + p) & 63)) & 1ull) == 0;
                else if (miss_mode == 2) called = x < 0x80;
                run = run && called;
                if (run) {
                    const uint32_t r = lut ? __ldg(lut + x) : x;
                    pc[p] |= 1u << t;
#pragma unroll
                    for (int k = 0; k < NB; ++k) al[p][k] |= ((r >> k) & 1u) << t;
                }
            }
        }
        uint32_t q = 0;
        if (miss_mode) {
#pragma unroll
            for (int p = 0; p < PL; ++p) planes[L.word(w, s, q++)] = pc[p];
        }
#pragma unroll
        for (int p = 0; p < PL; ++p)
#pragma unroll
            for (int k = 0; k < NB; ++k) planes[L.word(w, s, q++)] = al[p][k];
    }
}

// Resident packed rows (biallelic; allele bit = called and non-zero).  One warp per (site word, cell word): lane l
// holds the row word of site 32 w + l, and one ballot per cell turns the 32 x 32 bit block around so that lane c
// ends up with the site word of cell 32 q + c (a warp-ballot transpose).  Side-1 lanes hand their words to the
// side-0 lane of the same sample.
template <int PL>
__global__ void __launch_bounds__(256)
fm_k_sample_planes_packed(const uint32_t *__restrict__ abits, const uint32_t *__restrict__ cbits, uint32_t rw,
                          uint32_t V, uint32_t n_samples, uint32_t n_words, uint32_t n_cell_words, PwLayout L,
                          uint32_t *__restrict__ planes) {
    constexpr uint32_t FULL = 0xffffffffu;
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t n_tasks = (uint64_t)n_words * n_cell_words;
    const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t task = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; task < n_tasks; task += n_warps) {
        const uint32_t w = (uint32_t)(task / n_cell_words), q = (uint32_t)(task % n_cell_words);
        const uint32_t v = w * 32u + lane;
        uint32_t a = 0, c = 0;
        if (v < V) {
            a = __ldg(abits + (size_t)v * rw + q);
            if (cbits) c = __ldg(cbits + (size_t)v * rw + q);
        }
        uint32_t my_a = 0, my_c = 0;
#pragma unroll
        for (uint32_t b = 0; b < 32; ++b) {
            const uint32_t ba = __ballot_sync(FULL, (a >> b) & 1u);
            const uint32_t bc = cbits ? __ballot_sync(FULL, (c >> b) & 1u) : 0u;
            if (lane == b) {
                my_a = ba;
                my_c = bc;
            }
        }
        uint32_t a1 = 0, c1 = 0;
        if (PL == 2) {
            a1 = __shfl_down_sync(FULL, my_a, 1);
            c1 = __shfl_down_sync(FULL, my_c, 1);
        }
        const uint32_t s = (q * 32u + lane) / PL;
        if ((lane % PL) != 0 || s >= n_samples) continue;
        uint32_t p = 0;
        if (cbits) {
            const uint32_t pc1 = my_c & c1;
            planes[L.word(w, s, p++)] = my_c;
            if (PL == 2) planes[L.word(w, s, p++)] = pc1;
            planes[L.word(w, s, p++)] = my_a & my_c;
            if (PL == 2) planes[L.word(w, s, p++)] = a1 & pc1;
        } else {
            planes[L.word(w, s, p++)] = my_a;
            if (PL == 2) planes[L.word(w, s, p++)] = a1;
        }
    }
}

// ---------------------------------------------------------------------------------------------- pair counts
// Upper-triangle tiled bit-GEMM.  One CTA per 64 x 64 tile (bi <= bj) of sample pairs; warp kPwConsumerWarps is the
// producer: its lane 0 streams the K-chunks of both sample blocks (one block on diagonal tiles) into a kPwStages ring
// with 1-D bulk copies that complete on the stage's `full` mbarrier; the consumer warps release a stage through its
// `empty` mbarrier.  Consumer thread (ti, tj) owns samples i = 4 ti + {0..3} and j = 4 tj + {0..3}, 32 + 4 tj +
// {0..3} of the tile and keeps their 32 counts in registers.  Per site word and pair the cost is one LOP3 per
// identity plane, and on top 2 LOP3 + 2 POPC with a comparability plane (1 POPC without).
template <bool HC>
__global__ void __launch_bounds__((kPwConsumerWarps + 1) * 32)
fm_k_pairwise_counts(const uint32_t *__restrict__ planes, PwLayout L, uint32_t n_chunks, uint32_t n_samples,
                     uint32_t n_sites, uint32_t *__restrict__ diff_out, uint32_t *__restrict__ comp_out) {
    extern __shared__ __align__(128) uint8_t pw_smem[];
    const uint32_t tile_w = L.tile_words();
    const uint32_t stage_bytes = 2u * tile_w * 4u;
    uint64_t *bars = reinterpret_cast<uint64_t *>(pw_smem + (size_t)kPwStages * stage_bytes);
    const uint32_t bar_full = fm_smem_u32(bars), bar_empty = bar_full + 8u * kPwStages;
    // blockIdx.x -> (bi, bj), row-major over the upper triangle of the block grid
    uint32_t bi = 0, rem = blockIdx.x;
    while (rem >= L.n_blk - bi) {
        rem -= L.n_blk - bi;
        ++bi;
    }
    const uint32_t bj = bi + rem;
    const bool diag = bi == bj;
    if (threadIdx.x == 0) {
        for (uint32_t s = 0; s < kPwStages; ++s) {
            fm_mbar_init(bars + s, 1);
            fm_mbar_init(bars + kPwStages + s, kPwConsumerWarps);
        }
        fm_fence_mbar_init();
    }
    __syncthreads();
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (warp == kPwConsumerWarps) {
        // ------------------------------------------------------------------ producer
        if (lane == 0) {
            const uint32_t bytes = tile_w * 4u;
            for (uint32_t c = 0; c < n_chunks; ++c) {
                const uint32_t st = c % kPwStages;
                if (c >= kPwStages) fm_mbar_wait(bar_empty + 8u * st, ((c / kPwStages) - 1u) & 1u);
                uint8_t *dst = pw_smem + (size_t)st * stage_bytes;
                fm_mbar_expect_tx(bars + st, diag ? bytes : 2u * bytes);
                fm_bulk_g2s(dst, planes + ((size_t)c * L.n_blk + bi) * tile_w, bytes, bars + st);
                if (!diag) fm_bulk_g2s(dst + bytes, planes + ((size_t)c * L.n_blk + bj) * tile_w, bytes, bars + st);
            }
        }
        return;
    }

    // ---------------------------------------------------------------------- consumers
    const uint32_t ti = threadIdx.x >> 3, tj = threadIdx.x & 7;
    const uint32_t P = L.planes;
    uint32_t acc_d[4][8], acc_c[4][8];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 8; ++b) acc_d[a][b] = acc_c[a][b] = 0;
    for (uint32_t c = 0; c < n_chunks; ++c) {
        const uint32_t st = c % kPwStages;
        fm_mbar_wait(bar_full + 8u * st, (c / kPwStages) & 1u);
        const uint32_t si = fm_smem_u32(pw_smem + (size_t)st * stage_bytes) + ti * 16u;
        const uint32_t sj = fm_smem_u32(pw_smem + (size_t)st * stage_bytes + (diag ? 0u : tile_w * 4u)) + tj * 16u;
#pragma unroll 1
        for (uint32_t k = 0; k < kPwKT; ++k) {
            uint32_t x[4][8];
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int b = 0; b < 8; ++b) x[a][b] = 0;
            for (uint32_t p = HC ? 1u : 0u; p < P; ++p) {
                const uint32_t off = (p * kPwKT + k) * kPwBlk * 4u;
                const uint4 ui = fm_lds128(si + off), u0 = fm_lds128(sj + off), u1 = fm_lds128(sj + off + 128u);
                const uint32_t va[4] = {ui.x, ui.y, ui.z, ui.w};
                const uint32_t vb[8] = {u0.x, u0.y, u0.z, u0.w, u1.x, u1.y, u1.z, u1.w};
#pragma unroll
                for (int a = 0; a < 4; ++a)
#pragma unroll
                    for (int b = 0; b < 8; ++b) x[a][b] |= va[a] ^ vb[b];
            }
            if (HC) {
                const uint32_t off = k * kPwBlk * 4u;
                const uint4 ci = fm_lds128(si + off), c0 = fm_lds128(sj + off), c1 = fm_lds128(sj + off + 128u);
                const uint32_t va[4] = {ci.x, ci.y, ci.z, ci.w};
                const uint32_t vb[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
#pragma unroll
                for (int a = 0; a < 4; ++a)
#pragma unroll
                    for (int b = 0; b < 8; ++b) {
                        acc_d[a][b] += __popc(va[a] & vb[b] & x[a][b]);
                        acc_c[a][b] += __popc(va[a] & vb[b]);
                    }
            } else {
#pragma unroll
                for (int a = 0; a < 4; ++a)
#pragma unroll
                    for (int b = 0; b < 8; ++b) acc_d[a][b] += __popc(x[a][b]);
            }
        }
        __syncwarp();
        if (lane == 0) fm_mbar_arrive(bar_empty + 8u * st);
    }
    // condensed (pdist) order: pair (i, j), i < j, sits at i (2 n - i - 1) / 2 + j - i - 1
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const uint32_t gi = bi * kPwBlk + ti * 4u + a;
#pragma unroll
        for (int b = 0; b < 8; ++b) {
            const uint32_t gj = bj * kPwBlk + (b < 4 ? tj * 4u + b : 32u + tj * 4u + (b - 4));
            if (gi < gj && gj < n_samples) {
                const uint64_t idx = (uint64_t)gi * (2ull * n_samples - gi - 1) / 2 + (gj - gi - 1);
                diff_out[idx] = acc_d[a][b];
                if (comp_out) comp_out[idx] = HC ? acc_c[a][b] : n_sites;
            }
        }
    }
}

// condensed pair index -> (i, j)
__device__ __forceinline__ void fm_pw_pair(uint64_t idx, uint32_t n, uint32_t &i, uint32_t &j) {
    const double b = 2.0 * n - 1.0;
    int64_t r = (int64_t)floor((b - sqrt(fmax(b * b - 8.0 * (double)idx, 0.0))) * 0.5);
    r = r < 0 ? 0 : (r > (int64_t)n - 2 ? (int64_t)n - 2 : r);
    auto start = [n](int64_t row) { return (uint64_t)row * (2ull * n - (uint64_t)row - 1) / 2; };
    while (r > 0 && start(r) > idx) --r;
    while (r + 1 < (int64_t)n - 1 && start(r + 1) <= idx) ++r;
    i = (uint32_t)r;
    j = (uint32_t)(idx - start(r) + (uint64_t)r + 1);
}

// One warp per pair: re-walks the pair's site words (lane = word) and writes the positions of the differing sites in
// site order at out[pair_start[pair] ..] (ballot-free: popc + warp prefix sum per 32 words).
template <bool HC>
__global__ void __launch_bounds__(256)
fm_k_pairwise_positions(const uint32_t *__restrict__ planes, PwLayout L, uint32_t n_words, uint32_t n_samples,
                        uint64_t n_pairs, const uint64_t *__restrict__ pair_start, const int64_t *__restrict__ pos,
                        int64_t *__restrict__ out) {
    constexpr uint32_t FULL = 0xffffffffu;
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t pr = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (pr >= n_pairs) return;
    uint32_t i, j;
    fm_pw_pair(pr, n_samples, i, j);
    uint64_t o = pair_start[pr];
    for (uint32_t w0 = 0; w0 < n_words; w0 += 32) {
        const uint32_t w = w0 + lane;
        uint32_t d = 0;
        if (w < n_words) {
            uint32_t x = 0;
            for (uint32_t p = HC ? 1u : 0u; p < L.planes; ++p) x |= __ldg(planes + L.word(w, i, p)) ^ __ldg(planes + L.word(w, j, p));
            d = HC ? (__ldg(planes + L.word(w, i, 0)) & __ldg(planes + L.word(w, j, 0)) & x) : x;
        }
        const uint32_t cnt = __popc(d);
        uint32_t inc = cnt;
#pragma unroll
        for (uint32_t off = 1; off < 32; off <<= 1) {
            const uint32_t t = __shfl_up_sync(FULL, inc, off);
            if (lane >= off) inc += t;
        }
        uint64_t q = o + inc - cnt;
        while (d) {
            const uint32_t b = __ffs(d) - 1;
            out[q++] = pos[(size_t)w * 32 + b];
            d &= d - 1;
        }
        o += __shfl_sync(FULL, inc, 31);
    }
}

}  // namespace fm
