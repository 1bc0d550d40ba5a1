// fm_ld.cuh -- windowed linkage disequilibrium (r^2 and D') between kept sites of a haplotype set (DESIGN.md §0
// row f9, §3 and §4 "Haplotype LD"; definition in include/ferromic_gpu.h, fm_haplotype_ld).
//
// The pairwise-differences bit product with the axes swapped: kept sites are the 64-wide tile axis and haplotype
// words the K axis, so PwLayout describes the planes unchanged ("sample" = kept site, "site word" = word of 32
// haplotypes).  Plane 0 holds the alt bits (called, raw allele 1) and plane 1, present only when some kept site has
// a missing cell among the n haplotypes, the called bits.  A pair (i, j) of kept sites then needs
//   ab = popc(a_i & a_j)                                                           (always)
//   c = popc(c_i & c_j),  a = popc(a_i & c_j),  b = popc(c_i & a_j)                 (called plane only)
// and without the called plane c = n and a, b are the sites' alt counts.  All counts are exact integers; the FP64
// epilogue follows the header's operation order, so the outputs equal the numpy restatement bit for bit.
#pragma once
#include "fm_device.cuh"
#include "fm_haplotypes.cuh"  // HapCells
#include "fm_pairwise.cuh"    // PwLayout, PwRing, kPwBlk, kPwKT

namespace fm {

// 16 x 16 consumer threads, each owning 4 x 4 pairs of a 64 x 64 tile.  With the called plane a pair carries four
// counters; the 4 x 8 micro-tile of fm_k_pairwise_counts would hold 128 of them per thread.  4 x 4 holds 64, the
// count registers of the pairwise kernel, and compiles without spills (profiles/r08_ptxas_ld_kernels.txt).
constexpr uint32_t kLdConsumerWarps = 8;
constexpr uint32_t kLdNanBits = 0x7fc00000u;  // the quiet NaN numpy writes for float32('nan')

// Per kept site j (matrix row kept[j]): its alt count and position.
__global__ void __launch_bounds__(256)
fm_k_ld_sites(const uint32_t *__restrict__ kept, uint32_t M, uint32_t v_lo, const uint32_t *__restrict__ alt,
              const int64_t *__restrict__ pos, uint32_t *__restrict__ kalt, int64_t *__restrict__ kpos) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= M) return;
    const uint32_t v = kept[j];
    kalt[j] = alt[v - v_lo];
    kpos[j] = pos[v];
}

// Kept sites x selected haplotypes -> site-major planes of PwLayout{ceil(M / 64), planes}.  One warp per (32 kept
// sites, haplotype word): lane = haplotype, one ballot per site turns the 32 cells into the site's word, which lane
// t keeps for site t; the 32 site words are then one coalesced store per plane.  Padded sites and haplotypes stay
// zero (the planes are cleared before the launch).
__global__ void __launch_bounds__(256)
fm_k_ld_planes(HapCells cells, const uint32_t *__restrict__ off, uint32_t n, const uint32_t *__restrict__ kept,
               uint32_t M, uint32_t n_words, PwLayout L, uint32_t *__restrict__ planes) {
    constexpr uint32_t FULL = 0xffffffffu;
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t n_tasks = (uint64_t)((M + 31) / 32) * n_words;
    const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t task = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; task < n_tasks; task += n_warps) {
        const uint32_t g = (uint32_t)(task / n_words), w = (uint32_t)(task % n_words);
        const uint32_t h = w * 32u + lane, n_t = min(32u, M - g * 32u);
        const uint32_t col = h < n ? __ldg(off + h) : 0u;
        uint32_t my_a = 0, my_c = 0;
        for (uint32_t t = 0; t < n_t; ++t) {
            bool called = false, alt = false, other;
            if (h < n) cells.read(__ldg(kept + g * 32u + t), col, called, alt, other);
            const uint32_t ba = __ballot_sync(FULL, alt), bc = __ballot_sync(FULL, called);
            if (lane == t) {
                my_a = ba;
                my_c = bc;
            }
        }
        if (lane >= n_t) continue;
        const uint32_t s = g * 32u + lane;
        planes[L.word(w, s, 0)] = my_a;
        if (L.planes > 1) planes[L.word(w, s, 1)] = my_c;
    }
}

// r^2 and D' of one pair from its exact counts, in the operation order of include/ferromic_gpu.h.
__device__ __forceinline__ void fm_ld_stats(int64_t c, int64_t a, int64_t b, int64_t ab, float &r2, float &dp) {
    r2 = dp = __uint_as_float(kLdNanBits);
    if (c == 0 || a == 0 || a == c || b == 0 || b == c) return;
    const int64_t dn = c * ab - a * b;
    const double x = (double)dn;
    r2 = __double2float_rn((x * x) / ((double)(a * (c - a)) * (double)(b * (c - b))));
    if (dn > 0) dp = __double2float_rn(x / (double)min(a * (c - b), (c - a) * b));
    else if (dn < 0) dp = __double2float_rn(x / (double)min(a * b, (c - a) * (c - b)));
    else dp = 0.0f;
}

// Banded upper-triangle bit product over one slab of row blocks [rb0, rb0 + gridDim.x / tpr).  CTA t is tile
// (bi, bj) = (rb0 + t / tpr, bi + t % tpr); tpr = ceil(window / 64) + 1 tiles per row block cover every (i, d) with
// 1 <= d <= window exactly once.  Warp kLdConsumerWarps is the producer of the tile's PwRing; a tile past the last
// site block has no chunks and only writes its NaN cells.  Consumer thread (ti, tj) owns the sites
// i = 64 bi + 4 ti + {0..3} and j = 64 bj + tj + 16 {0..3}, so that for each of its pairs the 16 threads of a row
// write 16 consecutive floats.  out_r2 / out_dp hold the slab's rows: [(i - 64 rb0) * window + d - 1].
template <bool HC>
__global__ void __launch_bounds__((kLdConsumerWarps + 1) * 32)
fm_k_ld_band(const uint32_t *__restrict__ planes, PwLayout L, uint32_t n_chunks, uint32_t n, uint32_t M,
             uint32_t window, int64_t max_distance, uint32_t rb0, uint32_t tpr, const uint32_t *__restrict__ kalt,
             const int64_t *__restrict__ kpos, float *__restrict__ out_r2, float *__restrict__ out_dp) {
    extern __shared__ __align__(128) uint8_t ld_smem[];
    const PwRing<kLdConsumerWarps> ring(ld_smem, L);
    const uint32_t bi = rb0 + blockIdx.x / tpr, bj = bi + blockIdx.x % tpr;
    const bool diag = bi == bj;
    const uint32_t chunks = bj < L.n_blk ? n_chunks : 0u;
    ring.init();
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == kLdConsumerWarps) {
        if (lane == 0) ring.produce(planes, L, chunks, bi, bj);
        return;
    }

    // ---------------------------------------------------------------------- consumers
    const uint32_t ti = threadIdx.x >> 4, tj = threadIdx.x & 15;
    uint32_t acc_ab[4][4], acc_c[4][4], acc_a[4][4], acc_b[4][4];
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) acc_ab[x][y] = acc_c[x][y] = acc_a[x][y] = acc_b[x][y] = 0;
    for (uint32_t c = 0; c < chunks; ++c) {
        uint32_t si, sj;
        ring.acquire(c, diag, si, sj);
        si += ti * 16u;
        sj += tj * 4u;
#pragma unroll 2
        for (uint32_t k = 0; k < kPwKT; ++k) {
            const uint32_t off_a = k * kPwBlk * 4u, off_c = (kPwKT + k) * kPwBlk * 4u;
            const uint4 ua = fm_lds128(si + off_a);
            const uint32_t ai[4] = {ua.x, ua.y, ua.z, ua.w};
            uint32_t aj[4];
#pragma unroll
            for (int y = 0; y < 4; ++y) aj[y] = fm_lds32(sj + off_a + 64u * y);
            if (HC) {
                const uint4 uc = fm_lds128(si + off_c);
                const uint32_t ci[4] = {uc.x, uc.y, uc.z, uc.w};
                uint32_t cj[4];
#pragma unroll
                for (int y = 0; y < 4; ++y) cj[y] = fm_lds32(sj + off_c + 64u * y);
#pragma unroll
                for (int x = 0; x < 4; ++x)
#pragma unroll
                    for (int y = 0; y < 4; ++y) {
                        acc_ab[x][y] += __popc(ai[x] & aj[y]);
                        acc_c[x][y] += __popc(ci[x] & cj[y]);
                        acc_a[x][y] += __popc(ai[x] & cj[y]);
                        acc_b[x][y] += __popc(ci[x] & aj[y]);
                    }
            } else {
#pragma unroll
                for (int x = 0; x < 4; ++x)
#pragma unroll
                    for (int y = 0; y < 4; ++y) acc_ab[x][y] += __popc(ai[x] & aj[y]);
            }
        }
        ring.release(c, lane);
    }

    // ---------------------------------------------------------------------- epilogue
#pragma unroll
    for (int x = 0; x < 4; ++x) {
        const uint32_t gi = bi * kPwBlk + ti * 4u + x;
        if (gi >= M) continue;
        const uint32_t alt_i = HC ? 0u : kalt[gi];
        const size_t row = (size_t)(gi - rb0 * kPwBlk) * window;
#pragma unroll
        for (int y = 0; y < 4; ++y) {
            const uint32_t gj = bj * kPwBlk + tj + 16u * y;
            if (gj <= gi || gj - gi > window) continue;
            float r2 = __uint_as_float(kLdNanBits), dp = r2;
            if (gj < M && (max_distance < 0 || kpos[gj] - kpos[gi] <= max_distance)) {
                if (HC) fm_ld_stats(acc_c[x][y], acc_a[x][y], acc_b[x][y], acc_ab[x][y], r2, dp);
                else fm_ld_stats(n, alt_i, kalt[gj], acc_ab[x][y], r2, dp);
            }
            out_r2[row + (gj - gi - 1)] = r2;
            if (out_dp) out_dp[row + (gj - gi - 1)] = dp;
        }
    }
}

}  // namespace fm
