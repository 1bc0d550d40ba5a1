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

// FP64 r^2 of one pair with 0 < a < c and 0 < b < c, in the operation order of include/ferromic_gpu.h.
__device__ __forceinline__ double fm_ld_r2(int64_t c, int64_t a, int64_t b, int64_t dn) {
    const double x = (double)dn;
    return (x * x) / ((double)(a * (c - a)) * (double)(b * (c - b)));
}

// r^2 and D' of one pair from its exact counts, in the operation order of include/ferromic_gpu.h.
__device__ __forceinline__ void fm_ld_stats(int64_t c, int64_t a, int64_t b, int64_t ab, float &r2, float &dp) {
    r2 = dp = __uint_as_float(kLdNanBits);
    if (c == 0 || a == 0 || a == c || b == 0 || b == c) return;
    const int64_t dn = c * ab - a * b;
    const double x = (double)dn;
    r2 = __double2float_rn(fm_ld_r2(c, a, b, dn));
    if (dn > 0) dp = __double2float_rn(x / (double)min(a * (c - b), (c - a) * b));
    else if (dn < 0) dp = __double2float_rn(x / (double)min(a * b, (c - a) * (c - b)));
    else dp = 0.0f;
}

// A pair is linked when its FP64 r^2 exceeds the threshold; a NaN r^2 (c == 0, or a site monomorphic among the
// jointly called) never is.
__device__ __forceinline__ bool fm_ld_linked(int64_t c, int64_t a, int64_t b, int64_t ab, double r2_threshold) {
    if (c == 0 || a == 0 || a == c || b == 0 || b == c) return false;
    return fm_ld_r2(c, a, b, c * ab - a * b) > r2_threshold;
}

// Output of the bit epilogue of fm_k_ld_band: bit d - 1 of the forward row i (row_words u32 words from bits + i *
// row_words) is set when (i, i + d) is linked; *linked counts the linked pairs.
struct LdBits {
    double r2_threshold;
    uint32_t row_words;
    uint32_t *bits;
    unsigned long long *linked;
};

// Banded upper-triangle bit product over one slab of row blocks [rb0, rb0 + gridDim.x / tpr).  CTA t is tile
// (bi, bj) = (rb0 + t / tpr, bi + t % tpr); tpr = ceil(window / 64) + 1 tiles per row block cover every (i, d) with
// 1 <= d <= window exactly once.  Warp kLdConsumerWarps is the producer of the tile's PwRing; a tile past the last
// site block has no chunks and only writes its NaN cells.  Consumer thread (ti, tj) owns the sites
// i = 64 bi + 4 ti + {0..3} and j = 64 bj + tj + 16 {0..3}, so that for each of its pairs the 16 threads of a row
// write 16 consecutive floats.  out_r2 / out_dp hold the slab's rows: [(i - 64 rb0) * window + d - 1].
// BITS selects the bit epilogue instead (out_r2 / out_dp unused, rb0 = 0): each (x, y) of the micro-tile is one
// ballot, whose two 16-lane halves are 16 consecutive d of one row i and go to the row's words with one atomicOr each
// (OR is order-independent, so the bits do not depend on the tile schedule); one atomicAdd per CTA counts the pairs.
template <bool HC, bool BITS>
__global__ void __launch_bounds__((kLdConsumerWarps + 1) * 32)
fm_k_ld_band(const uint32_t *__restrict__ planes, PwLayout L, uint32_t n_chunks, uint32_t n, uint32_t M,
             uint32_t window, int64_t max_distance, uint32_t rb0, uint32_t tpr, const uint32_t *__restrict__ kalt,
             const int64_t *__restrict__ kpos, float *__restrict__ out_r2, float *__restrict__ out_dp, LdBits lb) {
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
    if constexpr (BITS) {
        __shared__ uint32_t cta_linked;
        if (threadIdx.x == 0) cta_linked = 0;
        asm volatile("bar.sync 1, %0;" ::"n"(kLdConsumerWarps * 32) : "memory");
        uint32_t n_linked = 0;
#pragma unroll
        for (int x = 0; x < 4; ++x) {
            const uint32_t gi = bi * kPwBlk + ti * 4u + x;
            const uint32_t alt_i = HC || gi >= M ? 0u : kalt[gi];
#pragma unroll
            for (int y = 0; y < 4; ++y) {
                const uint32_t gj = bj * kPwBlk + tj + 16u * y;
                bool linked = false;
                if (gj > gi && gj - gi <= window && gj < M && (max_distance < 0 || kpos[gj] - kpos[gi] <= max_distance)) {
                    if (HC) linked = fm_ld_linked(acc_c[x][y], acc_a[x][y], acc_b[x][y], acc_ab[x][y], lb.r2_threshold);
                    else linked = fm_ld_linked(n, alt_i, kalt[gj], acc_ab[x][y], lb.r2_threshold);
                }
                const uint32_t bal = __ballot_sync(0xffffffffu, linked);
                n_linked += __popc(bal);
                // lane 0 of each half: bit t of its 16 is d = gj(tj = 0) - gi + t, so bit d - 1 = start + t
                const uint32_t half = (bal >> (lane & 16u)) & 0xffffu;
                if ((lane & 15u) == 0 && half) {
                    const int32_t start = (int32_t)(bj * kPwBlk + 16u * y) - (int32_t)gi - 1;
                    // bits t < -start are pairs with gj <= gi and never set
                    const uint32_t b0 = start < 0 ? 0u : (uint32_t)start;
                    const uint64_t v = start < 0 ? (uint64_t)(half >> -start) : (uint64_t)half << (b0 & 31u);
                    uint32_t *row = lb.bits + (size_t)gi * lb.row_words + (b0 >> 5);
                    atomicOr(row, (uint32_t)v);
                    if (v >> 32) atomicOr(row + 1, (uint32_t)(v >> 32));  // a set bit above 31 is below w: in the row
                }
            }
        }
        if (lane == 0 && n_linked) atomicAdd(&cta_linked, n_linked);
        asm volatile("bar.sync 1, %0;" ::"n"(kLdConsumerWarps * 32) : "memory");
        if (threadIdx.x == 0 && cta_linked) atomicAdd(lb.linked, (unsigned long long)cta_linked);
        return;
    } else {
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
}

// Greedy pruning scan over the forward bit rows of the bit epilogue (row_words words a row): site j is retained
// unless a retained site i < j is linked to it.  The rule is a chain along the sites, so one CTA walks them 32 at a
// time.  `ring` (ring_mask + 1 >= row_words + 1 words, a power of two) holds the blocked bits of the sites ahead:
// word b & ring_mask is sites 32 b .. 32 b + 31.  Per block, warp 0 resolves the links inside the block with a serial
// bit loop (lane t holds row j0 + t's first word, shifted to block coordinates); then every thread ORs word k of the
// retained rows, shifted by t + 1, into ring words b + k and b + k + 1.  The rows of the next block are loaded before
// the chain of the current one (thread k holds word k of all 32 rows, for k < blockDim.x), since they do not depend
// on it.  retained[j] = 1 for a retained site, *n_retained their number.
constexpr uint32_t kLdScanThreads = 256;

__global__ void __launch_bounds__(kLdScanThreads)
fm_k_ld_prune_scan(const uint32_t *__restrict__ bits, uint32_t M, uint32_t row_words, uint32_t ring_mask,
                   uint8_t *__restrict__ retained, uint32_t *__restrict__ n_retained) {
    constexpr uint32_t FULL = 0xffffffffu;
    extern __shared__ uint32_t ring[];
    __shared__ uint32_t s_keep;
    const uint32_t tid = threadIdx.x, lane = tid & 31;
    for (uint32_t k = tid; k <= ring_mask; k += blockDim.x) ring[k] = 0;
    const uint32_t n_blocks = (M + 31) / 32;
    uint32_t nxt[32], w0_nxt = 0, count = 0;
    auto load = [&](uint32_t b) {
        const uint32_t j0 = b * 32u;
#pragma unroll
        for (uint32_t t = 0; t < 32; ++t)
            nxt[t] = tid < row_words && j0 + t < M ? __ldg(bits + (size_t)(j0 + t) * row_words + tid) : 0u;
        if (tid < 32) w0_nxt = j0 + lane < M ? __ldg(bits + (size_t)(j0 + lane) * row_words) : 0u;
    };
    load(0);
    __syncthreads();
    for (uint32_t b = 0; b < n_blocks; ++b) {
        uint32_t cur[32];
#pragma unroll
        for (uint32_t t = 0; t < 32; ++t) cur[t] = nxt[t];
        const uint32_t w0 = w0_nxt;
        if (b + 1 < n_blocks) load(b + 1);
        const uint32_t j0 = b * 32u, n_t = min(32u, M - j0);
        if (tid < 32) {
            uint32_t blocked = ring[b & ring_mask];
            const uint32_t intra = lane < 31 ? w0 << (lane + 1) : 0u;  // row j0 + lane's links inside the block
            uint32_t v[32];
#pragma unroll
            for (uint32_t t = 0; t < 32; ++t) v[t] = __shfl_sync(FULL, intra, t);
#pragma unroll
            for (uint32_t t = 0; t < 32; ++t)
                if (!((blocked >> t) & 1u)) blocked |= v[t];  // v[t] has no bit at or below t
            const uint32_t keep = ~blocked & (n_t == 32 ? FULL : (1u << n_t) - 1u);
            if (lane < n_t) retained[j0 + lane] = (keep >> lane) & 1u;
            if (lane == 0) {
                s_keep = keep;
                ring[b & ring_mask] = 0;  // the slot's next use is block b + ring_mask + 1
                count += __popc(keep);
            }
        }
        __syncthreads();
        const uint32_t keep = s_keep;
        for (uint32_t k = tid; k < row_words; k += blockDim.x) {
            uint32_t lo = 0, hi = 0;
#pragma unroll
            for (uint32_t t = 0; t < 32; ++t) {
                if (!((keep >> t) & 1u)) continue;
                const uint32_t r = k == tid ? cur[t] : __ldg(bits + (size_t)(j0 + t) * row_words + k);
                const uint64_t sh = (uint64_t)r << (t + 1);
                lo |= (uint32_t)sh;
                hi |= (uint32_t)(sh >> 32);
            }
            if (k && lo) atomicOr(&ring[(b + k) & ring_mask], lo);  // word 0's low part is this block: resolved
            if (hi) atomicOr(&ring[(b + k + 1) & ring_mask], hi);
        }
        __syncthreads();
    }
    if (tid == 0) *n_retained = count;
}

}  // namespace fm
