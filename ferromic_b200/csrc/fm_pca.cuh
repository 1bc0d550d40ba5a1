// fm_pca.cuh -- haplotype PCA by randomized subspace iteration (DESIGN.md §0 row f8, §3 and §4 "Haplotype PCA").
//
// Z[i, v] = s_v (x_iv - p_v) for a called cell and 0 for a missing one, over the n selected haplotypes i and the M
// kept sites v (filters and standardization in include/ferromic_gpu.h; site counts and filter in fm_haplotypes.cuh).
// The kernels here produce the per-site scales, the haplotype-major bit planes of the kept sites and the two FP64
// products every iteration needs:
//   W = Z^T Q  (M x l, sites <- haplotypes)     and     Y = Z R  (n x l, haplotypes <- sites).
// A cell's value is rebuilt from two bits: alt (called, raw allele 1) and called, with the per-site pair
// u1_v = s_v (1 - p_v), u0_v = s_v (0 - p_v):  z = alt ? u1 : (called ? u0 : 0).  These are the products
// s_v (x - p_v) of the definition, so every Z entry is the restatement's value bit for bit; only the summation
// order of the products differs.  Without missing cells among the kept sites there is no called plane and
// z = alt ? u1 : u0.  Every sum runs in a fixed order (no FP64 atomics), so equal inputs give equal bits.
#pragma once
#include "fm_device.cuh"
#include "fm_haplotypes.cuh"  // HapCells
#include "fm_kernels.cuh"     // fm_mix
#include "fm_pairwise.cuh"    // PwLayout, kPwBlk, kPwKT

namespace fm {

constexpr uint32_t kPcaCols = 8;                 // output columns per thread
constexpr uint32_t kPcaRows = 4;                 // output rows (sites or haplotypes) per thread
constexpr uint32_t kPcaChunk = kPwKT * 32;       // kept sites per K-chunk of the plane layout (256)
constexpr uint32_t kPcaHapBlocks = 4;            // haplotype blocks of 64 per CTA of the Z R product
constexpr uint32_t kPcaMaxRank = 64;             // l <= 64
constexpr uint32_t kPcaWordPitch = kPwBlk + 1;   // padded shared-memory pitch of a staged (plane, word) row

// Per kept site j (matrix row kept[j]): u[2j] = s (1 - p), u[2j + 1] = s (0 - p) with p = alt / called and
// s = 1 / sqrt(p (1 - p)); T += called (integer).
__global__ void __launch_bounds__(256)
fm_k_pca_scales(const uint32_t *__restrict__ kept, uint32_t M, uint32_t v_lo, const uint32_t *__restrict__ alt,
                const uint32_t *__restrict__ called, double *__restrict__ u, unsigned long long *__restrict__ total) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= M) return;
    const uint32_t r = kept[j] - v_lo;
    const uint32_t c = called[r];
    const double p = (double)alt[r] / (double)c;
    const double s = 1.0 / sqrt(p * (1.0 - p));
    u[2 * (size_t)j] = s * (1.0 - p);
    u[2 * (size_t)j + 1] = s * (0.0 - p);
    atomicAdd(total, (unsigned long long)c);
}

// Kept sites x selected haplotypes -> K-tiled, haplotype-major planes of PwLayout (plane 0 alt, plane 1 called when
// present).  One warp per (kept-site word, 32 haplotypes), lane = haplotype; padded words and haplotypes stay zero.
__global__ void __launch_bounds__(256)
fm_k_pca_planes(HapCells cells, const uint32_t *__restrict__ off, uint32_t n, const uint32_t *__restrict__ kept,
                uint32_t M, uint32_t n_words, PwLayout L, uint32_t *__restrict__ planes) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t groups = (n + 31) / 32;
    const uint64_t n_tasks = (uint64_t)n_words * groups;
    const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t task = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; task < n_tasks; task += n_warps) {
        const uint32_t w = (uint32_t)(task / groups), h = (uint32_t)(task % groups) * 32 + lane;
        if (h >= n) continue;
        const uint32_t col = __ldg(off + h);
        uint32_t a = 0, c = 0;
        const uint32_t n_t = min(32u, M - w * 32u);
        for (uint32_t t = 0; t < n_t; ++t) {
            bool called, alt, other;
            cells.read(__ldg(kept + w * 32u + t), col, called, alt, other);
            a |= (uint32_t)alt << t;
            c |= (uint32_t)called << t;
        }
        planes[L.word(w, h, 0)] = a;
        if (L.planes > 1) planes[L.word(w, h, 1)] = c;
    }
}

template <bool HC>
__device__ __forceinline__ double fm_pca_z(uint32_t a, uint32_t c, uint32_t bit, double u1, double u0) {
    if ((a >> bit) & 1u) return u1;
    if (!HC) return u0;
    return ((c >> bit) & 1u) ? u0 : 0.0;
}

// W = Z^T Q.  One CTA per K-chunk of 256 kept sites; 64 x n_cg threads, thread (sg, cg) owns the sites 4 sg .. 4 sg + 3
// of the chunk and the columns 8 cg .. 8 cg + 7.  Per 64-haplotype block the CTA stages the block's Q rows (zero past
// l and past n) and its bit words; each haplotype then costs a thread 4 cell values and 32 FMA.  W is M x l
// row-major; every entry sums the haplotypes in ascending order.
template <bool HC>
__global__ void __launch_bounds__(512)
fm_k_pca_zt_q(const uint32_t *__restrict__ planes, PwLayout L, const double *__restrict__ u,
              const double *__restrict__ Q, uint32_t n, uint32_t M, uint32_t l, double *__restrict__ W) {
    extern __shared__ __align__(16) uint8_t pca_smem[];
    const uint32_t n_cg = blockDim.x / 64, lp = n_cg * kPcaCols;
    double *qs = reinterpret_cast<double *>(pca_smem);                          // [64][lp]
    uint32_t *bs = reinterpret_cast<uint32_t *>(qs + (size_t)kPwBlk * lp);      // [planes * 8][65]
    const uint32_t c = blockIdx.x, tid = threadIdx.x, sg = tid & 63, cg = tid >> 6;
    const uint32_t k = sg >> 3, sh = (sg & 7) * 4;
    double u1[kPcaRows], u0[kPcaRows], acc[kPcaRows][kPcaCols];
#pragma unroll
    for (int r = 0; r < (int)kPcaRows; ++r) {
        const uint32_t j = c * kPcaChunk + sg * 4 + r;
        u1[r] = j < M ? u[2 * (size_t)j] : 0.0;
        u0[r] = j < M ? u[2 * (size_t)j + 1] : 0.0;
#pragma unroll
        for (int q = 0; q < (int)kPcaCols; ++q) acc[r][q] = 0.0;
    }
    const uint32_t tile_w = L.tile_words();
    for (uint32_t b = 0; b < L.n_blk; ++b) {
        __syncthreads();  // the previous block's tiles are consumed
        for (uint32_t e = tid; e < kPwBlk * lp; e += blockDim.x) {
            const uint32_t i = b * kPwBlk + e / lp, q = e % lp;
            qs[e] = (i < n && q < l) ? Q[(size_t)i * l + q] : 0.0;
        }
        const uint32_t *src = planes + ((size_t)c * L.n_blk + b) * tile_w;
        for (uint32_t e = tid; e < tile_w; e += blockDim.x) bs[(e / kPwBlk) * kPcaWordPitch + e % kPwBlk] = src[e];
        __syncthreads();
        const uint32_t *ba = bs + k * kPcaWordPitch, *bc = bs + (kPwKT + k) * kPcaWordPitch;
        const double2 *qrow = reinterpret_cast<const double2 *>(qs) + cg * (kPcaCols / 2);
#pragma unroll 2
        for (uint32_t i = 0; i < kPwBlk; ++i) {
            const uint32_t a = ba[i], cw = HC ? bc[i] : 0u;
            double z[kPcaRows];
#pragma unroll
            for (int r = 0; r < (int)kPcaRows; ++r) z[r] = fm_pca_z<HC>(a, cw, sh + r, u1[r], u0[r]);
            const double2 *qi = qrow + (size_t)i * (lp / 2);
#pragma unroll
            for (int q2 = 0; q2 < (int)kPcaCols / 2; ++q2) {
                const double2 qq = qi[q2];
#pragma unroll
                for (int r = 0; r < (int)kPcaRows; ++r) {
                    acc[r][2 * q2] = fma(z[r], qq.x, acc[r][2 * q2]);
                    acc[r][2 * q2 + 1] = fma(z[r], qq.y, acc[r][2 * q2 + 1]);
                }
            }
        }
    }
#pragma unroll
    for (int r = 0; r < (int)kPcaRows; ++r) {
        const uint32_t j = c * kPcaChunk + sg * 4 + r;
        if (j >= M) continue;
#pragma unroll
        for (int q = 0; q < (int)kPcaCols; ++q)
            if (cg * kPcaCols + q < l) W[(size_t)j * l + cg * kPcaCols + q] = acc[r][q];
    }
}

// Y = Z R, partial over a slice of K-chunks.  CTA (slice, hb) owns the haplotypes of kPcaHapBlocks blocks from
// 64 hb * kPcaHapBlocks on; 64 x n_cg threads, thread (hg, cg) owns the haplotypes 4 hg .. 4 hg + 3 of them and
// the columns 8 cg .. 8 cg + 7.  Per chunk the CTA stages the chunk's R rows (G generated inline when R is null:
// +1 when bit 63 of fm_mix(seed, matrix row, column) is clear, else -1), the site pairs u and the blocks' bit words.
// part[slice][n][l] holds the slice's sum over its sites in ascending order; fm_k_pca_fold adds the slices in order.
template <bool HC>
__global__ void __launch_bounds__(512)
fm_k_pca_z_r(const uint32_t *__restrict__ planes, PwLayout L, const double *__restrict__ u,
             const double *__restrict__ R, const uint32_t *__restrict__ kept, uint64_t seed, uint32_t n, uint32_t M,
             uint32_t l, uint32_t n_chunks, uint32_t chunks_per_slice, double *__restrict__ part) {
    extern __shared__ __align__(16) uint8_t pca_smem[];
    const uint32_t n_cg = blockDim.x / 64, lp = n_cg * kPcaCols;
    double *rs = reinterpret_cast<double *>(pca_smem);                        // [256][lp]
    double2 *us = reinterpret_cast<double2 *>(rs + (size_t)kPcaChunk * lp);   // [256]
    uint32_t *bs = reinterpret_cast<uint32_t *>(us + kPcaChunk);              // kPcaHapBlocks tiles
    const uint32_t slice = blockIdx.x, hb = blockIdx.y, tid = threadIdx.x, hg = tid & 63, cg = tid >> 6;
    const uint32_t b0 = hb * kPcaHapBlocks, nb = min(kPcaHapBlocks, L.n_blk - b0);
    const uint32_t tile_w = L.tile_words();
    const uint32_t bl = hg / 16, sl = (hg % 16) * 4;  // block and first haplotype of this thread inside the CTA
    double acc[kPcaRows][kPcaCols];
#pragma unroll
    for (int r = 0; r < (int)kPcaRows; ++r)
#pragma unroll
        for (int q = 0; q < (int)kPcaCols; ++q) acc[r][q] = 0.0;
    const uint32_t c_lo = slice * chunks_per_slice, c_hi = min(n_chunks, c_lo + chunks_per_slice);
    for (uint32_t c = c_lo; c < c_hi; ++c) {
        __syncthreads();
        for (uint32_t e = tid; e < kPcaChunk * lp; e += blockDim.x) {
            const uint32_t t = e / lp, q = e % lp, j = c * kPcaChunk + t;
            double x = 0.0;
            if (j < M && q < l) {
                if (R) x = R[(size_t)j * l + q];
                else x = (fm_mix(seed, __ldg(kept + j), q) >> 63) == 0 ? 1.0 : -1.0;
            }
            rs[e] = x;
        }
        for (uint32_t t = tid; t < kPcaChunk; t += blockDim.x) {
            const uint32_t j = c * kPcaChunk + t;
            us[t] = j < M ? make_double2(u[2 * (size_t)j], u[2 * (size_t)j + 1]) : make_double2(0.0, 0.0);
        }
        const uint4 *src = reinterpret_cast<const uint4 *>(planes + ((size_t)c * L.n_blk + b0) * tile_w);
        for (uint32_t e = tid; e < nb * tile_w / 4; e += blockDim.x) reinterpret_cast<uint4 *>(bs)[e] = src[e];
        __syncthreads();
        if (bl >= nb) continue;
        const uint32_t *tile = bs + bl * tile_w;
#pragma unroll 1
        for (uint32_t k = 0; k < kPwKT; ++k) {
            const uint4 av = *reinterpret_cast<const uint4 *>(tile + k * kPwBlk + sl);
            uint4 cv = make_uint4(0, 0, 0, 0);
            if (HC) cv = *reinterpret_cast<const uint4 *>(tile + (kPwKT + k) * kPwBlk + sl);
            const uint32_t a[4] = {av.x, av.y, av.z, av.w}, cw[4] = {cv.x, cv.y, cv.z, cv.w};
#pragma unroll 2
            for (uint32_t t = 0; t < 32; ++t) {
                const double2 uu = us[k * 32 + t];
                double z[kPcaRows];
#pragma unroll
                for (int r = 0; r < (int)kPcaRows; ++r) z[r] = fm_pca_z<HC>(a[r], cw[r], t, uu.x, uu.y);
                const double2 *ri = reinterpret_cast<const double2 *>(rs + (size_t)(k * 32 + t) * lp) + cg * (kPcaCols / 2);
#pragma unroll
                for (int q2 = 0; q2 < (int)kPcaCols / 2; ++q2) {
                    const double2 rr = ri[q2];
#pragma unroll
                    for (int r = 0; r < (int)kPcaRows; ++r) {
                        acc[r][2 * q2] = fma(z[r], rr.x, acc[r][2 * q2]);
                        acc[r][2 * q2 + 1] = fma(z[r], rr.y, acc[r][2 * q2 + 1]);
                    }
                }
            }
        }
    }
    if (bl >= nb) return;
#pragma unroll
    for (int r = 0; r < (int)kPcaRows; ++r) {
        const uint32_t i = (b0 + bl) * kPwBlk + sl + r;
        if (i >= n) continue;
#pragma unroll
        for (int q = 0; q < (int)kPcaCols; ++q)
            if (cg * kPcaCols + q < l) part[((size_t)slice * n + i) * l + cg * kPcaCols + q] = acc[r][q];
    }
}

// Y[e] = sum over the slices, in slice order, of part[slice][e] (e < n * l).
__global__ void __launch_bounds__(256)
fm_k_pca_fold(const double *__restrict__ part, uint32_t n_slices, uint64_t n_el, double *__restrict__ Y) {
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_el) return;
    double s = 0.0;
    for (uint32_t k = 0; k < n_slices; ++k) s += part[(size_t)k * n_el + e];
    Y[e] = s;
}

// C = W^T W, partial per CTA over an equal share of the M sites (CTA order fixed by the grid, not by the device):
// part[cta][a * l + b] = sum over its sites, in ascending order, of W[v][a] W[v][b].  Entry (a, b) and (b, a) run
// the same products, so the folded C is exactly symmetric.
__global__ void __launch_bounds__(256)
fm_k_pca_gram(const double *__restrict__ W, uint32_t M, uint32_t l, double *__restrict__ part) {
    const uint32_t per = (M + gridDim.x - 1) / gridDim.x;
    const uint32_t v_lo = min(M, blockIdx.x * per), v_hi = min(M, v_lo + per);
    for (uint32_t e = threadIdx.x; e < l * l; e += blockDim.x) {
        const uint32_t a = e / l, b = e % l;
        double s = 0.0;
        for (uint32_t v = v_lo; v < v_hi; ++v) s = fma(W[(size_t)v * l + a], W[(size_t)v * l + b], s);
        part[(size_t)blockIdx.x * l * l + e] = s;
    }
}

}  // namespace fm
