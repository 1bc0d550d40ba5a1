// fm_sfs.cuh -- site frequency spectra of one haplotype set (projected, per window) and of two sets (joint)
// (DESIGN.md §4 "Site frequency spectra"; estimator in include/ferromic_gpu.h).
//
// 1. fm_k_sfs_counts reads every candidate row once and counts (called, alt, other) over the cells of one or two
//    sets: u8 rows 16 bytes a lane with byte-SIMD compares, packed rows a u32 word a lane with popcounts.  It flags the
//    contributing rows, which cub::DeviceSelect compacts in row order; fm_k_sfs_gather lines up their counts.
// 2. fm_k_sfs_spectrum: one CTA owns a T1 x T2 tile of one spectrum and walks the contributing rows that touch it in
//    row order, so every entry is one FP64 sum in a fixed order (no atomics).  A 1-D window's rows are a contiguous
//    range of the compacted list; a joint tile's rows are its segment of the (tile, row) incidences, stably sorted.
#pragma once
#include "fm_haplotypes.cuh"

namespace fm {

constexpr uint32_t kSfsCountThreads = 256;
constexpr uint32_t kSfsTile1 = 128;   // 1-D spectrum: bins per CTA (one thread each)
constexpr uint32_t kSfsJointTile = 16;  // joint spectrum: 16 x 16 entries per CTA

// The cells of one or two haplotype sets.  u8 rows: memb holds, for each of the 16 alignments s = (v * stride) & 15 of
// a row start, Lb 16-byte blocks of membership bytes (bit 0: set 1, bit 1: set 2) so that a row's aligned 16-byte
// blocks line up with aligned membership blocks.  Packed rows: mask [sets][rw] member bits.
struct SfsCells {
    HapCells c;
    const uint8_t *memb;
    uint32_t memb_blocks;  // Lb
    const uint32_t *mask;
};

// 4 membership / missing bits -> 4 bytes of 0x00 / 0xff
__device__ __forceinline__ uint32_t sfs_nibble_bytes(uint32_t nib) { return ((nib * 0x00204081u) & 0x01010101u) * 0xffu; }

// (called, alt, other) of set 1 and set 2 at row v, summed over the warp's lanes into lane 0's registers.
template <bool TWO>
__device__ __forceinline__ void sfs_row_counts(const SfsCells &s, uint32_t v, uint32_t lane, uint32_t (&k)[6]) {
#pragma unroll
    for (int i = 0; i < 6; ++i) k[i] = 0;
    const HapCells &c = s.c;
    if (c.abits) {
        const uint32_t *ar = c.abits + (size_t)v * c.rw;
        const uint32_t *cr = c.cbits ? c.cbits + (size_t)v * c.rw : nullptr;
        for (uint32_t w = lane; w < c.rw; w += 32) {
            const uint32_t cw = cr ? __ldg(cr + w) : 0xffffffffu;
            const uint32_t aw = __ldg(ar + w) & cw;
            const uint32_t k1 = __ldg(s.mask + w);
            k[0] += __popc(cw & k1);
            k[1] += __popc(aw & k1);
            if (TWO) {
                const uint32_t k2 = __ldg(s.mask + c.rw + w);
                k[3] += __popc(cw & k2);
                k[4] += __popc(aw & k2);
            }
        }
    } else {
        const uint64_t e_row = (uint64_t)v * c.stride;
        const uint64_t b0 = e_row >> 4;
        const uint64_t nb = ((e_row + c.stride - 1) >> 4) - b0 + 1;
        const uint4 *rows = reinterpret_cast<const uint4 *>(c.data);  // the matrix is 16-byte aligned
        const uint4 *mb = reinterpret_cast<const uint4 *>(s.memb) + (size_t)(e_row & 15) * s.memb_blocks;
        for (uint32_t b = lane; b < nb; b += 32) {
            const uint4 x4 = __ldg(rows + b0 + b);
            const uint4 m4 = __ldg(mb + b);
            uint32_t miss = 0;
            if (c.miss_mode == 1) {
                const uint64_t e0 = (b0 + b) << 4;
                miss = (uint32_t)(__ldg(c.missing + (e0 >> 6)) >> (e0 & 63)) & 0xffffu;
            }
            const uint32_t xs[4] = {x4.x, x4.y, x4.z, x4.w}, ms[4] = {m4.x, m4.y, m4.z, m4.w};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const uint32_t x = xs[q];
                uint32_t called = 0xffffffffu;
                if (c.miss_mode == 1) called = ~sfs_nibble_bytes((miss >> (4 * q)) & 15u);
                else if (c.miss_mode == 2) called = __vcmpltu4(x, 0x80808080u);
                const uint32_t one = __vcmpeq4(x, 0x01010101u), more = __vcmpgtu4(x, 0x01010101u);
                const uint32_t c1 = called & ((ms[q] & 0x01010101u) * 0xffu);
                k[0] += __popc(c1);
                k[1] += __popc(c1 & one);
                k[2] += __popc(c1 & more);
                if (TWO) {
                    const uint32_t c2 = called & (((ms[q] >> 1) & 0x01010101u) * 0xffu);
                    k[3] += __popc(c2);
                    k[4] += __popc(c2 & one);
                    k[5] += __popc(c2 & more);
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 6; ++i) k[i] >>= 3;  // 8 bits a byte
    }
#pragma unroll
    for (int d = 16; d; d >>= 1)
#pragma unroll
        for (int i = 0; i < 6; ++i) k[i] += __shfl_xor_sync(0xffffffffu, k[i], d);
}

// Counting pass over rows [v_lo, v_lo + R): one warp a row, grid-strided.  cnt1 / cnt2 [R] = (called, alt);
// flag [R] = 1 for a contributing row; tot [3] += (candidates, projected_out, non_biallelic).  allow (nullable) limits
// the candidates to a site list.
template <bool TWO>
__global__ void __launch_bounds__(kSfsCountThreads)
fm_k_sfs_counts(SfsCells cells, uint32_t v_lo, uint32_t R, const uint8_t *__restrict__ allow, uint32_t m1, uint32_t m2,
                uint2 *__restrict__ cnt1, uint2 *__restrict__ cnt2, uint8_t *__restrict__ flag,
                unsigned long long *__restrict__ tot) {
    __shared__ uint32_t sh[3];
    if (threadIdx.x < 3) sh[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t warps = gridDim.x * (kSfsCountThreads / 32);
    uint32_t cand = 0, po = 0, nbi = 0;
    for (uint32_t r = blockIdx.x * (kSfsCountThreads / 32) + (threadIdx.x >> 5); r < R; r += warps) {
        if (allow && !allow[r]) {
            if (!lane) flag[r] = 0;
            continue;
        }
        uint32_t k[6];
        sfs_row_counts<TWO>(cells, v_lo + r, lane, k);
        if (lane) continue;
        const bool non_bi = k[2] > 0 || (TWO && k[5] > 0);
        const bool proj = !non_bi && (k[0] < m1 || (TWO && k[3] < m2));
        cand++;
        po += proj;
        nbi += non_bi;
        cnt1[r] = make_uint2(k[0], k[1]);
        if (TWO) cnt2[r] = make_uint2(k[3], k[4]);
        flag[r] = !non_bi && !proj;
    }
    if (!lane) {
        atomicAdd(&sh[0], cand);
        atomicAdd(&sh[1], po);
        atomicAdd(&sh[2], nbi);
    }
    __syncthreads();
    if (threadIdx.x < 3 && sh[threadIdx.x]) atomicAdd(tot + threadIdx.x, (unsigned long long)sh[threadIdx.x]);
}

// out1 / out2 [n] = the counts of the compacted contributing rows ci [n]
__global__ void __launch_bounds__(256)
fm_k_sfs_gather(const uint32_t *__restrict__ ci, uint32_t n, const uint2 *__restrict__ cnt1,
                const uint2 *__restrict__ cnt2, uint2 *__restrict__ out1, uint2 *__restrict__ out2) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t r = ci[i];
    out1[i] = cnt1[r];
    if (cnt2) out2[i] = cnt2[r];
}

// Window w's contributing rows: [lo_out[w], hi_out[w]) of the ascending row list ci [n], for rows [lo[w], hi[w]).
__global__ void __launch_bounds__(256)
fm_k_sfs_window_bounds(const uint32_t *__restrict__ ci, uint32_t n, const uint32_t *__restrict__ lo,
                       const uint32_t *__restrict__ hi, uint32_t n_windows, uint32_t *__restrict__ lo_out,
                       uint32_t *__restrict__ hi_out) {
    const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= n_windows) return;
    auto lower = [&](uint32_t key) {
        uint32_t a = 0, b = n;
        while (a < b) {
            const uint32_t mid = (a + b) >> 1;
            if (ci[mid] < key) a = mid + 1;
            else b = mid;
        }
        return a;
    };
    lo_out[w] = lower(lo[w]);
    hi_out[w] = max(lower(hi[w]), lo_out[w]);
}

// ------------------------------------------------------------------------------------ weights
// Loader's saddle-point form (R's dbinom_raw / dhyper): stirlerr(n) = log(n!) - log(sqrt(2 pi)) - (n + 1/2) log(n) + n
// and bd0(x, np) = x log(x / np) + np - x, each without cancellation.
__constant__ double kSfsStirlerr[16] = {
    0.0, 8.1061466795327258219670264e-2, 4.1340695955409294093822081e-2, 2.7677925684998339148789293e-2,
    2.0790672103765093111522772e-2, 1.6644691189821192163194865e-2, 1.3876128823070747998745727e-2,
    1.1896709945891770095055724e-2, 1.0411265261972096497478567e-2, 9.2554621827127329177286366e-3,
    8.3305634333628712564693187e-3, 7.5736754879518407949720242e-3, 6.9428401072095298656641527e-3,
    6.4089941880042070684396311e-3, 5.9513701127588477356244160e-3, 5.5547335519628013710386900e-3};

__device__ __forceinline__ double sfs_stirlerr(double n) {
    constexpr double S0 = 1.0 / 12, S1 = 1.0 / 360, S2 = 1.0 / 1260, S3 = 1.0 / 1680, S4 = 1.0 / 1188;
    if (n <= 15.0) return kSfsStirlerr[(int)n];
    const double nn = n * n;
    if (n > 500.0) return (S0 - S1 / nn) / n;
    if (n > 80.0) return (S0 - (S1 - S2 / nn) / nn) / n;
    if (n > 35.0) return (S0 - (S1 - (S2 - S3 / nn) / nn) / nn) / n;
    return (S0 - (S1 - (S2 - (S3 - S4 / nn) / nn) / nn) / nn) / n;
}

__device__ __forceinline__ double sfs_bd0(double x, double np) {
    if (fabs(x - np) < 0.1 * (x + np)) {
        double v = (x - np) / (x + np);
        double s = (x - np) * v;
        double ej = 2.0 * x * v;
        v = v * v;
        for (int j = 1; j < 1000; ++j) {
            ej *= v;
            const double s1 = s + ej / (double)(2 * j + 1);
            if (s1 == s) return s1;
            s = s1;
        }
    }
    return x * log(x / np) + np - x;
}

__device__ __forceinline__ double sfs_dbinom_raw(double x, double n, double p, double q) {
    if (p == 0.0) return x == 0.0 ? 1.0 : 0.0;
    if (q == 0.0) return x == n ? 1.0 : 0.0;
    if (x == 0.0) {
        if (n == 0.0) return 1.0;
        return exp(p < 0.1 ? -sfs_bd0(n, n * q) - n * p : n * log(q));
    }
    if (x == n) return exp(q < 0.1 ? -sfs_bd0(n, n * p) - n * q : n * log(p));
    const double lc = sfs_stirlerr(n) - sfs_stirlerr(x) - sfs_stirlerr(n - x) - sfs_bd0(x, n * p) - sfs_bd0(n - x, n * q);
    const double lf = 1.837877066409345483560659472811 + log(x) + log1p(-x / n);
    return exp(lc - 0.5 * lf);
}

// Weights h(j; N, a, m) of the bins j in [from, to] (inside the support [lo, hi], lo < hi) into dst[j - base]: the
// support's mode md by Loader's form, then the exact ratio walked outward one bin at a time -- upward from md
// (`up`, which also writes md) or downward from md - 1.  Every value is a fixed function of (N, a, m, j).
__device__ __forceinline__ void sfs_walk(uint32_t N, uint32_t a, uint32_t m, uint32_t lo, uint32_t hi, uint32_t from,
                                         uint32_t to, bool up, double *dst, uint32_t base) {
    const uint32_t md = min(max((uint32_t)(((uint64_t)(m + 1) * (a + 1)) / (N + 2)), lo), hi);
    if (up ? to < md : from >= md) return;
    const double p = (double)m / (double)N, q = (double)(N - m) / (double)N;
    const double h0 = sfs_dbinom_raw(md, a, p, q) * sfs_dbinom_raw(m - md, N - a, p, q) / sfs_dbinom_raw(m, N, p, q);
    double h = h0;
    uint32_t j = md;
    if (up) {
        if (j >= from) dst[j - base] = h;
        for (; j < to; ++j) {
            h *= (double)((uint64_t)(a - j) * (m - j)) / (double)((uint64_t)(j + 1) * (N - a - m + j + 1));
            if (j + 1 >= from) dst[j + 1 - base] = h;
        }
    } else {
        for (; j > from; --j) {
            h *= (double)((uint64_t)j * (N - a - m + j)) / (double)((uint64_t)(a - j + 1) * (m - j + 1));
            if (j - 1 <= to) dst[j - 1 - base] = h;
        }
    }
}

// support [lo, hi] of (N, a, m): j with C(a, j) C(N - a, m - j) != 0
__device__ __forceinline__ void sfs_support(uint2 na, uint32_t m, uint32_t &lo, uint32_t &hi) {
    lo = m + na.y > na.x ? m + na.y - na.x : 0u;
    hi = min(na.y, m);
}

// ------------------------------------------------------------------------------------ spectrum pass
// CTA b owns tile t = b % n_tiles of spectrum w = b / n_tiles: entries j1 in [t1 T1, t1 T1 + T1), j2 in [t2 T2, ...)
// with (t1, t2) = (t / tiles2, t % tiles2).  Its rows are [seg[g], seg_hi[g]) of `list` (null: the identity), with
// g = t when list is given (joint incidences) and g = w otherwise (1-D windows).  Row i has counts c1[i] and, when c2
// is given, c2[i]; without c2 the second axis is the single bin 0 of weight 1.  The CTA compacts the rows of each
// chunk that touch its tile (in order), computes their weights four threads a row (set 1 / set 2, up / down) into
// shared memory, and each thread adds h1 h2 of its entry row by row.  accumulate: start from out (a later chunk of
// joint rows) instead of 0.
template <int T1, int T2>
__global__ void __launch_bounds__(T1 *T2, 2)
fm_k_sfs_spectrum(const uint2 *__restrict__ c1, const uint2 *__restrict__ c2, uint32_t m1, uint32_t m2,
                  const uint32_t *__restrict__ list, const uint32_t *__restrict__ seg,
                  const uint32_t *__restrict__ seg_hi, uint32_t n_tiles, uint32_t tiles2, double *__restrict__ out,
                  uint64_t out_stride, int accumulate) {
    constexpr int NT = T1 * T2, B = NT / 4, NW = NT / 32;
    __shared__ uint32_t q_idx[NT];
    __shared__ uint32_t warp_n[NW];
    __shared__ uint32_t sup[B][4];
    __shared__ double w1[B][T1], w2[B][T2];
    const uint32_t t = blockIdx.x % n_tiles, w = blockIdx.x / n_tiles;
    const uint32_t j1_0 = (t / tiles2) * T1, j2_0 = (t % tiles2) * T2;
    const uint32_t tx = threadIdx.x % T1, ty = threadIdx.x / T1;
    const uint32_t j1 = j1_0 + tx, j2 = j2_0 + ty;
    const bool mine = j1 <= m1 && j2 <= m2;
    double *dst = out + (uint64_t)w * out_stride + (uint64_t)j1 * (m2 + 1) + j2;
    double acc = accumulate && mine ? *dst : 0.0;
    const uint32_t g = list ? t : w;
    const uint32_t s = seg[g], e = seg_hi[g];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t base = s; base < e; base += NT) {
        const uint32_t i = base + threadIdx.x;
        uint32_t idx = 0;
        bool hit = false;
        if (i < e) {
            idx = list ? list[i] : i;
            uint32_t lo, hi;
            sfs_support(c1[idx], m1, lo, hi);
            hit = lo < j1_0 + T1 && hi >= j1_0;
            if (c2) {
                sfs_support(c2[idx], m2, lo, hi);
                hit = hit && lo < j2_0 + T2 && hi >= j2_0;
            }
        }
        const uint32_t ball = __ballot_sync(0xffffffffu, hit);
        if (!lane) warp_n[warp] = __popc(ball);
        __syncthreads();
        uint32_t before = 0, total = 0;
#pragma unroll
        for (int k = 0; k < NW; ++k) {
            before += k < (int)warp ? warp_n[k] : 0u;
            total += warp_n[k];
        }
        if (hit) q_idx[before + __popc(ball & ((1u << lane) - 1u))] = idx;
        __syncthreads();
        for (uint32_t k0 = 0; k0 < total; k0 += B) {
            const uint32_t nb = min((uint32_t)B, total - k0);
            if (threadIdx.x < 4 * nb) {
                const uint32_t q = threadIdx.x >> 2, role = threadIdx.x & 3;
                const bool second = role >> 1, up = !(role & 1);
                const uint32_t r = q_idx[k0 + q];
                const uint2 na = second ? (c2 ? c2[r] : make_uint2(0u, 0u)) : c1[r];
                const uint32_t m = second ? m2 : m1, t_lo = second ? j2_0 : j1_0;
                const uint32_t t_hi = t_lo + (second ? T2 : T1) - 1;
                double *wd = second ? w2[q] : w1[q];
                uint32_t lo, hi;
                sfs_support(na, m, lo, hi);
                if (up) {
                    sup[q][2 * second] = lo;
                    sup[q][2 * second + 1] = hi;
                }
                const uint32_t from = max(lo, t_lo), to = min(hi, t_hi);
                if (from <= to) {
                    if (lo == hi) {
                        if (up) wd[lo - t_lo] = 1.0;
                    } else {
                        sfs_walk(na.x, na.y, m, lo, hi, from, to, up, wd, t_lo);
                    }
                }
            }
            __syncthreads();
            if (mine)
                for (uint32_t q = 0; q < nb; ++q)
                    if (j1 >= sup[q][0] && j1 <= sup[q][1] && j2 >= sup[q][2] && j2 <= sup[q][3])
                        acc += w1[q][tx] * w2[q][ty];
            __syncthreads();
        }
    }
    if (mine) *dst = acc;
}

// ------------------------------------------------------------------------------------ joint incidences
// count [n]: tiles of the joint spectrum that row i touches
__global__ void __launch_bounds__(256)
fm_k_sfs_incidence_count(const uint2 *__restrict__ c1, const uint2 *__restrict__ c2, uint32_t n, uint32_t m1,
                         uint32_t m2, unsigned long long *__restrict__ count) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t lo1, hi1, lo2, hi2;
    sfs_support(c1[i], m1, lo1, hi1);
    sfs_support(c2[i], m2, lo2, hi2);
    count[i] = (unsigned long long)(hi1 / kSfsJointTile - lo1 / kSfsJointTile + 1) * (hi2 / kSfsJointTile - lo2 / kSfsJointTile + 1);
}

// (tile, row) incidences of rows [i0, i1), row i's from offset[i] - offset[i0]
__global__ void __launch_bounds__(256)
fm_k_sfs_incidence_emit(const uint2 *__restrict__ c1, const uint2 *__restrict__ c2, uint32_t i0, uint32_t i1,
                        uint32_t m1, uint32_t m2, uint32_t tiles2, const unsigned long long *__restrict__ offset,
                        uint32_t *__restrict__ keys, uint32_t *__restrict__ rows) {
    const uint32_t i = i0 + blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= i1) return;
    uint32_t lo1, hi1, lo2, hi2;
    sfs_support(c1[i], m1, lo1, hi1);
    sfs_support(c2[i], m2, lo2, hi2);
    uint64_t o = offset[i] - offset[i0];
    for (uint32_t a = lo1 / kSfsJointTile; a <= hi1 / kSfsJointTile; ++a)
        for (uint32_t b = lo2 / kSfsJointTile; b <= hi2 / kSfsJointTile; ++b, ++o) {
            keys[o] = a * tiles2 + b;
            rows[o] = i;
        }
}

// seg [t] = first incidence of tile t in the sorted keys [n] (seg [n_tiles] = n)
__global__ void __launch_bounds__(256)
fm_k_sfs_segments(const uint32_t *__restrict__ keys, uint64_t n, uint32_t n_tiles, uint32_t *__restrict__ seg) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t > n_tiles) return;
    uint64_t a = 0, b = n;
    while (a < b) {
        const uint64_t mid = (a + b) >> 1;
        if (keys[mid] < t) a = mid + 1;
        else b = mid;
    }
    seg[t] = (uint32_t)a;
}

}  // namespace fm
