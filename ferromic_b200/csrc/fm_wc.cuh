// fm_wc.cuh -- K4: Weir & Cockerham variance components from per-group allele/called counts.
//
// Mirrors calculate_fst_wc_at_site_with_membership (stats.rs:1814-2032),
// calculate_variance_components (stats.rs:2034-2127) and the region aggregation of
// calculate_overall_fst_wc (stats.rs:2145-2374) for biallelic matrices.
//
// Work decomposition: the host cuts every window (region) of sites at multiples of kWcSegSites of the site index.
//   * pairs (fm_k_wc_pairs_pc): one CTA task = (segment, chunk of 352 pair slots), walked in site order; a producer
//     warp stages the per-group counts and divides the per-group allele frequencies once per site, the pair warps
//     (lane = pair) add each pair's (a, b) site after site in REGISTERS;
//   * overall (fm_k_wc_overall): one warp per segment evaluates the all-population components with one site per
//     lane (groups in order, exactly as calculate_variance_components) and then adds the 32 site values in site
//     order;
//   * multi-allelic matrices (fm_k_wc_multi): one CTA per segment, pair warps + one overall warp.
// fm_k_wc_fold adds the segment partials of a window in segment order.  Cut points depend only
// on the site index, so the result does not depend on the grid, on how windows are batched into
// calls, or on how sites are sharded over GPUs (shards are aligned to kWcSegSites).
//
// Arithmetic: every FP64 expression keeps the reference's operation order.  Work that the
// reference repeats is shared without changing a single rounding: per-group allele frequencies
// are divided once per site (not once per pair), and the terms of a pair that depend only on the
// sample sizes (n_bar, c^2, the a-denominator, n_bar/(n_bar-1)) are evaluated once for both
// alleles.  A pair that is
// monomorphic at a site contributes exactly (+0, +0) in the reference (p_i = p_j = p_bar in
// {0, 1}), so its FP64 work is skipped.
#pragma once
#include "fm_device.cuh"
#include "fm_kernels.cuh"

namespace fm {

constexpr uint32_t kWcSegSites = 1024;   // segment granularity (== 32 batches)
constexpr uint32_t kWcMaxPairWarps = 11; // multi-allelic kernel: 352 pair threads per CTA (>= the 325 pairs of 26 populations)
constexpr uint32_t kWcMaxKP = 8;         // multi-allelic kernel: pairs per lane (template parameter KP <= this)

struct WcParams {
    const uint32_t *const *alt;  // [G + 1] device pointers, each [V]; index G = haplotypes with no group
    const uint32_t *const *cnt;  // [G + 1]
    const uint32_t *const *acount;  // multi-allelic: [G + 1] pointers to per-allele counts [V][A] (else nullptr)
    uint32_t A;                  // alleles per site slot (2 for biallelic, 2^NB for multi-allelic)
    uint32_t G, n_pairs;
    uint32_t n_pair_warps;            // pair warps per CTA (block = (n_pair_warps + 1) * 32 threads)
    const uint16_t *pair_i, *pair_j;  // [n_pairs], i < j in label order
    const uint32_t *seg_lo, *seg_hi;  // [n_seg] site ranges, walked in order by one CTA each
    uint32_t n_seg;
    uint32_t out_base;                // per-site outputs are indexed v - out_base
    // per-site outputs, any may be nullptr
    int32_t *site_state;
    double *site_a, *site_b;
    uint32_t *site_sizes;        // [n_sites][G]
    double *pair_a, *pair_b;     // [n_sites][n_pairs]; NaN when the pair has no data at the site
    // per-segment partials
    double *part_overall;        // [n_seg][2]            sum a, sum b
    uint32_t *part_counts;       // [n_seg]               sites with an estimate (!= InsufficientData)
    double *part_pair;           // [n_seg][n_pairs][2]
    uint32_t *part_pair_n;       // [n_seg][n_pairs]      informative sites per pair
};

// a / b given y = RN(1 / b): Markstein's correction applied twice.  q0 = a*y is within 1.5 ulp, one
// residual step makes it faithful, the second makes it the correctly rounded quotient (Markstein 1990; the
// only excluded divisors have an all-ones significand, which integers, half-integers and their squares below
// 2^52 never have).  tools/check_recip_div.c: 4e8 random cases, 0 differences from IEEE division.  The FP64
// pipe sees 5 operations instead of the ~25-instruction division sequence with its slow-path branch.
__device__ __forceinline__ double fm_div_recip(double a, double b, double y) {
    double q = a * y;
    double r = __fma_rn(-b, q, a);
    q = __fma_rn(r, y, q);
    r = __fma_rn(-b, q, a);
    return __fma_rn(r, y, q);
}

// a / b from y = RN(1 / b) with ONE residual correction, for divisors that are "small integers up to a power of
// two": b = n * 2^k with an integer 1 <= n < 2^40 (here n_i + n_j, half of it, half of it minus one, and
// (n_i + n_j)^2 / 2).  Proof of exactness: q0 = RN(a * y) is within 1.5 ulp of a / b, and the corrected value
// q0 + (a - b*q0) * y differs from a / b by at most 2^-53 * 1.5 ulp, so RN of it is RN(a / b) unless a / b lies
// within 3 * 2^-54 ulp of a rounding midpoint m.  But a - n * 2^k * m is a non-zero multiple of ulp(a / b) * 2^k / 2
// (a has 53 bits, m 54, and the exponents differ by at least log2 n), so |a / b - m| >= ulp / (2n) > 2^-41 ulp: no
// quotient by such a divisor comes that close to a midpoint.  (An arbitrary 53-bit divisor can come within 2^-54
// ulp -- the a-denominator 1 - c^2 therefore keeps the two-step fm_div_recip.)
__device__ __forceinline__ double fm_div_recip_int(double a, double b, double y) {
    const double q = a * y;
    const double r = __fma_rn(-b, q, a);
    return __fma_rn(r, y, q);
}

struct WcTables {            // indexed by an integer n = 0 .. n_max (n_max >= largest n_i + n_j of any pair)
    const double *inv_n;     // RN(1 / n)
    const double *inv_2nb2;  // RN(1 / (2 * (n/2) * (n/2))) = RN(2 / n^2): the c^2 divisor of a pair with n_i + n_j = n
    uint32_t n_max;
};


// RN(1 / b) for a normal b far from the exponent limits (here b = 1 - c^2 in (0, 1]): hardware seed
// (MUFU.RCP64H, ~23 bits), two Newton steps and one residual correction of the then faithful estimate.  Branch
// free; tests/test_gpu_wc_arith.py compares it with IEEE 1.0 / b over 2^24 divisors.  The one divisor shape the
// residual correction cannot round (Markstein) is an all-ones significand, e.g. 1 - 2^-53 -> 1.0 instead of
// 1 + 2^-52; the callers' divisors cannot take that form.
__device__ __forceinline__ double fm_recip_rn(double b) {
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(b));
    double e = __fma_rn(-b, y, 1.0);
    y = __fma_rn(y, e, y);
    e = __fma_rn(-b, y, 1.0);
    y = __fma_rn(y, e, y);
    e = __fma_rn(-b, y, 1.0);
    return __fma_rn(y, e, y);
}

// One (pair, site) evaluation of calculate_variance_components with r = 2 (stats.rs:2034-2127), summed over
// both alleles (stats.rs:1939-1983).  Only called for a pair that is polymorphic at the site, so both alleles
// are present among the samples (has0 && has1) and n_i + n_j >= 3.  Straight-line code: the two alleles (and,
// in the caller, SU sites) are independent dependency chains the FP64 pipe can interleave.
// vi / vj: (p0, p1, n, alt) of the two groups as doubles.
__device__ __forceinline__ void fm_wc_pair_site(const double4 vi, const double4 vj, uint32_t nsum, const WcTables &T,
                                                double &pa, double &pb) {
    const double n1 = vi.z, n2 = vj.z;
    const double nsd = n1 + n2;         // exact: integers
    const double n_bar = nsd / 2.0;     // exact
    const double nbm1 = n_bar - 1.0;    // exact
    const double r_nsd = __ldg(T.inv_n + nsum);
    const double r_nbar = 2.0 * r_nsd;                        // RN(1 / n_bar), exact scaling
    const double r_nbm1 = 2.0 * __ldg(T.inv_n + (nsum - 2));  // RN(1 / (n_bar - 1))
    // size-only terms.  Exact shortcuts (every intermediate is a small dyadic rational, nothing rounds):
    // n2 - n_bar == -(n1 - n_bar), so (n1 - n_bar)^2 + (n2 - n_bar)^2 == 2 d1^2; and 2 * n_bar * n_bar == nsd * n_bar.
    const double d1 = n1 - n_bar;
    const double ssd = 2.0 * (d1 * d1);
    const double c_squared = fm_div_recip_int(ssd, nsd * n_bar, __ldg(T.inv_2nb2 + nsum));
    const double aden = 1.0 - c_squared;   // c_squared / (r - 1) with r - 1 == 1
    // 1 - c^2 is 1 exactly or at most 1 - 1/(n_i + n_j)^2: never the all-ones significand fm_recip_rn excludes
    const double raden = fm_recip_rn(aden);
    const double ratio = fm_div_recip_int(n_bar, nbm1, r_nbm1);
    const double asd = vi.w + vj.w;     // exact
    // allele 0, then allele 1 (ascending order, stats.rs:1859)
    const double gp0 = fm_div_recip_int(nsd - asd, nsd, r_nsd), gp1 = fm_div_recip_int(asd, nsd, r_nsd);
    const double q10 = vi.x - gp0, q20 = vj.x - gp0, q11 = vi.y - gp1, q21 = vj.y - gp1;
    const double num0 = n1 * q10 * q10 + n2 * q20 * q20;  // 0.0 + (n1*q1)*q1, then + (n2*q2)*q2
    const double num1 = n1 * q11 * q11 + n2 * q21 * q21;
    const double s20 = fm_div_recip_int(num0, n_bar, r_nbar), s21 = fm_div_recip_int(num1, n_bar, r_nbar);
    // x = p(1 - p) - ((r - 1) / r) s^2 with (r - 1) / r == 0.5: halving is exact, so the fused form rounds once,
    // exactly where the reference's subtraction does
    const double x0 = __fma_rn(-0.5, s20, gp0 * (1.0 - gp0)), x1 = __fma_rn(-0.5, s21, gp1 * (1.0 - gp1));
    const double ta0 = fm_div_recip(s20 - fm_div_recip_int(x0, nbm1, r_nbm1), aden, raden);
    const double ta1 = fm_div_recip(s21 - fm_div_recip_int(x1, nbm1, r_nbm1), aden, raden);
    pa = ta0 + ta1;  // 0.0 + ta0 == ta0 up to the sign of a zero
    pb = ratio * x0 + ratio * x1;
}

// ---- K4 pairs, producer / consumer form.  The first round-2 version staged a 32-site batch with all threads of
// the CTA and paid three CTA barriers per batch (ncu: 0.8 of the 4.9 resident warps per scheduler parked at a
// barrier, FP64 pipe 61 % busy): the pair warps drift apart while they share the FP64 pipe and then wait for the
// slowest.  Here the last warp of the CTA is a PRODUCER and the other warps are pair warps (lane = pair) that never
// meet at a CTA barrier: the producer prefetches the raw counts of the sub-batch two steps ahead with 4-byte
// cp.async copies (no registers, no stall), derives the per-(site, group) allele frequencies of the current one
// (each divided once per site, not once per pair) and publishes the stage through an mbarrier; a pair warp waits for
// the stage's `full` barrier, adds its 32 pairs site after site -- every pair sum is accumulated sequentially in
// site order inside a segment, the association of the reference's `.sum()` (stats.rs:2288-2289) -- and releases the
// stage through its `empty` barrier.  kWcPcStages stages let the pair warps drift two sub-batches apart.
// 1M sites x 325 pairs: 3.2 -> 2.7 ms (B200).
constexpr uint32_t kWcPcSites = 16;   // sites per stage
constexpr uint32_t kWcPcStages = 4;
constexpr uint32_t kWcPcAhead = 2;    // sub-batches whose counts are in flight while one is being prepared
constexpr uint32_t kWcPcPairWarps = 11;

__host__ __device__ inline uint32_t fm_wc_pitch(uint32_t G) { return G | 1u; }  // odd row pitch: fewer bank conflicts
__host__ __device__ inline size_t fm_wc_stage_bytes(uint32_t G) {
    return (size_t)kWcPcSites * fm_wc_pitch(G) * (sizeof(double4) + sizeof(uint2));
}
__host__ __device__ inline size_t fm_wc_pc_smem(uint32_t G) { return kWcPcStages * fm_wc_stage_bytes(G) + 2 * kWcPcStages * 8 + 16; }

// walks the sub-batches of the CTA's tasks (task = (segment, chunk of pair slots), grid-strided) in order
struct WcCursor {
    uint32_t task, v, hi;
    __device__ __forceinline__ void open(const WcParams &P, uint32_t n_chunks, uint32_t n_tasks) {
        while (task < n_tasks) {
            const uint32_t si = task / n_chunks;
            v = P.seg_lo[si];
            hi = P.seg_hi[si];
            if (v < hi) return;
            task += gridDim.x;
        }
    }
    __device__ __forceinline__ void advance(const WcParams &P, uint32_t n_chunks, uint32_t n_tasks) {
        v += kWcPcSites;
        if (v >= hi) {
            task += gridDim.x;
            open(P, n_chunks, n_tasks);
        }
    }
};

template <int SU>
__global__ void __launch_bounds__((kWcPcPairWarps + 1) * 32, 2)
fm_k_wc_pairs_pc(const WcParams P, const WcTables T, uint32_t n_chunks) {
    extern __shared__ __align__(16) uint8_t wc_smem[];
    constexpr uint32_t FULL = 0xffffffffu;
    constexpr uint32_t NS = kWcPcStages, SB = kWcPcSites, NWC = kWcPcPairWarps;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t G = P.G, GP = fm_wc_pitch(P.G), NP = P.n_pairs;
    const size_t stage_bytes = fm_wc_stage_bytes(G);
    uint64_t *bars = reinterpret_cast<uint64_t *>(wc_smem + NS * stage_bytes);
    const uint32_t bar_full = fm_smem_u32(bars), bar_empty = bar_full + 8u * NS;
    const uint32_t n_tasks = P.n_seg * n_chunks;
    if (threadIdx.x == 0) {
        for (uint32_t s = 0; s < NS; ++s) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 32;" ::"r"(bar_full + 8u * s));
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar_empty + 8u * s), "r"(NWC));
        }
        fm_fence_mbar_init();
    }
    __syncthreads();
    auto stage_val = [&](uint32_t st) { return reinterpret_cast<double4 *>(wc_smem + st * stage_bytes); };
    auto stage_cnt = [&](uint32_t st) { return reinterpret_cast<uint2 *>(wc_smem + st * stage_bytes + (size_t)SB * GP * sizeof(double4)); };

    if (warp == NWC) {
        // ------------------------------------------------------------------ producer warp
        WcCursor ci{blockIdx.x, 0, 0}, cp{blockIdx.x, 0, 0};
        ci.open(P, n_chunks, n_tasks);
        cp.open(P, n_chunks, n_tasks);
        uint32_t n_issue = 0, n_proc = 0;
        auto issue = [&]() {  // raw counts of sub-batch ci -> stage n_issue % NS (asynchronous)
            if (ci.task < n_tasks) {
                const uint32_t st = n_issue % NS;
                if (n_issue >= NS) fm_mbar_wait(bar_empty + 8u * st, ((n_issue / NS) - 1u) & 1u);
                uint2 *cn = stage_cnt(st);
                const uint32_t nb = min(SB, ci.hi - ci.v);
                for (uint32_t i = lane; i < SB * G; i += 32) {  // 16 consecutive sites of one group per half-warp
                    const uint32_t g = i / SB, s = i % SB;
                    uint2 *dst = cn + s * GP + g;
                    if (s < nb) {
                        const uint32_t d = fm_smem_u32(dst);
                        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(P.alt[g] + ci.v + s) : "memory");
                        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d + 4u), "l"(P.cnt[g] + ci.v + s) : "memory");
                    } else {
                        *dst = make_uint2(0u, 0u);  // sites past the segment end: no data, never evaluated
                    }
                }
                ci.advance(P, n_chunks, n_tasks);
                ++n_issue;
            }
            asm volatile("cp.async.commit_group;" ::: "memory");  // one group per call, empty at the end of the walk
        };
        for (uint32_t k = 0; k < kWcPcAhead; ++k) issue();
        while (cp.task < n_tasks) {
            issue();
            asm volatile("cp.async.wait_group %0;" ::"n"(kWcPcAhead) : "memory");  // the counts of sub-batch n_proc landed
            __syncwarp();
            const uint32_t st = n_proc % NS;
            const uint2 *cn = stage_cnt(st);
            double4 *val = stage_val(st);
            for (uint32_t i = lane; i < SB * G; i += 32) {
                const uint32_t g = i / SB, s = i % SB;
                const uint2 c = cn[s * GP + g];
                double4 o = make_double4(0.0, 0.0, 0.0, 0.0);
                if (c.y > 0) {
                    const double nd = (double)c.y, ad = (double)c.x;
                    const double y = __ldg(T.inv_n + c.y);
                    o = make_double4(fm_div_recip_int((double)(c.y - c.x), nd, y), fm_div_recip_int(ad, nd, y), nd, ad);
                }
                val[s * GP + g] = o;
            }
            fm_mbar_arrive(bar_full + 8u * st);  // every producer lane: its stores (and landed copies) are released
            cp.advance(P, n_chunks, n_tasks);
            ++n_proc;
        }
        asm volatile("cp.async.wait_all;" ::: "memory");
        return;
    }

    // ---------------------------------------------------------------------- pair warps
    uint32_t n_cons = 0;
    for (uint32_t task = blockIdx.x; task < n_tasks; task += gridDim.x) {
        const uint32_t si = task / n_chunks, chunk = task - si * n_chunks;
        const uint32_t lo = P.seg_lo[si], hi = P.seg_hi[si];
        if (lo >= hi) continue;  // the producer skips empty segments too
        const uint32_t p = chunk * (NWC * 32) + warp * 32 + lane;
        const bool pvalid = p < NP;
        const uint32_t pi = pvalid ? __ldg(P.pair_i + p) : 0u, pj = pvalid ? __ldg(P.pair_j + p) : 0u;
        double acc_a = 0.0, acc_b = 0.0;
        uint32_t acc_n = 0;
        for (uint32_t v0 = lo; v0 < hi; v0 += SB, ++n_cons) {
            const uint32_t nb = min(SB, hi - v0);
            const uint32_t st = n_cons % NS;
            fm_mbar_wait(bar_full + 8u * st, (n_cons / NS) & 1u);
            const uint2 *cnts = stage_cnt(st);
            const double4 *val = stage_val(st);
            // pairwise components (r == 2), sites in order, SU at a time as independent dependency chains.  A group
            // with called samples implies an allele is present at the site (stats.rs:1826-1837), so the pair's own
            // counts decide everything (stats.rs:1950-1952).
            for (uint32_t s0 = 0; s0 < nb; s0 += SU) {
                double pa[SU], pb[SU];
                bool has[SU], poly[SU];
                uint32_t nsum[SU];
                bool any_poly = false;
#pragma unroll
                for (int t = 0; t < SU; ++t) {
                    const uint2 *sc = cnts + (s0 + t) * GP;  // s0 + t < SB; sites past nb hold zeros
                    const uint2 ci = sc[pi], cj = sc[pj];
                    has[t] = pvalid && ci.y > 0 && cj.y > 0;
                    const uint32_t asum = ci.x + cj.x;
                    nsum[t] = ci.y + cj.y;
                    // polymorphic in this pair and n_bar - 1 >= 1e-9 (anything else adds exactly +0)
                    poly[t] = has[t] && asum != 0 && asum != nsum[t] && nsum[t] > 2;
                    any_poly = any_poly || poly[t];
                    pa[t] = 0.0;
                    pb[t] = 0.0;
                }
                if (__any_sync(FULL, any_poly)) {
                    double ea[SU], eb[SU];
#pragma unroll
                    for (int t = 0; t < SU; ++t) {
                        // a lane whose pair is not polymorphic here runs on whatever the stage holds (only the table
                        // index is clamped) and drops the result: it would have waited for its neighbours anyway
                        const double4 *sv = val + (s0 + t) * GP;
                        fm_wc_pair_site(sv[pi], sv[pj], poly[t] ? nsum[t] : 4u, T, ea[t], eb[t]);
                    }
#pragma unroll
                    for (int t = 0; t < SU; ++t) {
                        pa[t] = poly[t] ? ea[t] : 0.0;
                        pb[t] = poly[t] ? eb[t] : 0.0;
                    }
                }
#pragma unroll
                for (int t = 0; t < SU; ++t) {
                    if (has[t]) {  // site order: stats.rs:2288-2289
                        acc_a += pa[t];
                        acc_b += pb[t];
                        acc_n += 1;
                    }
                    if (P.pair_a && pvalid && s0 + t < nb) {
                        const size_t o = (size_t)(v0 + s0 + t - P.out_base) * NP + p;
                        P.pair_a[o] = has[t] ? pa[t] : fm_nan();
                        P.pair_b[o] = has[t] ? pb[t] : fm_nan();
                    }
                }
            }
            __syncwarp();
            if (lane == 0) fm_mbar_arrive(bar_empty + 8u * st);
        }
        if (pvalid) {
            P.part_pair[((size_t)si * NP + p) * 2] = acc_a;
            P.part_pair[((size_t)si * NP + p) * 2 + 1] = acc_b;
            P.part_pair_n[(size_t)si * NP + p] = acc_n;
        }
    }
}

// test hook: y[i] = fm_recip_rn(b[i]) and q[i] = fm_div_recip(a[i], b[i], RN(1 / b[i]))
__global__ void fm_k_wc_arith_probe(const double *__restrict__ a, const double *__restrict__ b, double *__restrict__ y,
                                    double *__restrict__ q, double *__restrict__ q3, uint64_t n) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        y[i] = fm_recip_rn(b[i]);
        q[i] = fm_div_recip(a[i], b[i], 1.0 / b[i]);
        if (q3) q3[i] = fm_div_recip_int(a[i], b[i], 1.0 / b[i]);
    }
}

// ---- K4 overall: the all-population components, one WARP per segment, one site per lane (groups in order,
// exactly as calculate_variance_components, stats.rs:2034-2127, over the groups with data: stats.rs:1907-1918),
// then the 32 site values are added in site order (stats.rs:2172-2184, 2222-2229).  Counts come straight from
// the per-group arrays (coalesced: lane = site).
__global__ void __launch_bounds__(128)
fm_k_wc_overall(const WcParams P, const WcTables T) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t GW = (gridDim.x * blockDim.x) >> 5;
    const uint32_t G = P.G, G1 = P.G + 1;
    for (uint32_t si = gw; si < P.n_seg; si += GW) {
        const uint32_t lo = P.seg_lo[si], hi = P.seg_hi[si];
        double sum_a = 0.0, sum_b = 0.0;  // identical in every lane
        uint32_t n_informative = 0;
        for (uint32_t v0 = lo; v0 < hi; v0 += 32) {
            const uint32_t nb = min(32u, hi - v0);
            double site_a = 0.0, site_b = 0.0;
            int state = 3;  // InsufficientDataForEstimation: no allele at all at this site
            bool any = false;
            if (lane < nb) {
                const uint32_t v = v0 + lane;
                uint32_t t_alt = 0, t_n = 0, m_alt = 0, m_n = 0, m_r = 0;
                for (uint32_t g = 0; g < G1; ++g) {
                    const uint32_t a = __ldg(P.alt[g] + v), n = __ldg(P.cnt[g] + v);
                    t_alt += a;
                    t_n += n;
                    if (g < G && n > 0) {
                        m_alt += a;
                        m_n += n;
                        m_r += 1;
                    }
                }
                const bool has0 = t_n > t_alt, has1 = t_alt > 0;
                any = has0 || has1;  // pop_sizes_populated (stats.rs:1919-1923, 1987)
                if (any && m_r >= 2) {  // fewer than two groups with data: no allele contributes
                    const double r = (double)m_r;
                    const double n_bar = (double)m_n / r;
                    if (!((n_bar - 1.0) < 1e-9)) {
                        const double gp0 = (double)(m_n - m_alt) / (double)m_n;
                        const double gp1 = (double)m_alt / (double)m_n;
                        double ssd = 0.0, ns0 = 0.0, ns1 = 0.0;  // sums in group order
                        for (uint32_t g = 0; g < G; ++g) {
                            const uint32_t n = __ldg(P.cnt[g] + v);
                            if (n > 0) {
                                const uint32_t a = __ldg(P.alt[g] + v);
                                const double nd = (double)n;
                                const double d = nd - n_bar;
                                ssd += d * d;
                                const double y = __ldg(T.inv_n + n);
                                const double f0 = fm_div_recip_int((double)(n - a), nd, y), f1 = fm_div_recip_int((double)a, nd, y);
                                const double q0 = f0 - gp0, q1 = f1 - gp1;
                                ns0 += nd * q0 * q0;
                                ns1 += nd * q1 * q1;
                            }
                        }
                        const double c_squared = ssd / (r * n_bar * n_bar);
                        const double a_den = 1.0 - (c_squared / (r - 1.0));
                        const double nb_ratio = n_bar / (n_bar - 1.0);
                        const bool s_ok = (r - 1.0) > 1e-9 && n_bar > 1e-9;
                        // sum over alleles in ascending order: allele 0 first (stats.rs:1859, 1939-1940)
                        if (has0) {
                            const double s2 = s_ok ? ns0 / ((r - 1.0) * n_bar) : 0.0;
                            const double x = gp0 * (1.0 - gp0) - ((r - 1.0) / r) * s2;
                            site_a += (s2 - (x / (n_bar - 1.0))) / a_den;
                            site_b += nb_ratio * x;
                        }
                        if (has1) {
                            const double s2 = s_ok ? ns1 / ((r - 1.0) * n_bar) : 0.0;
                            const double x = gp1 * (1.0 - gp1) - ((r - 1.0) / r) * s2;
                            site_a += (s2 - (x / (n_bar - 1.0))) / a_den;
                            site_b += nb_ratio * x;
                        }
                    }
                }
                if (any) state = fm_fst_state(site_a, site_b);
                const uint32_t o = v - P.out_base;
                if (P.site_state) P.site_state[o] = state;
                if (P.site_a) P.site_a[o] = site_a;
                if (P.site_b) P.site_b[o] = site_b;
                if (P.site_sizes)
                    for (uint32_t g = 0; g < G; ++g) P.site_sizes[(size_t)o * G + g] = any ? __ldg(P.cnt[g] + v) : 0u;
            }
            const uint32_t any_mask = __ballot_sync(0xffffffffu, any);
            for (uint32_t s = 0; s < nb; ++s) {
                const double a_s = __shfl_sync(0xffffffffu, site_a, s);
                const double b_s = __shfl_sync(0xffffffffu, site_b, s);
                if ((any_mask >> s) & 1u) {
                    sum_a += a_s;
                    sum_b += b_s;
                    ++n_informative;
                }
            }
        }
        if (lane == 0) {
            P.part_overall[2 * (size_t)si] = sum_a;
            P.part_overall[2 * (size_t)si + 1] = sum_b;
            P.part_counts[si] = n_informative;
        }
    }
}

// Multi-allelic variant (max_allele 2..15): same decomposition, with the reference's loop over
// every allele present at the site (stats.rs:1849-1859, 1939-1983) instead of the two alleles of
// a biallelic site.  An allele that is absent from a pair, or fixed in it, contributes exactly
// (+0, +0) and is skipped.
__host__ __device__ inline size_t fm_wc_multi_cta_smem(uint32_t G, uint32_t A) {
    // freq [32][G][A] f64 | cn [32][G+1] u32 | ca [32][G+1][A] u32 | info [32] u32
    return (size_t)32 * G * A * 8 + (size_t)32 * (G + 1) * 4 + (size_t)32 * (G + 1) * A * 4 + 32 * 4 + 16;
}

template <int KP>
__global__ void __launch_bounds__((kWcMaxPairWarps + 1) * 32, 1)
fm_k_wc_multi(const WcParams P) {
    extern __shared__ __align__(16) uint8_t wc_smem[];
    const uint32_t tid = threadIdx.x, nt = blockDim.x;
    const uint32_t lane = tid & 31, warp = tid >> 5;
    const uint32_t G = P.G, G1 = P.G + 1, NP = P.n_pairs, A = P.A;
    const uint32_t NW = P.n_pair_warps;
    double *freq = reinterpret_cast<double *>(wc_smem);                          // [32][G][A]
    uint32_t *cn = reinterpret_cast<uint32_t *>(freq + (size_t)32 * G * A);      // [32][G1] called
    uint32_t *ca = cn + (size_t)32 * G1;                                         // [32][G1][A] allele counts
    uint32_t *info = ca + (size_t)32 * G1 * A;                                   // [32] mask of alleles present
    const bool overall_warp = warp == NW;
    uint32_t pi[KP], pj[KP];
    bool pvalid[KP];
#pragma unroll
    for (int k = 0; k < KP; ++k) {
        const uint32_t p = warp * 32 + lane + (uint32_t)k * NW * 32;
        pvalid[k] = !overall_warp && p < NP;
        pi[k] = pvalid[k] ? __ldg(P.pair_i + p) : 0u;
        pj[k] = pvalid[k] ? __ldg(P.pair_j + p) : 0u;
    }
    for (uint32_t si = blockIdx.x; si < P.n_seg; si += gridDim.x) {
        const uint32_t lo = P.seg_lo[si], hi = P.seg_hi[si];
        double acc_a[KP], acc_b[KP];
        uint32_t acc_n[KP];
#pragma unroll
        for (int k = 0; k < KP; ++k) {
            acc_a[k] = 0.0;
            acc_b[k] = 0.0;
            acc_n[k] = 0;
        }
        double sum_a = 0.0, sum_b = 0.0;
        uint32_t n_informative = 0;
        for (uint32_t v0 = lo; v0 < hi; v0 += 32) {
            const uint32_t nb = min(32u, hi - v0);
            __syncthreads();
            for (uint32_t g = warp; g < G1; g += (nt >> 5))
                if (lane < nb) {
                    cn[lane * G1 + g] = __ldg(P.cnt[g] + v0 + lane);
                    const uint32_t *src = P.acount[g] + (size_t)(v0 + lane) * A;
                    for (uint32_t a = 0; a < A; ++a) ca[(lane * G1 + g) * A + a] = __ldg(src + a);
                }
            __syncthreads();
            for (uint32_t i = tid; i < nb * G * A; i += nt) {
                const uint32_t s = i / (G * A), r = i - s * G * A, g = r / A, a = r - g * A;
                const uint32_t n = cn[s * G1 + g];
                if (n > 0) freq[(s * G + g) * A + a] = (double)ca[(s * G1 + g) * A + a] / (double)n;
            }
            if (warp == 0 && lane < nb) {  // alleles present over ALL samples (stats.rs:1826-1837)
                uint32_t mask = 0;
                for (uint32_t a = 0; a < A; ++a) {
                    uint32_t t = 0;
                    for (uint32_t g = 0; g < G1; ++g) t += ca[(lane * G1 + g) * A + a];
                    if (t) mask |= 1u << a;
                }
                info[lane] = mask;
            }
            __syncthreads();
            if (overall_warp) {
                double site_a = 0.0, site_b = 0.0;
                int state = 3;
                bool any = false;
                if (lane < nb) {
                    const uint32_t *sn = cn + lane * G1;
                    const uint32_t *sa = ca + (size_t)lane * G1 * A;
                    const double *fr = freq + (size_t)lane * G * A;
                    const uint32_t present = info[lane];
                    any = present != 0;
                    uint32_t m_n = 0, m_r = 0;
                    for (uint32_t g = 0; g < G; ++g)
                        if (sn[g] > 0) {
                            m_n += sn[g];
                            m_r += 1;
                        }
                    if (any && m_r >= 2) {
                        const double r = (double)m_r;
                        const double n_bar = (double)m_n / r;
                        if (!((n_bar - 1.0) < 1e-9)) {
                            double ssd = 0.0;
                            for (uint32_t g = 0; g < G; ++g)
                                if (sn[g] > 0) {
                                    const double d = (double)sn[g] - n_bar;
                                    ssd += d * d;
                                }
                            const double c_squared = ssd / (r * n_bar * n_bar);
                            const double a_den = 1.0 - (c_squared / (r - 1.0));
                            const double nb_ratio = n_bar / (n_bar - 1.0);
                            const bool s_ok = (r - 1.0) > 1e-9 && n_bar > 1e-9;
                            for (uint32_t a = 0; a < A; ++a) {  // ascending allele order (stats.rs:1859)
                                if (!((present >> a) & 1u)) continue;
                                uint32_t m_t = 0;
                                for (uint32_t g = 0; g < G; ++g)
                                    if (sn[g] > 0) m_t += sa[g * A + a];
                                const double gp = (double)m_t / (double)m_n;
                                double ns = 0.0;
                                for (uint32_t g = 0; g < G; ++g)
                                    if (sn[g] > 0) {
                                        const double q = fr[g * A + a] - gp;
                                        ns += (double)sn[g] * q * q;
                                    }
                                const double s2 = s_ok ? ns / ((r - 1.0) * n_bar) : 0.0;
                                const double x = gp * (1.0 - gp) - ((r - 1.0) / r) * s2;
                                site_a += (s2 - (x / (n_bar - 1.0))) / a_den;
                                site_b += nb_ratio * x;
                            }
                        }
                    }
                    if (any) state = fm_fst_state(site_a, site_b);
                    const uint32_t o = v0 + lane - P.out_base;
                    if (P.site_state) P.site_state[o] = state;
                    if (P.site_a) P.site_a[o] = site_a;
                    if (P.site_b) P.site_b[o] = site_b;
                    if (P.site_sizes)
                        for (uint32_t g = 0; g < G; ++g) P.site_sizes[(size_t)o * G + g] = any ? sn[g] : 0u;
                }
                const uint32_t any_mask = __ballot_sync(0xffffffffu, any);
                for (uint32_t s = 0; s < nb; ++s) {
                    const double a_s = __shfl_sync(0xffffffffu, site_a, s);
                    const double b_s = __shfl_sync(0xffffffffu, site_b, s);
                    if ((any_mask >> s) & 1u) {
                        sum_a += a_s;
                        sum_b += b_s;
                        ++n_informative;
                    }
                }
            } else {
                for (uint32_t s = 0; s < nb; ++s) {
                    const uint32_t *sn = cn + s * G1;
                    const uint32_t *sa = ca + (size_t)s * G1 * A;
                    const double *fr = freq + (size_t)s * G * A;
                    const uint32_t present = info[s];
                    const bool any = present != 0;
#pragma unroll
                    for (int k = 0; k < KP; ++k) {
                        if (!pvalid[k]) continue;
                        const uint32_t i = pi[k], j = pj[k];
                        const uint32_t ni = sn[i], nj = sn[j];
                        double pa = 0.0, pb = 0.0;
                        const bool has = any && ni > 0 && nj > 0;
                        if (has) {
                            const uint32_t nsum = ni + nj;
                            const double n1 = (double)ni, n2 = (double)nj, nsd = (double)nsum;
                            const double n_bar = nsd / 2.0;
                            if (!((n_bar - 1.0) < 1e-9)) {
                                const double d1 = n1 - n_bar, d2 = n2 - n_bar;
                                double ssd = 0.0;
                                ssd += d1 * d1;
                                ssd += d2 * d2;
                                const double c_squared = ssd / (2.0 * n_bar * n_bar);
                                const double a_den = 1.0 - (c_squared / 1.0);
                                const double nb_ratio = n_bar / (n_bar - 1.0);
                                for (uint32_t a = 0; a < A; ++a) {
                                    if (!((present >> a) & 1u)) continue;
                                    const uint32_t asum = sa[i * A + a] + sa[j * A + a];
                                    if (asum == 0 || asum == nsum) continue;  // exactly (+0, +0)
                                    const double gp = (double)asum / nsd;
                                    const double q1 = fr[i * A + a] - gp, q2 = fr[j * A + a] - gp;
                                    double num = 0.0;
                                    num += n1 * q1 * q1;
                                    num += n2 * q2 * q2;
                                    const double s2 = num / (1.0 * n_bar);
                                    const double x = gp * (1.0 - gp) - (1.0 / 2.0) * s2;
                                    pa += (s2 - (x / (n_bar - 1.0))) / a_den;
                                    pb += nb_ratio * x;
                                }
                            }
                            acc_a[k] += pa;
                            acc_b[k] += pb;
                            acc_n[k] += 1;
                        }
                        if (P.pair_a) {
                            const uint32_t p = warp * 32 + lane + (uint32_t)k * NW * 32;
                            const size_t o = (size_t)(v0 + s - P.out_base) * NP + p;
                            P.pair_a[o] = has ? pa : fm_nan();
                            P.pair_b[o] = has ? pb : fm_nan();
                        }
                    }
                }
            }
        }
        if (overall_warp) {
            if (lane == 0) {
                P.part_overall[2 * (size_t)si] = sum_a;
                P.part_overall[2 * (size_t)si + 1] = sum_b;
                P.part_counts[si] = n_informative;
            }
        } else {
#pragma unroll
            for (int k = 0; k < KP; ++k) {
                if (!pvalid[k]) continue;
                const uint32_t p = warp * 32 + lane + (uint32_t)k * NW * 32;
                P.part_pair[((size_t)si * NP + p) * 2] = acc_a[k];
                P.part_pair[((size_t)si * NP + p) * 2 + 1] = acc_b[k];
                P.part_pair_n[(size_t)si * NP + p] = acc_n[k];
            }
        }
    }
}

// Window totals: window w owns segments [wseg[w], wseg[w+1]).  Fixed association: the window's segments are taken
// in chunks of kWcFoldChunk (counted from the window's first segment); a chunk is added in segment order, the chunk
// sums are added in chunk order.  One CTA per (window, block of 32 slots): slot p < n_pairs is a pair, p == n_pairs
// the overall components; lanes run over p, so the segment rows are read coalesced.  The warps of the CTA take
// consecutive chunks (all 3 * kWcFoldChunk loads of a chunk issued before the first add), warp 0 then adds the
// round's chunk sums in chunk order.  (The first version walked all segments with one thread per slot: 326 threads,
// 0.46 ms for the 977 segments of a 1M-site window -- 13 % of the W&C call.)
constexpr uint32_t kWcFoldChunk = 16;
constexpr uint32_t kWcFoldMaxWarps = 16;

__global__ void __launch_bounds__(kWcFoldMaxWarps * 32)
fm_k_wc_fold(const double *__restrict__ part_overall, const uint32_t *__restrict__ part_counts,
             const double *__restrict__ part_pair, const uint32_t *__restrict__ part_pair_n,
             const uint32_t *__restrict__ wseg, uint32_t n_windows, uint32_t n_pairs, uint32_t n_pb,
             double *__restrict__ out_overall /*[n_w][2]*/, uint64_t *__restrict__ out_sites /*[n_w]*/,
             double *__restrict__ out_pair /*[n_w][n_pairs][2]*/, uint64_t *__restrict__ out_pair_n) {
    __shared__ double sh_a[kWcFoldMaxWarps][32], sh_b[kWcFoldMaxWarps][32];
    __shared__ uint64_t sh_n[kWcFoldMaxWarps][32];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5, NW = blockDim.x >> 5;
    for (uint32_t unit = blockIdx.x; unit < n_windows * n_pb; unit += gridDim.x) {
        const uint32_t w = unit / n_pb, p = (unit - w * n_pb) * 32 + lane;
        const uint32_t s0 = wseg[w], s1 = wseg[w + 1];
        const bool live = p <= n_pairs, ov = p == n_pairs;
        const double *pa = ov ? part_overall : part_pair + 2 * (size_t)p;
        const uint32_t *pn = ov ? part_counts : part_pair_n + p;
        const size_t stride = ov ? 1 : n_pairs;  // segment stride in (a, b) pairs / counts
        double a = 0.0, b = 0.0;  // running sums (warp 0)
        uint64_t n = 0;
        const uint32_t n_chunks = (s1 - s0 + kWcFoldChunk - 1) / kWcFoldChunk;
        for (uint32_t r0 = 0; r0 < n_chunks; r0 += NW) {
            const uint32_t c = r0 + warp;
            if (c < n_chunks) {
                const uint32_t c0 = s0 + c * kWcFoldChunk;
                double xa[kWcFoldChunk], xb[kWcFoldChunk];
                uint32_t xn[kWcFoldChunk];
#pragma unroll
                for (uint32_t i = 0; i < kWcFoldChunk; ++i) {
                    const bool in = live && c0 + i < s1;
                    const size_t o = (size_t)(in ? c0 + i : s0) * stride;
                    xa[i] = in ? pa[2 * o] : 0.0;
                    xb[i] = in ? pa[2 * o + 1] : 0.0;
                    xn[i] = in ? pn[o] : 0u;
                }
                double ca = 0.0, cb = 0.0;
                uint64_t cn = 0;
#pragma unroll
                for (uint32_t i = 0; i < kWcFoldChunk; ++i) {
                    if (c0 + i < s1) {
                        ca += xa[i];
                        cb += xb[i];
                        cn += xn[i];
                    }
                }
                sh_a[warp][lane] = ca;
                sh_b[warp][lane] = cb;
                sh_n[warp][lane] = cn;
            }
            __syncthreads();
            if (warp == 0) {
                const uint32_t m = min(NW, n_chunks - r0);
                for (uint32_t k = 0; k < m; ++k) {
                    a += sh_a[k][lane];
                    b += sh_b[k][lane];
                    n += sh_n[k][lane];
                }
            }
            __syncthreads();
        }
        if (warp == 0 && live) {
            if (ov) {
                out_overall[2 * (size_t)w] = a;
                out_overall[2 * (size_t)w + 1] = b;
                out_sites[w] = n;
            } else {
                const size_t o = (size_t)w * n_pairs + p;
                out_pair[2 * o] = a;
                out_pair[2 * o + 1] = b;
                out_pair_n[o] = n;
            }
        }
    }
}

}  // namespace fm
