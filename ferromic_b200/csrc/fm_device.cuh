// fm_device.cuh -- PTX helpers (TMA bulk copy + mbarrier) and the per-site FP64 estimator
// formulas.  Every formula keeps the reference's operation order (src/stats.rs, cited per
// function); the translation unit is compiled with -fmad=false so nothing is contracted.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define FM_FST_EPSILON 1e-12 /* stats.rs:26 */

// ---------------------------------------------------------------------------------- PTX
__device__ __forceinline__ uint32_t fm_smem_u32(const void *p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void fm_mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(fm_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fm_fence_mbar_init() {
    // make the initialised barriers visible to the async (TMA) proxy
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void fm_mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(fm_smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
// 1-D TMA bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP).
__device__ __forceinline__ void fm_bulk_g2s(void *dst, const void *src, uint32_t bytes,
                                            uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
            "r"(fm_smem_u32(dst)),
        "l"(src), "r"(bytes), "r"(fm_smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ bool fm_mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(fm_smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void fm_mbar_wait(uint64_t *bar, uint32_t parity) {
    while (!fm_mbar_try_wait(bar, parity)) {
    }
}
// the same wait and a plain arrival, on a shared-memory address (fm_smem_u32 of the barrier)
__device__ __forceinline__ void fm_mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void fm_mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t fm_lds32(uint32_t saddr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(saddr));
    return v;
}
__device__ __forceinline__ uint4 fm_lds128(uint32_t saddr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(saddr));
    return v;
}
__device__ __forceinline__ uint32_t fm_popc4(const uint4 &v) {
    return __popc(v.x) + __popc(v.y) + __popc(v.z) + __popc(v.w);
}

// ---------------------------------------------------------------------------------- math
#define FM_HD __host__ __device__ __forceinline__

FM_HD double fm_nan() {
#ifdef __CUDA_ARCH__
    return __longlong_as_double(0x7ff8000000000000LL);
#else
    return __builtin_nan("");
#endif
}

// dense_pi_from_counts (stats.rs:1700-1709)
FM_HD bool fm_pi_dense_counts(uint32_t total_called, uint32_t alt_count, double &out) {
    if (total_called < 2) return false;
    double n = (double)total_called;
    double alt = (double)alt_count;
    double ref_count = (double)(total_called - alt_count);
    double sum_sq = ref_count * ref_count + alt * alt;
    out = n / (n - 1.0) * (1.0 - sum_sq / (n * n));
    return true;
}
// no-bitmap biallelic form (stats.rs:4490-4507 and 3223-3256): exact 0 when alt in {0,n}
FM_HD bool fm_pi_dense_nomissing(uint32_t total, uint32_t alt, double &out) {
    if (total < 2) return false;
    if (alt == 0 || alt == total) {
        out = 0.0;
        return true;
    }
    double n = (double)total;
    double scale = n / (n - 1.0);
    double inv_n_sq = 1.0 / (n * n);
    double alt_f = (double)alt;
    double ref_f = (double)(total - alt);
    double sum_sq = ref_f * ref_f + alt_f * alt_f;
    out = scale * (1.0 - sum_sq * inv_n_sq);
    return true;
}
// pi_from_components (stats.rs:2723-2733) with sum_counts_sq = ref^2 + alt^2 (exact integers)
FM_HD bool fm_pi_components(uint32_t total_called, uint32_t alt_count, double &out) {
    if (total_called < 2) return false;
    double r = (double)(total_called - alt_count), a = (double)alt_count;
    double sum_counts_sq = r * r + a * a;
    double n = (double)total_called;
    double inv_n = 1.0 / n;
    double sum_p2 = sum_counts_sq * inv_n * inv_n;
    out = n / (n - 1.0) * (1.0 - sum_p2);
    return true;
}
#define FM_PIFORM_COUNTS 0
#define FM_PIFORM_NOMISSING 1
#define FM_PIFORM_COMPONENTS 2
FM_HD bool fm_pi_form(int form, uint32_t n, uint32_t alt, double &out) {
    if (form == FM_PIFORM_COUNTS) return fm_pi_dense_counts(n, alt, out);
    if (form == FM_PIFORM_NOMISSING) return fm_pi_dense_nomissing(n, alt, out);
    return fm_pi_components(n, alt, out);
}

// dense_dxy_from_biallelic_counts (stats.rs:1712-1733)
FM_HD bool fm_dxy_dense_biallelic(uint32_t n1, uint32_t alt1, uint32_t n2, uint32_t alt2,
                                  double &out) {
    if (n1 == 0 || n2 == 0) return false;
    double n1_f = (double)n1, n2_f = (double)n2;
    double alt1_f = (double)alt1 / n1_f;
    double alt2_f = (double)alt2 / n2_f;
    double ref1 = 1.0 - alt1_f, ref2 = 1.0 - alt2_f;
    double dot = ref1 * ref2 + alt1_f * alt2_f;
    if (dot < 0.0) dot = 0.0;
    double dxy = 1.0 - dot;
    if (dxy < 0.0)
        dxy = 0.0;
    else if (dxy > 1.0)
        dxy = 1.0;
    out = dxy;
    return true;
}
// dxy_from_counts (stats.rs:2907-2935) == the dot form of calculate_dxy_dense (:2557-2591)
FM_HD bool fm_dxy_dot(uint32_t n1, uint32_t alt1, uint32_t n2, uint32_t alt2, double &out) {
    if (n1 == 0 || n2 == 0) return false;
    double inv1 = 1.0 / (double)n1, inv2 = 1.0 / (double)n2;
    uint32_t r1 = n1 - alt1, r2 = n2 - alt2;
    double dot = 0.0;
    if (r1 != 0 && r2 != 0) dot += ((double)r1 * inv1) * ((double)r2 * inv2);
    if (alt1 != 0 && alt2 != 0) dot += ((double)alt1 * inv1) * ((double)alt2 * inv2);
    double dxy = 1.0 - dot;
    dxy = dxy > 0.0 ? dxy : 0.0; /* .max(0.0) */
    dxy = dxy < 1.0 ? dxy : 1.0; /* .min(1.0) */
    out = dxy;
    return true;
}
// summaries form (stats.rs:1578-1588): integer numerator
FM_HD bool fm_dxy_summaries(uint32_t n1, uint32_t alt1, uint32_t n2, uint32_t alt2, double &out) {
    if (n1 == 0 || n2 == 0) return false;
    uint64_t r1 = n1 - alt1, r2 = n2 - alt2;
    double denom_pairs = (double)((uint64_t)n1 * (uint64_t)n2);
    double dxy = (double)((uint64_t)alt1 * r2 + r1 * (uint64_t)alt2) / denom_pairs;
    if (dxy < 0.0)
        dxy = 0.0;
    else if (dxy > 1.0)
        dxy = 1.0;
    out = dxy;
    return true;
}
// pi form inside aggregate_hudson_components_from_summaries (stats.rs:1595-1606)
FM_HD double fm_pi_summaries(uint32_t n, uint32_t alt) {
    double denom = (double)((uint64_t)n * (uint64_t)(n - 1));
    uint32_t ref = n - alt;
    return denom > 0.0 ? 2.0 * (double)alt * (double)ref / denom : 0.0;
}

struct fm_hudson_vals {
    double dxy, pi1, pi2, fst, num, den; // NaN == None
};

// (dxy, pi1, pi2) -> (fst, num, den): stats.rs:1736-1757 / 2984-3001 / 3143-3158
FM_HD void fm_hudson_components(bool has_d, double d, bool has1, double p1, bool has2, double p2,
                                fm_hudson_vals &o) {
    const double NaN = fm_nan();
    o.dxy = has_d ? d : NaN;
    o.pi1 = has1 ? p1 : NaN;
    o.pi2 = has2 ? p2 : NaN;
    o.fst = NaN;
    o.num = NaN;
    o.den = NaN;
    if (has_d && has1 && has2) {
        if (d > FM_FST_EPSILON) {
            double nm = d - 0.5 * (p1 + p2);
            o.fst = nm / d;
            o.num = nm;
            o.den = d;
        } else {
            double pi_avg = 0.5 * (p1 + p2);
            if (fabs(pi_avg) <= FM_FST_EPSILON) {
                o.num = 0.0;
                o.den = 0.0;
            }
        }
    }
}

#define FM_HV_DENSE_MISSING 0   /* dense_hudson_sites_biallelic, Some(bits) arm (stats.rs:3192-3217) */
#define FM_HV_DENSE_NOMISSING 1 /* same, None arm (stats.rs:3218-3274) */
#define FM_HV_SPARSE 2          /* hudson_site_from_variant (stats.rs:2969-3014) */
FM_HD void fm_hudson_site(int variant, uint32_t n1, uint32_t a1, uint32_t n2, uint32_t a2,
                          fm_hudson_vals &o) {
    double d = 0.0, p1 = 0.0, p2 = 0.0;
    bool has_d, has1, has2;
    if (variant == FM_HV_SPARSE) {
        has1 = fm_pi_components(n1, a1, p1);
        has2 = fm_pi_components(n2, a2, p2);
        has_d = fm_dxy_dot(n1, a1, n2, a2, d);
    } else if (variant == FM_HV_DENSE_NOMISSING) {
        has1 = fm_pi_dense_nomissing(n1, a1, p1);
        has2 = fm_pi_dense_nomissing(n2, a2, p2);
        has_d = fm_dxy_dense_biallelic(n1, a1, n2, a2, d);
    } else {
        has1 = fm_pi_dense_counts(n1, a1, p1);
        has2 = fm_pi_dense_counts(n2, a2, p2);
        has_d = fm_dxy_dense_biallelic(n1, a1, n2, a2, d);
    }
    fm_hudson_components(has_d, d, has1, p1, has2, p2, o);
}

// calculate_variance_components (stats.rs:2034-2127) for r == 2 (pairwise W&C)
FM_HD void fm_wc_pair_components(uint32_t n1, uint32_t t1, uint32_t n2, uint32_t t2, double &a,
                                 double &b) {
    const double r = 2.0;
    double n_bar = (double)((uint64_t)n1 + (uint64_t)n2) / r;
    if ((n_bar - 1.0) < 1e-9) {
        a = 0.0;
        b = 0.0;
        return;
    }
    double p1 = (double)t1 / (double)n1, p2 = (double)t2 / (double)n2;
    double global_p = (double)((uint64_t)t1 + (uint64_t)t2) / (double)((uint64_t)n1 + (uint64_t)n2);
    double d1 = (double)n1 - n_bar, d2 = (double)n2 - n_bar;
    double sum_sq_diff_n = 0.0;
    sum_sq_diff_n += d1 * d1;
    sum_sq_diff_n += d2 * d2;
    double c_squared = sum_sq_diff_n / (r * n_bar * n_bar);
    double q1 = p1 - global_p, q2 = p2 - global_p;
    double numerator_s_squared = 0.0;
    numerator_s_squared += (double)n1 * q1 * q1;
    numerator_s_squared += (double)n2 * q2 * q2;
    double s_squared = numerator_s_squared / ((r - 1.0) * n_bar);
    double x_wc = global_p * (1.0 - global_p) - ((r - 1.0) / r) * s_squared;
    double a_numerator_term = s_squared - (x_wc / (n_bar - 1.0));
    double a_denominator_factor = 1.0 - (c_squared / (r - 1.0));
    a = a_numerator_term / a_denominator_factor;
    b = (n_bar / (n_bar - 1.0)) * x_wc;
}

// fst_estimate_from_components threshold ladder (stats.rs:1781-1812): returns state code
FM_HD int fm_fst_state(double a, double b) {
    double den = a + b;
    if (den > FM_FST_EPSILON) return 0;
    if (den < -FM_FST_EPSILON) return 1;
    if (fabs(a) > FM_FST_EPSILON) return 0;
    return 2;
}
