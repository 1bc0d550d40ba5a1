// fm_falsta.cuh -- SURVEY §8(f3): body lines of the per-site FALSTA tracks written by the CLI
// (append_diversity_falsta / append_fst_falsta, process.rs:3740-4041).  A track body is ONE line of
// region_len comma-joined tokens: a default token at positions without a record, and the record's
// value rendered as  NaN -> "NA",  0.0 -> "0",  (+-inf -> "Infinity" / "-Infinity" in the FST
// tracks),  otherwise Rust's `{:.6}`.  The reference allocates a String per position and re-scans
// every record per track; here one kernel chain renders the line on the device:
//   scatter (last record at a position wins) -> token lengths -> exclusive scan -> write.
// `{:.6}` is reproduced exactly: the binary value m * 2^e is scaled by 10^6 in 128-bit integer
// arithmetic and rounded half-to-even on the exact remainder, as Rust's (and C's) correctly rounded
// formatter does.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace fm {

// Renders one value; returns its length (buf needs >= 56 bytes).
__host__ __device__ inline uint32_t fm_falsta_token(double v, int mode, char *buf) {
    auto put = [&](const char *s) {
        uint32_t n = 0;
        while (s[n]) {
            buf[n] = s[n];
            ++n;
        }
        return n;
    };
    if (v != v) return put("NA");
#ifdef __CUDA_ARCH__
    const unsigned long long bits = (unsigned long long)__double_as_longlong(v);
#else
    unsigned long long bits;
    __builtin_memcpy(&bits, &v, 8);
#endif
    const bool neg = (bits >> 63) != 0;
    const uint32_t ex = (uint32_t)((bits >> 52) & 0x7ffu);
    const unsigned long long frac = bits & 0xfffffffffffffull;
    if (ex == 0x7ffu) {  // infinity (NaN handled above)
        if (mode == FM_FALSTA_FST) return put(neg ? "-Infinity" : "Infinity");
        return put(neg ? "-inf" : "inf");
    }
    if (ex == 0 && frac == 0 && mode != FM_FALSTA_TSV) return put("0");  // v == 0.0 (either sign)
    const unsigned long long m = ex ? (frac | (1ull << 52)) : frac;
    const int e = ex ? (int)ex - 1075 : -1074;
    unsigned __int128 N = (unsigned __int128)m * 1000000u;  // < 2^73
    unsigned __int128 q;
    if (e >= 0) {
        q = e > 50 ? ~(unsigned __int128)0 : (N << e);  // |v| >= 2^103 does not occur for these statistics
    } else {
        const int k = -e;
        if (k >= 127) {
            q = 0;
        } else {
            q = N >> k;
            const unsigned __int128 rem = N & ((((unsigned __int128)1) << k) - 1);
            const unsigned __int128 half = ((unsigned __int128)1) << (k - 1);
            if (rem > half || (rem == half && (q & 1))) q += 1;  // round half to even on the exact value
        }
    }
    unsigned __int128 ip = q / 1000000u;
    uint32_t fp = (uint32_t)(q % 1000000u);
    char tmp[48];
    uint32_t nd = 0;
    do {
        tmp[nd++] = (char)('0' + (uint32_t)(ip % 10u));
        ip /= 10u;
    } while (ip != 0);
    uint32_t n = 0;
    if (neg) buf[n++] = '-';
    while (nd) buf[n++] = tmp[--nd];
    buf[n++] = '.';
    for (int d = 5; d >= 0; --d) {
        buf[n + d] = (char)('0' + fp % 10u);
        fp /= 10u;
    }
    return n + 6;
}

// last record at a position wins (the reference overwrites line[idx] in record order)
__global__ void __launch_bounds__(256)
fm_k_falsta_scatter(const int64_t *__restrict__ pos1, uint32_t n, uint64_t rs, uint64_t re, int *__restrict__ idx) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint64_t p = (uint64_t)(pos1[i] - 1);  // `(pos - 1) as usize` wraps for pos <= 0 (process.rs:318)
        if (p >= rs && p < re) atomicMax(idx + (p - rs), (int)i);
    }
}

// Track t of a call renders values[t * n + i]; all tracks of a call share the record positions.
// Every token is followed by one separator byte (',' inside a line, '\n' between tracks) except the
// very last token of the call.
struct U32ToU64 {  // widens token lengths for the 64-bit prefix sum
    __host__ __device__ __forceinline__ uint64_t operator()(uint32_t x) const { return (uint64_t)x; }
};

__global__ void __launch_bounds__(256)
fm_k_falsta_lengths(const int *__restrict__ idx, const double *__restrict__ values, uint64_t n, uint64_t region_len,
                    uint32_t n_tracks, int mode, uint32_t *__restrict__ lens, uint32_t test_inflate) {
    const uint32_t dflt = mode == FM_FALSTA_FST ? 2u : 1u;
    const uint64_t total = region_len * n_tracks;
    for (uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; g < total;
         g += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t t = g / region_len, j = g - t * region_len;
        const int i = idx[j];
        uint32_t len = dflt;
        if (i >= 0) {
            char buf[56];
            len = fm_falsta_token(values[t * n + (uint64_t)i], mode, buf);
        }
        lens[g] = len + (g + 1 < total ? 1u : 0u) + test_inflate;  // test_inflate: length-query tests of > 4 GiB bodies
    }
}

__global__ void __launch_bounds__(256)
fm_k_falsta_write(const int *__restrict__ idx, const double *__restrict__ values, uint64_t n, uint64_t region_len,
                  uint32_t n_tracks, int mode, const uint64_t *__restrict__ offs, char *__restrict__ out,
                  const uint64_t *__restrict__ track_shift) {
    const uint64_t total = region_len * n_tracks;
    for (uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; g < total;
         g += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t t = g / region_len, j = g - t * region_len;
        const int i = idx[j];
        char *dst = out + offs[g] + (track_shift ? track_shift[t] : 0);
        uint32_t len;
        if (i >= 0) {
            char buf[56];
            len = fm_falsta_token(values[t * n + (uint64_t)i], mode, buf);
            for (uint32_t k = 0; k < len; ++k) dst[k] = buf[k];
        } else if (mode == FM_FALSTA_FST) {
            dst[0] = 'N';
            dst[1] = 'A';
            len = 2;
        } else {
            dst[0] = '0';
            len = 1;
        }
        if (g + 1 < total) dst[len] = (j + 1 < region_len) ? ',' : '\n';
    }
}

// Headed text (fm_falsta_tracks_bgzf): heads[t] + line t + '\n' per track.  The lines were written with track t
// shifted by track_shift[t] = the bytes of heads 0..t; block t copies heads[t] (bytes [head_off[t], head_off[t + 1])
// of `heads`) in front of line t, whose first token the scan put at line_start[t] (unshifted).  The last block
// closes the text with '\n' at out[end].
__global__ void __launch_bounds__(128)
fm_k_falsta_heads(const char *__restrict__ heads, const uint64_t *__restrict__ head_off,
                  const uint64_t *__restrict__ line_start, const uint64_t *__restrict__ track_shift, uint32_t n_tracks,
                  uint64_t end, char *__restrict__ out) {
    const uint32_t t = blockIdx.x;
    const uint64_t h0 = head_off[t], hn = head_off[t + 1] - h0;
    char *dst = out + line_start[t] + track_shift[t] - hn;
    for (uint64_t k = threadIdx.x; k < hn; k += blockDim.x) dst[k] = heads[h0 + k];
    if (t + 1 == n_tracks && threadIdx.x == 0) out[end] = '\n';
}

}  // namespace fm
