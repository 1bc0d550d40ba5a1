// fm_hapfreq.cuh -- distinct haplotypes per window with Garud's H1, H12, H123, H2/H1 and haplotype diversity
// (DESIGN.md §0 row f12, §4 "Haplotype frequencies"; estimator and hash in include/ferromic_gpu.h,
// fm_haplotype_frequencies).
//
// 1. fm_k_hapfreq_planes transposes the kept sites into haplotype-major key bits: word w of haplotype h (kept sites
//    [64 w, 64 w + 64), bit t = site 64 w + t) is keys[w * n + h], so the n haplotypes' words of one site word are
//    contiguous and both the stores here and the loads of the hash kernel are coalesced.  A called row of the same
//    layout is built only when some kept site has a missing cell.
// 2. fm_k_hapfreq_hash: one thread per (window, haplotype) streams the window's key words (funnel shift for a start
//    off a word boundary, the last word masked) through the documented hash, and writes (hash, haplotype).  A
//    haplotype with a missing cell in the window gets the hash ~0 and kHapfreqExcluded in its value.
// 3. cub::DeviceSegmentedSort::SortPairs, windows as segments (host side).
// 4. fm_k_hapfreq_count: one CTA per window.  A segmented scan over the sorted hashes gives every entry its run's
//    first used member; every member's key is compared word by word with it, and each run's size and a mismatch bit
//    are accumulated with atomics in `aux`.  A run without a mismatch is one class; a run with one is split into exact
//    classes in the same kernel.  The class sizes then reduce to K, sum c^2 and the top three, and thread 0 evaluates
//    the FP64 statistics in the header's order.  Nothing is kept per haplotype in shared memory, so any n < 2^26 fits.
#pragma once
#include "fm_haplotypes.cuh"

#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>

namespace fm {

constexpr uint32_t kHapfreqCountThreads = 256;
constexpr uint32_t kHapfreqExcluded = 0x80000000u;  // value bit: the haplotype has a missing cell in the window
constexpr uint32_t kHapfreqIdx = 0x03ffffffu;       // value bits of the haplotype index (n < 2^26)
constexpr uint32_t kHapfreqNone = 0xffffffffu;      // no used member yet / not a member
constexpr uint32_t kHapfreqDone = 0xfffffffeu;      // a member already put into a class (collision split)
constexpr uint32_t kHapfreqImpure = 0x80000000u;    // aux bit: some member's key differs from the run's first

// The hash of include/ferromic_gpu.h: Horner's rule mod 2^64 over the key's words, then the MurmurHash3 finalizer.
constexpr uint64_t kHapfreqMul = 0x9e3779b97f4a7c15ull;
__host__ __device__ __forceinline__ uint64_t hapfreq_finalize(uint64_t h) {
    h ^= h >> 33;
    h *= 0xff51afd7ed558ccdull;
    h ^= h >> 33;
    h *= 0xc4ceb9fe1a85ec53ull;
    h ^= h >> 33;
    return h;
}

// A window's key words: kept sites [first, first + sites) are bits [first, first + sites) of a haplotype's row.
struct HapfreqWin {
    uint32_t fw, shift, nwords;
    uint64_t last_mask;
    __device__ __forceinline__ HapfreqWin(uint32_t first, uint32_t sites) {
        fw = first >> 6;
        shift = first & 63;
        nwords = (sites + 63) >> 6;
        last_mask = (sites & 63) ? (1ull << (sites & 63)) - 1 : ~0ull;
    }
    // Word j of haplotype h's key; rows hold KW + 1 word rows (the last one zero), so word fw + j + 1 always exists.
    __device__ __forceinline__ uint64_t word(const uint64_t *__restrict__ rows, uint32_t n, uint32_t h, uint32_t j) const {
        const uint64_t lo = __ldg(rows + (size_t)(fw + j) * n + h), hi = __ldg(rows + (size_t)(fw + j + 1) * n + h);
        const uint64_t x = shift ? (lo >> shift) | (hi << (64 - shift)) : lo;
        return j + 1 == nwords ? x & last_mask : x;
    }
    __device__ __forceinline__ bool same(const uint64_t *__restrict__ rows, uint32_t n, uint32_t a, uint32_t b) const {
        for (uint32_t j = 0; j < nwords; ++j)
            if (word(rows, n, a, j) != word(rows, n, b, j)) return false;
        return true;
    }
};

// Kept sites x selected haplotypes -> keys (and called bits) [KW][n].  One warp per tile of 64 kept sites x 32
// haplotypes (task = word * ceil(n / 32) + haplotype block, so the warps of a block store adjacent 256-byte runs):
// lane = haplotype, so each site's 32 cells are one coalesced read of a row and each lane's 64 bits are already its
// haplotype's word (the transpose of fm_k_ld_planes, whose ballots build site words).  Sites past M stay 0.
__global__ void __launch_bounds__(256)
fm_k_hapfreq_planes(HapCells cells, const uint32_t *__restrict__ off, uint32_t n, const uint32_t *__restrict__ kept,
                    uint32_t M, uint32_t KW, uint64_t *__restrict__ keys, uint64_t *__restrict__ called_rows) {
    constexpr uint32_t FULL = 0xffffffffu;
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t n_hb = (n + 31) / 32;
    const uint64_t n_tasks = (uint64_t)KW * n_hb;
    const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t task = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; task < n_tasks; task += n_warps) {
        const uint32_t w = (uint32_t)(task / n_hb), hb = (uint32_t)(task % n_hb);
        const uint32_t h = hb * 32u + lane, s0 = w * 64u, nt = min(64u, M - s0);
        const uint32_t col = h < n ? __ldg(off + h) : 0u;
        const uint32_t k0 = lane < nt ? __ldg(kept + s0 + lane) : 0u;
        const uint32_t k1 = lane + 32u < nt ? __ldg(kept + s0 + 32u + lane) : 0u;
        uint64_t a = 0, c = 0;
#pragma unroll 8
        for (uint32_t t = 0; t < nt; ++t) {
            const uint32_t v = __shfl_sync(FULL, t < 32u ? k0 : k1, t & 31u);
            bool cl = false, al = false, other;
            if (h < n) cells.read(v, col, cl, al, other);
            a |= (uint64_t)al << t;
            c |= (uint64_t)cl << t;
        }
        if (h >= n) continue;
        keys[(size_t)w * n + h] = a;
        if (called_rows) called_rows[(size_t)w * n + h] = c;
    }
}

// One thread per (window w0 + e / n, haplotype e % n) of a batch of elems = windows * n entries.
__global__ void __launch_bounds__(256)
fm_k_hapfreq_hash(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ called_rows, uint32_t n,
                  const uint32_t *__restrict__ wfirst, const uint32_t *__restrict__ wsites, uint32_t w0, uint64_t elems,
                  uint64_t *__restrict__ hash_out, uint32_t *__restrict__ val_out) {
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= elems) return;
    const uint32_t w = w0 + (uint32_t)(e / n), h = (uint32_t)(e % n);
    const HapfreqWin win(__ldg(wfirst + w), __ldg(wsites + w));
    bool used = true;
    if (called_rows)
        for (uint32_t j = 0; j < win.nwords; ++j)
            used &= win.word(called_rows, n, h, j) == (j + 1 == win.nwords ? win.last_mask : ~0ull);
    uint64_t x = 0;
    for (uint32_t j = 0; j < win.nwords; ++j) x = x * kHapfreqMul + win.word(keys, n, h, j);
    hash_out[e] = used ? hapfreq_finalize(x) : ~0ull;
    val_out[e] = used ? h : (h | kHapfreqExcluded);
}

// Segmented min-scan element: head starts a run of equal hashes, rep = the smallest used position seen in it.
struct HapfreqRun {
    uint32_t head, rep;
};
struct HapfreqRunOp {
    __device__ __forceinline__ HapfreqRun operator()(const HapfreqRun &a, const HapfreqRun &b) const {
        return b.head ? b : HapfreqRun{a.head, min(a.rep, b.rep)};
    }
};
struct HapfreqCarry {  // the running prefix of the tiles of one segment
    HapfreqRun run;
    __device__ __forceinline__ HapfreqRun operator()(const HapfreqRun &tile_total) {
        const HapfreqRun prev = run;
        run = HapfreqRunOp()(run, tile_total);
        return prev;
    }
};

// Per-thread then per-window totals of the class sizes: K, N = sum c, s2 = sum c^2 and the top three (descending).
struct HapfreqAcc {
    unsigned long long s2;
    uint32_t k, used, t0, t1, t2;
    __device__ __forceinline__ void top(uint32_t c) {
        if (c > t0) {
            t2 = t1;
            t1 = t0;
            t0 = c;
        } else if (c > t1) {
            t2 = t1;
            t1 = c;
        } else if (c > t2) {
            t2 = c;
        }
    }
    __device__ __forceinline__ void add(uint32_t c) {
        k += 1;
        used += c;
        s2 += (unsigned long long)c * c;
        top(c);
    }
};
struct HapfreqAccOp {
    __device__ __forceinline__ HapfreqAcc operator()(const HapfreqAcc &a, const HapfreqAcc &b) const {
        HapfreqAcc r{a.s2 + b.s2, a.k + b.k, a.used + b.used, a.t0, a.t1, a.t2};
        r.top(b.t0);
        r.top(b.t1);
        r.top(b.t2);
        return r;
    }
};

// Per-window device outputs (index: window), and the batch's class-size scratch (index: window of the batch).
struct HapfreqDev {
    uint32_t *n_used, *distinct, *top;  // top [3 per window]
    unsigned long long *sum_sq;
    double *h1, *h12, *h123, *h2_h1, *diversity;
    uint32_t *cls;      // nullable: class sizes, window w of the batch at [w * n, w * n + K)
    uint32_t *cls_k;    // with cls: K of window w of the batch
};

// One CTA per window of a batch: entries [w * n, (w + 1) * n) of the sorted (hash, value) pairs.  rep and aux are
// per-entry scratch of the batch (aux cleared before the launch).
__global__ void __launch_bounds__(kHapfreqCountThreads)
fm_k_hapfreq_count(const uint64_t *__restrict__ keys, uint32_t n, const uint32_t *__restrict__ wfirst,
                   const uint32_t *__restrict__ wsites, uint32_t w0, const uint64_t *__restrict__ hk,
                   const uint32_t *__restrict__ hv, uint32_t *__restrict__ rep, uint32_t *__restrict__ aux,
                   HapfreqDev out, unsigned long long *__restrict__ collisions) {
    using Scan = cub::BlockScan<HapfreqRun, kHapfreqCountThreads>;
    using Reduce = cub::BlockReduce<HapfreqAcc, kHapfreqCountThreads>;
    __shared__ union {
        typename Scan::TempStorage scan;
        typename Reduce::TempStorage reduce;
    } tmp;
    __shared__ uint32_t cls_fill;
    const uint32_t b = blockIdx.x, w = w0 + b, t = threadIdx.x;
    const size_t seg = (size_t)b * n;
    const HapfreqWin win(__ldg(wfirst + w), __ldg(wsites + w));
    if (t == 0) cls_fill = 0;

    // 1. every used entry's run representative, its key check, and the run sizes
    HapfreqCarry carry{{0u, kHapfreqNone}};
    for (uint32_t base = 0; base < n; base += kHapfreqCountThreads) {
        const uint32_t i = base + t;
        const bool in = i < n;
        const uint64_t h = in ? hk[seg + i] : 0;
        const uint32_t v = in ? hv[seg + i] : kHapfreqExcluded;
        const bool used = in && !(v & kHapfreqExcluded);
        HapfreqRun x{(uint32_t)(!in || i == 0 || hk[seg + i - 1] != h), used ? i : kHapfreqNone}, y;
        Scan(tmp.scan).InclusiveScan(x, y, HapfreqRunOp(), carry);
        __syncthreads();  // tmp is reused by the next tile
        if (in) rep[seg + i] = used ? y.rep : kHapfreqNone;
        uint32_t add = 0;
        if (used) {
            add = 1;
            if (y.rep != i && !win.same(keys, n, v & kHapfreqIdx, hv[seg + y.rep] & kHapfreqIdx)) add |= kHapfreqImpure;
        }
        // one atomic per distinct representative of the warp
        const uint32_t key = used ? y.rep : kHapfreqNone;
        const uint32_t peers = __match_any_sync(0xffffffffu, key);
        const uint32_t total = __reduce_add_sync(peers, add & ~kHapfreqImpure);
        const uint32_t impure = __reduce_or_sync(peers, add & kHapfreqImpure);
        if (used && (t & 31) == (uint32_t)(__ffs(peers) - 1)) {
            atomicAdd(aux + seg + y.rep, total);  // n < 2^26: never reaches the mismatch bit
            if (impure) atomicOr(aux + seg + y.rep, kHapfreqImpure);
        }
    }
    __syncthreads();

    // 2. classes: a clean run is one; a run with a mismatch is split exactly, first unassigned member first
    HapfreqAcc acc{0ull, 0u, 0u, 0u, 0u, 0u};
    auto emit = [&](uint32_t c) {
        acc.add(c);
        if (out.cls) out.cls[seg + atomicAdd(&cls_fill, 1u)] = c;
    };
    for (uint32_t i = t; i < n; i += kHapfreqCountThreads) {
        if (__ldcg(rep + seg + i) != i) continue;
        const uint32_t a = __ldcg(aux + seg + i);
        if (!(a & kHapfreqImpure)) {
            emit(a);
            continue;
        }
        atomicAdd(collisions, 1ull);
        const uint64_t h = hk[seg + i];
        uint32_t end = i + 1;
        while (end < n && hk[seg + end] == h) ++end;
        for (uint32_t r = i; r < end; ++r) {
            const uint32_t vr = hv[seg + r];
            if ((vr & kHapfreqExcluded) || __ldcg(rep + seg + r) == kHapfreqDone) continue;
            uint32_t c = 0;
            for (uint32_t j = r; j < end; ++j) {
                const uint32_t vj = hv[seg + j];
                if ((vj & kHapfreqExcluded) || __ldcg(rep + seg + j) == kHapfreqDone) continue;
                if (j == r || win.same(keys, n, vj & kHapfreqIdx, vr & kHapfreqIdx)) {
                    rep[seg + j] = kHapfreqDone;
                    ++c;
                }
            }
            emit(c);
        }
    }
    const HapfreqAcc tot = Reduce(tmp.reduce).Reduce(acc, HapfreqAccOp());
    if (t) return;
    const uint64_t N = tot.used, s2 = tot.s2, c1 = tot.t0, c2 = tot.t1, c3 = tot.t2;
    out.n_used[w] = (uint32_t)N;
    out.distinct[w] = tot.k;
    out.top[3 * (size_t)w] = (uint32_t)c1;
    out.top[3 * (size_t)w + 1] = (uint32_t)c2;
    out.top[3 * (size_t)w + 2] = (uint32_t)c3;
    out.sum_sq[w] = s2;
    if (out.cls_k) out.cls_k[b] = tot.k;
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    const double nn = (double)(N * N);
    out.h1[w] = N ? (double)s2 / nn : nan;
    out.h12[w] = N ? (double)(s2 + 2 * c1 * c2) / nn : nan;
    out.h123[w] = N ? (double)(s2 + 2 * (c1 * c2 + c1 * c3 + c2 * c3)) / nn : nan;
    out.h2_h1[w] = N ? (double)(s2 - c1 * c1) / (double)s2 : nan;
    out.diversity[w] = N > 1 ? (double)(N * N - s2) / (double)(N * (N - 1)) : nan;
}

// Class sizes of a batch, compacted: window w's K sizes go to [coff[w], coff[w] + K) of dst.
__global__ void __launch_bounds__(256)
fm_k_hapfreq_gather(const uint32_t *__restrict__ cls, uint32_t n, uint64_t elems, const uint32_t *__restrict__ cls_k,
                    const uint32_t *__restrict__ coff, uint32_t *__restrict__ dst) {
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= elems) return;
    const uint32_t w = (uint32_t)(e / n), j = (uint32_t)(e % n);
    if (j < cls_k[w]) dst[coff[w] + j] = cls[e];
}

}  // namespace fm
