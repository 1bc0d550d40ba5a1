// fm_gpu.cu -- C-ABI implementation (include/ferromic_gpu.h): handle management, the host-side
// guard/dispatch logic of the reference's public stats.rs functions, kernel launches and the
// deterministic final reductions.  No CPU fallback: every compute entry point needs a device.
#include "../../include/ferromic_gpu.h"
#include "fm_kernels.cuh"
#include "fm_wc.cuh"
#include "fm_comm.cuh"
#include "fm_multi.cuh"
#include "fm_falsta.cuh"
#include "fm_vcf.cuh"
#include "fm_pairwise.cuh"

#include <nvtx3/nvToolsExt.h>

#include <cub/device/device_scan.cuh>
#include <thrust/iterator/transform_iterator.h>
#include <cuda/std/functional>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <map>
#include <set>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

// fm_host_pack.cpp (plain host code): u8 rows -> packed bit words
const char *fm_host_pack_rows(const uint8_t *rows, const uint64_t *missing_whole_or_null, int missing_mode,
                              size_t first_row, size_t n_rows, size_t n_total_rows, size_t stride,
                              uint32_t *allele_bits, uint32_t *called_bits_or_null, int n_threads);
const char *fm_host_pack_rows_sparse(const uint8_t *rows, const uint64_t *missing_whole_or_null, int missing_mode,
                                     size_t first_row, size_t n_rows, size_t n_total_rows, size_t stride,
                                     uint32_t *allele_bits, uint64_t *row_start, void *missing_cols, size_t capacity,
                                     int col_bytes, int n_threads, size_t *needed);
const char *fm_host_pack_rows_generic(const uint8_t *rows, const uint64_t *missing, int mode, size_t first_row,
                                      size_t n_rows, size_t n_total_rows, size_t stride, uint32_t *abits,
                                      uint32_t *cbits);

namespace {

thread_local std::string t_err;
// Device selection (SURVEY 5 / 8b): fm_set_devices -- or the environment variable FERROMIC_GPU_DEVICES, a comma
// separated list of CUDA ordinals, read once -- restricts the library to a subset of the visible GPUs; a host thread
// that never called fm_set_device works on the first allowed device, fm_set_device accepts only allowed ordinals.
thread_local int t_device_sel = -1;  // -1: not chosen yet on this thread
std::mutex g_dev_mu;
std::vector<int> g_devices;          // empty: every visible device is allowed
bool g_devices_init = false;
void devices_init_locked() {
    if (g_devices_init) return;
    g_devices_init = true;
    const char *e = getenv("FERROMIC_GPU_DEVICES");
    if (!e || !*e) return;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        n = 0;
    }
    std::string tok;
    for (const char *p = e;; ++p) {
        if (*p == ',' || *p == 0) {
            if (!tok.empty()) {
                char *end = nullptr;
                const long d = strtol(tok.c_str(), &end, 10);
                if (end && *end == 0 && d >= 0 && d < n &&
                    std::find(g_devices.begin(), g_devices.end(), (int)d) == g_devices.end())
                    g_devices.push_back((int)d);
                tok.clear();
            }
            if (*p == 0) break;
        } else if (*p != ' ')
            tok.push_back(*p);
    }
}
bool device_allowed(int d) {
    std::lock_guard<std::mutex> lk(g_dev_mu);
    devices_init_locked();
    return g_devices.empty() || std::find(g_devices.begin(), g_devices.end(), d) != g_devices.end();
}
int cur_dev() {
    if (t_device_sel < 0) {
        std::lock_guard<std::mutex> lk(g_dev_mu);
        devices_init_locked();
        t_device_sel = g_devices.empty() ? 0 : g_devices[0];
    }
    return t_device_sel;
}
#define t_device (cur_dev())
thread_local fm_timings t_tim = {};
std::atomic<uint64_t> g_launches{0};

struct FmError {
    fm_status code;
    std::string msg;
};

[[noreturn]] void fail(fm_status code, const std::string &msg) { throw FmError{code, msg}; }

#define CK(call)                                                                              \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess) {                                                              \
            char buf_[512];                                                                   \
            snprintf(buf_, sizeof(buf_), "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                     __FILE__, __LINE__);                                                     \
            cudaError_t last_ = cudaGetLastError();                                           \
            (void)last_;                                                                      \
            fail(e_ == cudaErrorNoDevice || e_ == cudaErrorInsufficientDriver ? FM_ERR_NO_DEVICE \
                                                                               : FM_ERR_CUDA, \
                 buf_);                                                                       \
        }                                                                                     \
    } while (0)

// NVTX ranges around the stages of the path (SURVEY 5: tracing): ingest / repack / plane pass / exchange / W&C /
// VCF / FALSTA show up as named ranges in Nsight Systems and ncu --nvtx; free when no profiler is attached.
struct NvtxRange {
    explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
    NvtxRange(const NvtxRange &) = delete;
    NvtxRange &operator=(const NvtxRange &) = delete;
};
#define FM_NVTX(name) NvtxRange nvtx_range_(name)

template <class F>
fm_status guarded(F &&f) {
    try {
        f();
        return FM_OK;
    } catch (const FmError &e) {
        t_err = e.msg;
        return e.code;
    } catch (const std::bad_alloc &) {
        t_err = "out of host memory";
        return FM_ERR_INVALID_ARG;
    } catch (const std::exception &e) {
        t_err = e.what();
        return FM_ERR_INVALID_ARG;
    } catch (...) {
        t_err = "unknown error";
        return FM_ERR_INVALID_ARG;
    }
}

void require_device() {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        fail(FM_ERR_NO_DEVICE,
             "no CUDA device available: ferromic_gpu has no CPU fallback on this path");
    }
}

// The calling thread's stream.  A scope may redirect it (StreamScope): the streaming ingest runs the per-site pass
// of a chunk on its own compute stream with the very code of the public call.
thread_local cudaStream_t t_stream_override = nullptr;
cudaStream_t stream() { return t_stream_override ? t_stream_override : cudaStreamPerThread; }
struct StreamScope {
    cudaStream_t saved;
    explicit StreamScope(cudaStream_t s) : saved(t_stream_override) { t_stream_override = s; }
    ~StreamScope() { t_stream_override = saved; }
};

uint32_t env_u32_early(const char *name, uint32_t dflt) {
    const char *v = getenv(name);
    if (!v || !*v) return dflt;
    const long x = strtol(v, nullptr, 10);
    return x > 0 ? (uint32_t)x : dflt;
}

// Caching device allocator.  A released handle's bitplanes / staging buffers go to a per-device
// free list keyed by (rounded) size and are handed to the next request instead of back to the
// driver: cudaMalloc + cudaFree of multi-GB buffers cost far more than the kernels and vary by
// 10x between calls.  Every cached block carries an event recorded on the freeing thread's
// stream; the next owner's stream waits on it, so reuse is safe across threads.
// fm_trim_pool() returns the cached memory to the driver.
struct CachedBlock {
    void *p;
    cudaEvent_t ev;
};
struct DeviceCache {
    std::mutex mu;
    std::multimap<size_t, CachedBlock> free_blocks;  // rounded size -> block
    std::unordered_map<const void *, size_t> live;    // live pointer -> rounded size
};
DeviceCache &cache_of(int device) {
    static DeviceCache caches[64];
    return caches[(device >= 0 && device < 64) ? device : 0];
}
size_t round_alloc(size_t bytes) {
    if (bytes < ((size_t)1 << 20)) return (std::max<size_t>(bytes, 16) + 511) & ~(size_t)511;
    return (bytes + (((size_t)2 << 20) - 1)) & ~(((size_t)2 << 20) - 1);
}
void cache_release_all(int device) {
    DeviceCache &c = cache_of(device);
    std::lock_guard<std::mutex> lk(c.mu);
    for (auto &kv : c.free_blocks) {
        cudaEventSynchronize(kv.second.ev);
        cudaEventDestroy(kv.second.ev);
        cudaFree(kv.second.p);
    }
    c.free_blocks.clear();
}
void *dev_alloc(size_t bytes) {
    int dev = 0;
    CK(cudaGetDevice(&dev));
    const size_t want = round_alloc(bytes);
    DeviceCache &c = cache_of(dev);
    {
        std::unique_lock<std::mutex> lk(c.mu);
        auto it = c.free_blocks.lower_bound(want);
        if (it != c.free_blocks.end() && it->first <= want + want / 4 + 4096) {
            CachedBlock b = it->second;
            const size_t sz = it->first;
            c.free_blocks.erase(it);
            c.live[b.p] = sz;
            lk.unlock();
            cudaStreamWaitEvent(stream(), b.ev, 0);  // work of the previous owner
            cudaEventDestroy(b.ev);
            return b.p;
        }
    }
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaErrorMemoryAllocation) {  // give the cached blocks back and retry once
        cudaGetLastError();
        cache_release_all(dev);
        e = cudaMalloc(&p, want);
    }
    CK(e);
    std::lock_guard<std::mutex> lk(c.mu);
    c.live[p] = want;
    return p;
}
void dev_free(const void *p) {
    if (!p) return;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return;
    DeviceCache &c = cache_of(dev);
    size_t sz = 0;
    {
        std::lock_guard<std::mutex> lk(c.mu);
        auto it = c.live.find(p);
        if (it == c.live.end()) return;  // not ours (caller-owned device buffers are never freed here)
        sz = it->second;
        c.live.erase(it);
    }
    CachedBlock b{const_cast<void *>(p), nullptr};
    if (cudaEventCreateWithFlags(&b.ev, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventRecord(b.ev, stream()) != cudaSuccess) {
        cudaGetLastError();
        if (b.ev) cudaEventDestroy(b.ev);
        cudaDeviceSynchronize();
        cudaFree(b.p);
        return;
    }
    std::lock_guard<std::mutex> lk(c.mu);
    c.free_blocks.emplace(sz, b);
}

// Host -> device copies of caller memory.  Pinned (page-locked / registered) buffers go straight to
// the copy engine.  Pageable buffers -- a Rust Vec<u8>, a numpy array -- would be staged by the
// driver through one internal bounce buffer with a single-threaded memcpy (5-10 GB/s); instead the
// library keeps a few pinned bounce buffers per process, fills them with several host threads and
// lets the DMA of piece i overlap the memcpy of piece i+1.  On return the source is no longer
// referenced; the device side of the copy is ordered on `st`.
struct BouncePool {
    static constexpr size_t kPiece = (size_t)32 << 20;
    static constexpr int kBuffers = 4;
    std::mutex mu;
    uint8_t *buf[kBuffers] = {};
    cudaEvent_t ev[kBuffers] = {};
    bool busy[kBuffers] = {};
    int next = 0;
    int threads = 0;
    ~BouncePool() {
        for (int i = 0; i < kBuffers; ++i) {
            if (buf[i]) cudaFreeHost(buf[i]);
            if (ev[i]) cudaEventDestroy(ev[i]);
        }
    }
    void copy(void *dst, const void *src, size_t bytes, cudaStream_t st) {
        std::lock_guard<std::mutex> lk(mu);  // one pageable upload at a time per process
        if (!threads) {
            const unsigned hw = std::thread::hardware_concurrency();
            threads = (int)std::max(1u, std::min(32u, env_u32_early("FM_HOST_THREADS", hw ? std::min(hw / 2, 8u) : 4)));
        }
        const uint8_t *s8 = static_cast<const uint8_t *>(src);
        uint8_t *d8 = static_cast<uint8_t *>(dst);
        for (size_t o = 0; o < bytes; o += kPiece) {
            const size_t n = std::min(kPiece, bytes - o);
            const int b = next;
            next = (next + 1) % kBuffers;
            if (!buf[b]) {
                CK(cudaHostAlloc((void **)&buf[b], kPiece, cudaHostAllocDefault));
                CK(cudaEventCreateWithFlags(&ev[b], cudaEventDisableTiming));
            }
            if (busy[b]) CK(cudaEventSynchronize(ev[b]));  // its previous DMA has drained
            const int T = (int)std::min<size_t>((size_t)threads, (n + ((size_t)4 << 20) - 1) / ((size_t)4 << 20));
            if (T <= 1) {
                std::memcpy(buf[b], s8 + o, n);
            } else {
                std::vector<std::thread> pool;
                const size_t slice = ((n + T - 1) / T + 63) & ~(size_t)63;
                for (int t = 1; t < T; ++t) {
                    const size_t lo = std::min(n, slice * t), hi = std::min(n, slice * (t + 1));
                    if (hi > lo) pool.emplace_back([=] { std::memcpy(buf[b] + lo, s8 + o + lo, hi - lo); });
                }
                std::memcpy(buf[b], s8 + o, std::min(n, slice));
                for (auto &th : pool) th.join();
            }
            CK(cudaMemcpyAsync(d8 + o, buf[b], n, cudaMemcpyHostToDevice, st));
            CK(cudaEventRecord(ev[b], st));
            busy[b] = true;
        }
    }
};
BouncePool g_bounce;

// Pinned host buffers for the pack-and-upload ingest (fm_ingest_rows_pack): cudaHostAlloc of tens of MB costs
// milliseconds, so buffers are kept for the life of the process and handed from one ingest to the next.
struct PinnedPool {
    static constexpr size_t kBytes = (size_t)32 << 20;
    std::mutex mu;
    std::vector<uint8_t *> free_list;
    uint8_t *take() {
        {
            std::lock_guard<std::mutex> lk(mu);
            if (!free_list.empty()) {
                uint8_t *p = free_list.back();
                free_list.pop_back();
                return p;
            }
        }
        uint8_t *p = nullptr;
        CK(cudaHostAlloc((void **)&p, kBytes, cudaHostAllocDefault));
        return p;
    }
    void give(uint8_t *p) {
        if (!p) return;
        std::lock_guard<std::mutex> lk(mu);
        free_list.push_back(p);
    }
};
PinnedPool g_pinned;

bool host_is_pinned(const void *p) {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeManaged;
}

// Device alias of a caller's host buffer when the WHOLE range [p, p + bytes) lies inside one page-locked allocation
// (cudaHostAlloc / cudaHostRegister): kernels can then store results straight into it over PCIe instead of writing
// HBM and copying afterwards.  nullptr for pageable memory or when the range cannot be proved.
void *mapped_host_range(const void *p, size_t bytes) {
    if (!p || !bytes) return nullptr;
    static const uint32_t off = env_u32_early("FM_NO_DIRECT_TRACKS", 0);
    if (off) return nullptr;
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    if (at.type != cudaMemoryTypeHost || !at.devicePointer) return nullptr;
    typedef int (*range_fn)(unsigned long long *, size_t *, unsigned long long);  // cuMemGetAddressRange
    static range_fn get_range = [] {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &fn, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess) {
            cudaGetLastError();
            fn = nullptr;
        }
        return reinterpret_cast<range_fn>(fn);
    }();
    if (!get_range) return nullptr;
    unsigned long long base = 0;
    size_t size = 0;
    const unsigned long long dp = (unsigned long long)(uintptr_t)at.devicePointer;
    if (get_range(&base, &size, dp) != 0) return nullptr;
    if (dp < base || dp - base > size || bytes > size - (dp - base)) return nullptr;
    return at.devicePointer;
}

// copy caller memory to the device on `st`; the source may be reused as soon as this returns
// only if the caller synchronises `st` (pinned) -- pageable sources are already released.
void h2d(void *dst, const void *src, size_t bytes, cudaStream_t st) {
    if (!bytes) return;
    if (bytes < ((size_t)1 << 20) || host_is_pinned(src))
        CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st));
    else
        g_bounce.copy(dst, src, bytes, st);
}

// Event pairs are recycled per host thread and device: cudaEventCreate / Destroy cost microseconds each, and the
// small calls (a sharded Hudson step is ~250 us) create several timers.
struct TimerEventPool {
    std::vector<std::pair<int, cudaEvent_t>> free_events;
    ~TimerEventPool() {
        for (auto &e : free_events) cudaEventDestroy(e.second);
    }
    cudaEvent_t take(int dev) {
        for (size_t i = 0; i < free_events.size(); ++i)
            if (free_events[i].first == dev) {
                cudaEvent_t e = free_events[i].second;
                free_events[i] = free_events.back();
                free_events.pop_back();
                return e;
            }
        cudaEvent_t e;
        CK(cudaEventCreate(&e));
        return e;
    }
    void give(int dev, cudaEvent_t e) {
        if (free_events.size() < 64) free_events.emplace_back(dev, e);
        else cudaEventDestroy(e);
    }
};
thread_local TimerEventPool t_timer_events;

// One non-blocking side stream per (host thread, device) for small kernels that run underneath a large one.
struct SideStreams {
    cudaStream_t s[64] = {};
    ~SideStreams() {
        for (cudaStream_t x : s)
            if (x) cudaStreamDestroy(x);
    }
    cudaStream_t get(int dev) {
        const int d = (dev >= 0 && dev < 64) ? dev : 0;
        if (!s[d]) CK(cudaStreamCreateWithFlags(&s[d], cudaStreamNonBlocking));
        return s[d];
    }
};
thread_local SideStreams t_side_streams;

// Streams of the streaming ingests are recycled per device: creating and destroying a stream is a trip into the
// kernel driver, which serialises across the processes of a multi-GPU job (fm_ingest_begin took 1.4-12 ms with four
// ranks on one host against 0.6 ms alone).  A stream goes back to the pool idle (synchronised).
struct StreamPool {
    std::mutex mu;
    std::vector<std::pair<int, cudaStream_t>> free_list;
    cudaStream_t take(int dev) {
        {
            std::lock_guard<std::mutex> lk(mu);
            for (size_t i = 0; i < free_list.size(); ++i)
                if (free_list[i].first == dev) {
                    cudaStream_t st = free_list[i].second;
                    free_list[i] = free_list.back();
                    free_list.pop_back();
                    return st;
                }
        }
        cudaStream_t st = nullptr;
        CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        return st;
    }
    void give(int dev, cudaStream_t st) {
        if (!st) return;
        std::lock_guard<std::mutex> lk(mu);
        if (free_list.size() < 16) {
            free_list.emplace_back(dev, st);
            return;
        }
        cudaStreamDestroy(st);
    }
};
StreamPool g_stream_pool;

struct Timer {
    cudaEvent_t a, b;
    int dev = 0;
    Timer() {
        if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
        a = t_timer_events.take(dev);
        b = t_timer_events.take(dev);
    }
    ~Timer() {
        t_timer_events.give(dev, a);
        t_timer_events.give(dev, b);
    }
    void start() { CK(cudaEventRecord(a, stream())); }
    void stop() { CK(cudaEventRecord(b, stream())); }
    float ms() {
        CK(cudaEventSynchronize(b));
        float t = 0.f;
        CK(cudaEventElapsedTime(&t, a, b));
        return t;
    }
};

struct EventPairs {
    std::vector<cudaEvent_t> ev;
    ~EventPairs() {
        for (auto e : ev) cudaEventDestroy(e);
    }
    cudaEvent_t next() {
        cudaEvent_t e;
        CK(cudaEventCreate(&e));
        ev.push_back(e);
        return e;
    }
};

template <class T>
struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    DevBuf() = default;
    explicit DevBuf(size_t count) { alloc(count); }
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    void alloc(size_t count) {
        release();
        n = count;
        if (count) p = static_cast<T *>(dev_alloc(count * sizeof(T)));
    }
    void release() {
        if (p) dev_free(p);
        p = nullptr;
        n = 0;
    }
    ~DevBuf() { release(); }
    void upload(const T *h, size_t count) {
        if (count) CK(cudaMemcpyAsync(p, h, count * sizeof(T), cudaMemcpyHostToDevice, stream()));
    }
    void download(T *h, size_t count) const {
        if (count) CK(cudaMemcpyAsync(h, p, count * sizeof(T), cudaMemcpyDeviceToHost, stream()));
    }
};

int sm_count(int device) {
    static std::mutex mu;
    static std::vector<int> cache(64, 0);
    std::lock_guard<std::mutex> lk(mu);
    if (device < 64 && cache[device]) return cache[device];
    int n = 0;
    CK(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device));
    if (device < 64) cache[device] = n;
    return n;
}

inline int64_t sat_sub(int64_t a, int64_t b) {
    if (b > 0 && a < std::numeric_limits<int64_t>::min() + b) return std::numeric_limits<int64_t>::min();
    if (b < 0 && a > std::numeric_limits<int64_t>::max() + b) return std::numeric_limits<int64_t>::max();
    return a - b;
}

inline int64_t region_len(int64_t rs, int64_t re) {  // QueryRegion::len (process.rs:573-584)
    if (rs > re) return 0;
    int64_t as = rs < 0 ? 0 : rs;
    int64_t ae;
    if (re < as)
        ae = as;
    else {
        ae = re == std::numeric_limits<int64_t>::max() ? re : re + 1;
        if (ae < as) ae = as;
    }
    return ae > as ? ae - as : 0;
}

}  // namespace

// Host copy of a matrix's variant positions: a page-locked buffer (pooled, see PosPool) so that the upload to the
// device is a true asynchronous DMA, with a plain heap fallback.  The vector subset the library uses.
struct HostPos {
    int64_t *p = nullptr;
    size_t n = 0, cap = 0;
    bool pinned = false;
    HostPos() = default;
    HostPos(const HostPos &) = delete;
    HostPos &operator=(const HostPos &) = delete;
    HostPos(HostPos &&o) noexcept : p(o.p), n(o.n), cap(o.cap), pinned(o.pinned) { o.p = nullptr; o.n = o.cap = 0; }
    HostPos &operator=(HostPos &&o) noexcept {
        if (this != &o) {
            reset();
            p = o.p; n = o.n; cap = o.cap; pinned = o.pinned;
            o.p = nullptr; o.n = o.cap = 0;
        }
        return *this;
    }
    ~HostPos() { reset(); }
    void reset() {
        if (p) {
            if (pinned) cudaFreeHost(p);
            else delete[] p;
        }
        p = nullptr;
        n = cap = 0;
    }
    void reserve_fresh(size_t count) {  // contents are not kept
        if (count <= cap) return;
        reset();
        const size_t want = (std::max<size_t>(count, 1) + 131071) & ~(size_t)131071;  // 1 MB steps
        void *q = nullptr;
        // small matrices stay on the heap: page-locking costs more than their whole upload
        if (count >= ((size_t)1 << 18) && cudaHostAlloc(&q, want * sizeof(int64_t), cudaHostAllocDefault) == cudaSuccess) {
            p = static_cast<int64_t *>(q);
            pinned = true;
        } else {
            cudaGetLastError();
            p = new int64_t[want];
            pinned = false;
        }
        cap = want;
    }
    void resize(size_t count) {
        reserve_fresh(count);
        n = count;
    }
    int64_t *data() { return p; }
    const int64_t *data() const { return p; }
    size_t size() const { return n; }
    const int64_t *begin() const { return p; }
    const int64_t *end() const { return p + n; }
    int64_t &operator[](size_t i) { return p[i]; }
    const int64_t &operator[](size_t i) const { return p[i]; }
    bool operator!=(const HostPos &o) const { return n != o.n || (n && std::memcmp(p, o.p, n * sizeof(int64_t)) != 0); }
};

// ------------------------------------------------------------------------------------ handles
struct fm_matrix {
    std::atomic<int> refs{1};
    int device = 0;
    const uint8_t *d_data = nullptr;
    const uint64_t *d_missing = nullptr;
    bool has_missing = false;  // matrix carries missingness (d_missing is null after a streaming ingest)
    bool in_band = false;      // missingness is in band: cells >= 0x80 (negative int8) are missing, no bitmap
    bool streamed = false;     // u8 data was never resident: groups had to be declared before ingest
    bool owns = true;
    // packed rows (2-bit ingest format, fm_ingest_rows_packed / fm_matrix_create_packed): full-row allele /
    // called bit words stay resident (0.25 B per genotype), so groups can be created at any time
    bool packed = false;
    uint32_t *d_abits = nullptr, *d_cbits = nullptr;
    uint32_t rw = 0;           // u32 words per packed row = ceil(stride / 32)
    size_t V = 0, S = 0, ploidy = 0, stride = 0;
    uint8_t max_allele = 0;
    // max_allele > 15: the distinct allele values of the matrix (at most 16, value 0 always among them) are mapped to
    // dense ranks in ascending order before they are bit-sliced; every estimator only depends on which alleles are
    // equal and on their ascending order (stats.rs:1859), so the ranks give the reference's results
    uint8_t plane_max_allele = 0;   // largest value the bitplanes have to hold (== max_allele without a remap)
    uint8_t *d_lut = nullptr;       // [256] value -> rank, or nullptr
    HostPos pos;               // host copy of the positions, page-locked when possible (uploads straight from it)
    int64_t *d_pos = nullptr;
    bool sorted = true;
};

struct fm_group {
    fm_matrix *m = nullptr;
    std::vector<uint32_t> off;
    uint32_t n = 0;   // haplotype capacity
    uint32_t wq = 0;  // uint4 per plane row
    uint4 *d_allele = nullptr;
    uint4 *d_called = nullptr;  // multi-allelic groups of a matrix with missing data (fm_k_allele_counts needs allele 0)
    // tail layout (biallelic plane groups written by the compress plans): wq counts the FULL 16-byte words of a row,
    // the last n % 128 haplotypes live in tw u32 words per row in d_tail_a (fm_kernels.cuh GroupPlanes)
    uint32_t tw = 0;
    uint32_t *d_tail_a = nullptr;
    // biallelic plane groups of a matrix with missing data: K1 writes d_cnt (the called count of every site) when it
    // repacks the rows, in place of a called plane; d_cnt is then an input of the plane pass, not a cache of it
    bool cnt_in = false;
    double *d_tab = nullptr;   // 3 x (n+1) doubles: 1/k, k/(k-1), 1/H_{k-1}
    uint32_t *d_off = nullptr; // device copy of `off` (K1)
    std::mutex mu;
    bool have_counts = false;       // d_alt (and d_cnt) hold the counts of every site
    uint32_t *d_alt = nullptr, *d_cnt = nullptr;
    uint32_t n_bits = 1;            // allele bitplanes (1 = biallelic; 2..4 = multi-allelic matrix)
    uint32_t *d_acount = nullptr;   // multi-allelic: cached per-allele counts [V][1 << n_bits]
    bool count_only = false;        // no bitplanes: counts are produced straight from the u8 rows (partitions)
    uint64_t seg = 0, unc = 0;
    double pi_sum = 0.0;  // dense_pi_from_counts form over all sites
};

struct fm_partition {
    fm_matrix *m = nullptr;
    size_t G = 0;
    std::vector<fm_group *> groups;  // one bitplane group per subpopulation
    fm_group *rest = nullptr;        // haplotypes with no group (needed for "alleles present")
    std::mutex mu;
    uint32_t *d_counts_slab = nullptr;  // (alt, called) arrays of all G + 1 count-only groups in one block
    double *d_wc_tab = nullptr;      // K4 reciprocal tables: RN(1/n) | RN(2/n^2), n = 0 .. wc_n_max
    uint32_t wc_n_max = 0;
};

namespace {

void set_dev(const fm_matrix *m) { CK(cudaSetDevice(m->device)); }

// site index range of variants with rs <= pos <= re (positions sorted ascending)
void site_range(const fm_matrix *m, int64_t rs, int64_t re, uint32_t &lo, uint32_t &hi) {
    if (!m->sorted)
        fail(FM_ERR_UNSUPPORTED, "region queries need variant positions sorted ascending");
    lo = (uint32_t)(std::lower_bound(m->pos.begin(), m->pos.end(), rs) - m->pos.begin());
    hi = (uint32_t)(std::upper_bound(m->pos.begin(), m->pos.end(), re) - m->pos.begin());
    if (hi < lo) hi = lo;
}

uint32_t env_u32(const char *name, uint32_t dflt) {
    const char *v = getenv(name);
    if (!v || !*v) return dflt;
    const long x = strtol(v, nullptr, 10);
    return x > 0 ? (uint32_t)x : dflt;
}

// batches [b_lo, b_lo + n_batches) of the sites [v_lo, v_hi) (batch b = sites [32b, 32b+32))
fm::PassGeom batch_range(uint32_t v_lo, uint32_t v_hi) {
    fm::PassGeom G{};
    G.v_lo = v_lo;
    G.v_hi = v_hi;
    G.b_lo = v_lo / 32;
    G.n_batches = v_hi > v_lo ? (v_hi + 31) / 32 - G.b_lo : 0;
    return G;
}

// Lanes per site (log2) of the row pass over rows of wq uint4: enough lanes to cover a row's uint4 columns
// (quarter-warps then read contiguous 128-byte spans), raised until a step of 32 >> lg sites fits a warp's ring
// twice.  5: the rows are too wide for the row pass and take the column-chunked pass.
uint32_t row_lanes_log2(uint32_t wq) {
    uint32_t lg = 0;
    while ((1u << lg) < std::min(wq, 8u)) ++lg;
    while (lg < 5 && (uint64_t)wq * 16u * (32u >> lg) * 2 > fm::kWarpSmemBytes) ++lg;
    return lg;
}

// Geometry of the column-chunked pass over group g's rows (row_lanes_log2(g->wq) == 5).  Rows wider than a warp's
// ring (biobank cohorts) are consumed in column chunks by fewer warps with deeper rings: more bytes in flight per
// warp and the per-step bookkeeping amortised.
fm::PassGeom make_geom(const fm_group *g, uint32_t v_lo, uint32_t v_hi) {
    static const uint32_t chunk_warps = std::min<uint32_t>(env_u32("FM_CHUNK_WARPS", 8), fm::kWarpsPerCta);
    static const uint32_t chunk_step = env_u32("FM_CHUNK_STEP_BYTES", 14336);  // swept on B200: profiles/r01_sweep_chunked.txt
    fm::PassGeom G = batch_range(v_lo, v_hi);
    const uint32_t row_bytes = g->wq * 16u;
    G.warps = (uint64_t)row_bytes * 2 > fm::kWarpSmemBytes ? chunk_warps : fm::kWarpsPerCta;
    G.warp_smem_bytes = (fm::kWarpsPerCta * fm::kWarpSmemBytes / G.warps) & ~127u;
    G.cq = g->wq;
    G.n_chunks = 1;
    if ((uint64_t)row_bytes * 2 > G.warp_smem_bytes) {  // a single row does not fit twice: chunk its columns
        G.cq = std::max(1u, chunk_step / 16u);
        G.n_chunks = (g->wq + G.cq - 1) / G.cq;
    }
    G.stage_bytes = (G.cq * 16u + 127u) & ~127u;
    G.n_stages = std::min<uint32_t>(fm::kMaxStages, G.warp_smem_bytes / G.stage_bytes);
    if (G.n_stages < 2) fail(FM_ERR_INVALID_ARG, "internal: pipeline stage does not fit");
    G.n_sites_total = (uint32_t)g->m->V;
    return G;
}

// Zeroed device counters for the dynamic batch scheduler: kSchedCounters counters in separate
// 128-byte lines per launch, handed out from a pool that is re-zeroed on the stream when it wraps.
struct CounterPool {
    uint32_t *d = nullptr;
    int device = -1;
    uint32_t next = 0;
    static constexpr uint32_t kLaunches = 64;
    static constexpr uint32_t kWordsPerLaunch = fm::kSchedCounters * fm::kSchedStrideWords;
    uint32_t *take(int dev) {
        if (device != dev) {  // a host thread normally stays on one device
            d = nullptr;
            d = static_cast<uint32_t *>(dev_alloc((size_t)kLaunches * kWordsPerLaunch * sizeof(uint32_t)));
            device = dev;
            next = kLaunches;
        }
        if (next == kLaunches) {
            CK(cudaMemsetAsync(d, 0, (size_t)kLaunches * kWordsPerLaunch * sizeof(uint32_t), stream()));
            next = 0;
        }
        return d + (size_t)(next++) * kWordsPerLaunch;
    }
};
thread_local CounterPool t_counters;

// bytes a plane pass reads for one group and site: allele row, tail words, called count
uint64_t plane_site_bytes(const fm::GroupPlanes &g) { return g.wq * 16u + g.tw * 4u + (g.cnt ? 4u : 0u); }

// Both plane passes use a whole SM's 224 KB of rings.  The dynamic shared-memory limit is a per-device function
// attribute: set it once per (kernel, device).
void allow_rings_once(const void *kern, int device) {
    static std::mutex mu;
    static std::set<std::pair<const void *, int>> done;
    std::lock_guard<std::mutex> lk(mu);
    if (!done.insert({kern, device}).second) return;
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(fm::kWarpsPerCta * fm::kWarpSmemBytes)));
}

void launch_chunked(fm::ChunkParams P, int device) {
    const fm::PassGeom &G = P.geom;
    if (G.n_batches == 0) return;
    P.geom.batch_counter = t_counters.take(device);
    allow_rings_once(reinterpret_cast<const void *>(fm::fm_k_plane_pass_chunked), device);
    const uint32_t grid = std::min<uint32_t>((uint32_t)sm_count(device), (G.n_batches + G.warps - 1) / G.warps);
    fm::fm_k_plane_pass_chunked<<<grid, G.warps * 32, (size_t)G.warps * G.warp_smem_bytes, stream()>>>(P);
    CK(cudaGetLastError());
    g_launches++;
    t_tim.stats_launches++;
    t_tim.stats_bytes = (uint64_t)(G.v_hi - G.v_lo) * plane_site_bytes(P.g);
}

fm::GroupPlanes planes_of(const fm_group *g);

// One launch of the row pass (fm_k_plane_pass_seq) over a list of segments (one per unit: independent (region, group)
// units; pair units: Hudson pairs over shared sites), planned once and launchable any number of times.
struct RowPlan {
    fm::RowParams P{};
    uint32_t lg = 0;
    bool inline_table = false, pair = false;
    uint64_t bytes = 0;  // plane bytes one launch reads
    DevBuf<fm::RowSeg> d_segs;
    DevBuf<uint32_t> d_prefix;
    std::vector<uint32_t> prefix;  // host copy: batches before unit u
};

// Fills rounds / b_lo of every segment, the geometry and the unit prefix; up to kMaxSeq segments go into the kernel
// parameters, a longer table is uploaded.  hud != nullptr: pair units (segments 2u and 2u + 1) with the Hudson
// epilogue hud[u] each, at most kMaxSeq / 2 of them.  Returns false when the segments cannot share a launch
// (column-chunked rows): the caller then goes unit by unit.
bool plan_rows(std::vector<fm::RowSeg> &segs, const std::vector<fm::HudsonEpilogue> *hud, RowPlan &plan) {
    const uint32_t gpu = hud ? 2u : 1u;  // segments per unit
    if (segs.empty() || segs.size() % gpu) return false;
    const size_t n_units = segs.size() / gpu;
    if (hud && (hud->size() != n_units || segs.size() > (size_t)fm::kMaxSeq))
        fail(FM_ERR_INVALID_ARG, "internal: pair units take one Hudson epilogue each and travel in the parameters");
    static const uint32_t step_target = env_u32("FM_STEP_BYTES", fm::kStepBytesTarget);
    uint32_t max_wq = 0;
    for (const fm::RowSeg &sg : segs) max_wq = std::max(max_wq, sg.g.wq);
    const uint32_t lg = row_lanes_log2(max_wq);
    if (lg >= 5) return false;
    uint32_t max_step = 0;
    plan.prefix.assign(n_units + 1, 0);
    uint64_t total = 0;
    plan.bytes = 0;
    for (size_t u = 0; u < n_units; ++u) {
        const fm::RowSeg &s0 = segs[u * gpu];
        const uint32_t nb = s0.v_hi > s0.v_lo ? (s0.v_hi + 31) / 32 - s0.v_lo / 32 : 0;
        for (uint32_t g = 0; g < gpu; ++g) {
            fm::RowSeg &sg = segs[u * gpu + g];
            if (sg.v_lo != s0.v_lo || sg.v_hi != s0.v_hi) return false;
            // several rounds of (32 >> lg) sites per step while the step stays near the target size
            const uint32_t round_bytes = sg.g.wq * 16u * (32u >> lg);
            uint32_t rounds = 1;
            while (rounds * 2 <= (1u << lg) && round_bytes * rounds * 2 <= step_target) rounds *= 2;
            sg.rounds = rounds;
            sg.b_lo = sg.v_lo / 32;
            max_step = std::max(max_step, round_bytes * rounds);
            plan.bytes += (uint64_t)(sg.v_hi - sg.v_lo) * plane_site_bytes(sg.g);
        }
        plan.prefix[u] = (uint32_t)total;
        total += nb;
        if (total >= (1ull << 31)) return false;
    }
    plan.prefix[n_units] = (uint32_t)total;
    fm::RowParams &P = plan.P;
    P = fm::RowParams{};
    fm::PassGeom &G = P.geom;
    G.warps = fm::kWarpsPerCta;
    G.warp_smem_bytes = fm::kWarpSmemBytes;
    G.stage_bytes = (max_step + 127u) & ~127u;
    G.n_stages = std::min<uint32_t>(fm::kMaxStages, G.warp_smem_bytes / G.stage_bytes);
    if (G.n_stages < 2) return false;
    G.n_batches = (uint32_t)total;
    plan.lg = lg;
    plan.pair = hud != nullptr;
    plan.inline_table = segs.size() <= (size_t)fm::kMaxSeq;
    if (plan.inline_table) {  // the whole table fits the kernel parameters
        std::copy(segs.begin(), segs.end(), P.inline_segs);
        std::copy(plan.prefix.begin(), plan.prefix.end(), P.inline_prefix);
        if (hud) std::copy(hud->begin(), hud->end(), P.inline_hud);
    } else {
        // (pageable sources are staged by the driver before cudaMemcpyAsync returns: the host vectors may go away)
        plan.d_segs.alloc(segs.size());
        plan.d_segs.upload(segs.data(), segs.size());
        plan.d_prefix.alloc(n_units + 1);
        plan.d_prefix.upload(plan.prefix.data(), n_units + 1);
        P.segs = plan.d_segs.p;
        P.unit_prefix = plan.d_prefix.p;
    }
    P.n_units = (uint32_t)n_units;
    return true;
}

template <int LG>
void launch_rows_t(const RowPlan &plan, const fm::RowParams &P, uint32_t grid, int device) {
    void (*kern)(fm::RowParams) = plan.pair           ? fm::fm_k_plane_pass_seq<LG, true, true>
                                  : plan.inline_table ? fm::fm_k_plane_pass_seq<LG, true, false>
                                                      : fm::fm_k_plane_pass_seq<LG, false, false>;
    allow_rings_once(reinterpret_cast<const void *>(kern), device);
    kern<<<grid, fm::kWarpsPerCta * 32, (size_t)fm::kWarpsPerCta * fm::kWarpSmemBytes, stream()>>>(P);
}

void launch_rows(const RowPlan &plan, int device) {
    if (plan.P.geom.n_batches == 0) return;
    fm::RowParams P = plan.P;
    P.geom.batch_counter = t_counters.take(device);
    const uint64_t warps_needed = (uint64_t)P.geom.n_batches * (plan.pair ? 2u : 1u);
    const uint32_t grid = (uint32_t)std::min<uint64_t>(sm_count(device), (warps_needed + fm::kWarpsPerCta - 1) / fm::kWarpsPerCta);
    switch (plan.lg) {
        case 0: launch_rows_t<0>(plan, P, grid, device); break;
        case 1: launch_rows_t<1>(plan, P, grid, device); break;
        case 2: launch_rows_t<2>(plan, P, grid, device); break;
        case 3: launch_rows_t<3>(plan, P, grid, device); break;
        case 4: launch_rows_t<4>(plan, P, grid, device); break;
        default: fail(FM_ERR_INVALID_ARG, "internal: bad row pass geometry");
    }
    CK(cudaGetLastError());
    g_launches++;
    t_tim.stats_launches++;
    t_tim.stats_bytes = plan.bytes;
}

// super-batches [s_lo, s_lo + n_super) that fm_k_reduce_partials folds for the batches of G
void super_range(const fm::PassGeom &G, uint32_t &s_lo, uint32_t &n_super) {
    s_lo = G.b_lo / fm::kSuperBatches;
    n_super = (G.b_lo + G.n_batches + fm::kSuperBatches - 1) / fm::kSuperBatches - s_lo;
}

// per-batch partials -> one row of nd doubles / nu u32 sums per super-batch, on the device
void launch_reduce(const double *pd, int nd, const uint32_t *pu, int nu, const fm::PassGeom &G, double *sd,
                   uint64_t *su, cudaStream_t st = nullptr) {
    if (!st) st = stream();
    uint32_t s_lo, n_super;
    super_range(G, s_lo, n_super);
    fm::fm_k_reduce_partials<<<(n_super + 3) / 4, 128, 0, st>>>(pd, nd, pu, nu, G.b_lo, G.n_batches,
                                                                 s_lo, n_super, sd, su);
    CK(cudaGetLastError());
    g_launches++;
}

// reduce per-batch partials to per-super-batch on device, finish sequentially on the host
void finish_partials(const double *d_pd, int nd, const uint32_t *d_pu, int nu, const fm::PassGeom &G,
                     double *out_d, uint64_t *out_u) {
    for (int i = 0; i < nd; ++i) out_d[i] = 0.0;
    for (int i = 0; i < nu; ++i) out_u[i] = 0;
    if (G.n_batches == 0) return;
    uint32_t s_lo, n_super;
    super_range(G, s_lo, n_super);
    DevBuf<double> sd((size_t)n_super * std::max(nd, 1));
    DevBuf<uint64_t> su((size_t)n_super * std::max(nu, 1));
    launch_reduce(d_pd, nd, d_pu, nu, G, sd.p, su.p);
    std::vector<double> hd((size_t)n_super * std::max(nd, 1));
    std::vector<uint64_t> hu((size_t)n_super * std::max(nu, 1));
    sd.download(hd.data(), (size_t)n_super * nd);
    su.download(hu.data(), (size_t)n_super * nu);
    CK(cudaStreamSynchronize(stream()));
    for (uint32_t s = 0; s < n_super; ++s) {  // fixed order: independent of grid / GPU count
        for (int i = 0; i < nd; ++i) out_d[i] += hd[(size_t)s * nd + i];
        for (int i = 0; i < nu; ++i) out_u[i] += hu[(size_t)s * nu + i];
    }
}

void set_tables(fm::DivEpilogue &e, const fm_group *g) {
    const size_t tn = (size_t)g->n + 1;
    e.tab_inv_n = g->d_tab;
    e.tab_scale = g->d_tab + tn;
    e.tab_theta = g->d_tab + 2 * tn;
}

fm::GroupPlanes planes_of(const fm_group *g) {
    return fm::GroupPlanes{g->d_allele, g->cnt_in ? g->d_cnt : nullptr, g->wq, g->n, g->d_tail_a, g->tw};
}

// where a pass over all sites caches its called counts: nowhere when K1 already wrote them
uint32_t *called_cache(fm_group *g) { return g->cnt_in ? nullptr : g->d_cnt; }

// the cached-count arrays of a biallelic group (d_cnt exists from creation on when K1 fills it)
void alloc_counts(fm_group *g) {
    const size_t V = std::max<size_t>(g->m->V, 1);
    if (!g->d_alt) g->d_alt = static_cast<uint32_t *>(dev_alloc(V * sizeof(uint32_t)));
    if (!g->d_cnt) g->d_cnt = static_cast<uint32_t *>(dev_alloc(V * sizeof(uint32_t)));
}

// K5a: mask / filtered-position bit per site, one word per batch
void launch_site_flags(const fm_matrix *m, uint32_t v_lo, uint32_t v_hi, uint32_t b_lo, uint32_t n_batches,
                       const int64_t *d_mask, uint32_t n_mask, const int64_t *d_filt, uint32_t n_filt,
                       uint32_t *d_flags, cudaStream_t st = nullptr) {
    if (!st) st = stream();
    const uint32_t fb = std::max(1u, std::min<uint32_t>((n_batches + 7) / 8, 8u * (uint32_t)sm_count(m->device)));
    fm::fm_k_site_flags<<<fb, 256, 0, st>>>(m->d_pos, v_lo, v_hi, b_lo, n_batches, d_mask, n_mask, d_filt,
                                                   n_filt, d_flags);
    CK(cudaGetLastError());
    g_launches++;
}

struct DivResult {
    double pi_sum;
    uint64_t seg, unc;
};

void ensure_counts(fm_group *g);

// Multi-allelic groups (fm_multi.cuh): diversity statistics of [v_lo, v_hi) from the cached
// per-allele counts.  form: FM_MULTI_DENSE (calculate_pi_dense general) or FM_MULTI_SPARSE.
DivResult run_multi_diversity(fm_group *g, uint32_t v_lo, uint32_t v_hi, int form, double *d_pi, double *d_theta,
                              const int64_t *d_mask, uint32_t n_mask, const int64_t *d_filt, uint32_t n_filt) {
    DivResult r{0.0, 0, 0};
    const fm::PassGeom G = batch_range(v_lo, v_hi);
    if (G.n_batches == 0) return r;
    DevBuf<double> part_pi(G.n_batches);
    DevBuf<uint32_t> part_u((size_t)G.n_batches * 2);
    fm::DivEpilogue e{};
    e.pi_out = d_pi;
    e.theta_out = d_theta;
    set_tables(e, g);
    e.part_pi = part_pi.p;
    e.part_u = part_u.p;
    DevBuf<uint32_t> flags;
    Timer tm;
    tm.start();
    if (d_pi && (d_mask || d_filt)) {
        flags.alloc(G.n_batches);
        launch_site_flags(g->m, v_lo, v_hi, G.b_lo, G.n_batches, d_mask, n_mask, d_filt, n_filt, flags.p);
        e.site_flags = flags.p;
    }
    const uint32_t blocks = std::min<uint32_t>((G.n_batches + 7) / 8, 8u * sm_count(g->m->device));
    fm::fm_k_multi_div_from_counts<<<blocks, 256, 0, stream()>>>(g->d_acount, g->d_cnt, 1u << g->n_bits, form, e, v_lo,
                                                                  v_hi, G.b_lo, G.n_batches);
    CK(cudaGetLastError());
    g_launches++;
    tm.stop();
    double od[1];
    uint64_t ou[2];
    finish_partials(part_pi.p, 1, part_u.p, 2, G, od, ou);
    t_tim.stats_ms += tm.ms();
    r.pi_sum = od[0];
    r.seg = ou[0];
    r.unc = ou[1];
    return r;
}

// per-allele counts of a multi-allelic group (K2m) + the general dense summary scalars
void ensure_multi_counts_locked(fm_group *g) {
    set_dev(g->m);
    const size_t V = g->m->V;
    const uint32_t A = 1u << g->n_bits;
    if (!g->d_acount) {
        g->d_acount = static_cast<uint32_t *>(dev_alloc(std::max<size_t>(V, 1) * A * sizeof(uint32_t)));
        g->d_cnt = static_cast<uint32_t *>(dev_alloc(std::max<size_t>(V, 1) * sizeof(uint32_t)));
    }
    if (V) {
        uint32_t lg = 0;
        while ((1u << lg) < std::min(g->wq, 32u)) ++lg;
        const uint32_t sps = 32u >> lg;
        const uint64_t warps_needed = ((uint64_t)V + sps - 1) / sps;
        const uint32_t blocks = (uint32_t)std::min<uint64_t>((warps_needed + 7) / 8, 16ull * sm_count(g->m->device));
        const size_t ps = std::max<size_t>(V, 1) * g->wq;
        Timer tm;
        tm.start();
        switch (g->n_bits) {
            case 2: fm::fm_k_allele_counts<2><<<blocks, 256, 0, stream()>>>(g->d_allele, ps, g->d_called, g->wq, g->n, lg, 0, (uint32_t)V, g->d_acount, g->d_cnt); break;
            case 3: fm::fm_k_allele_counts<3><<<blocks, 256, 0, stream()>>>(g->d_allele, ps, g->d_called, g->wq, g->n, lg, 0, (uint32_t)V, g->d_acount, g->d_cnt); break;
            default: fm::fm_k_allele_counts<4><<<blocks, 256, 0, stream()>>>(g->d_allele, ps, g->d_called, g->wq, g->n, lg, 0, (uint32_t)V, g->d_acount, g->d_cnt); break;
        }
        CK(cudaGetLastError());
        g_launches++;
        t_tim.stats_launches++;
        t_tim.stats_bytes = (uint64_t)V * g->wq * 16u * (g->n_bits + (g->d_called ? 1u : 0u));
        tm.stop();
        t_tim.stats_ms += tm.ms();
    }
    g->have_counts = true;  // run_multi_diversity reads the cached counts
    DivResult r = run_multi_diversity(g, 0, (uint32_t)V, FM_MULTI_DENSE, nullptr, nullptr, nullptr, 0, nullptr, 0);
    g->seg = r.seg;
    g->unc = r.unc;
    g->pi_sum = r.pi_sum;
}

// segment of the row pass: group g over [v_lo, v_hi) into the diversity epilogue e
fm::RowSeg div_seg(const fm_group *g, const fm::DivEpilogue &e, uint32_t v_lo, uint32_t v_hi) {
    fm::RowSeg s{};
    s.g = planes_of(g);
    s.div = e;
    s.v_lo = v_lo;
    s.v_hi = v_hi;
    s.n_sites_total = (uint32_t)g->m->V;
    return s;
}

// Run the diversity statistics for sites [v_lo, v_hi): fused plane pass when counts are not
// cached (optionally caching them when the range is the whole matrix), light kernel otherwise.
DivResult run_diversity(fm_group *g, uint32_t v_lo, uint32_t v_hi, int pi_form, double *d_pi,
                        double *d_theta, const int64_t *d_mask, uint32_t n_mask, const int64_t *d_filt,
                        uint32_t n_filt, bool store_counts) {
    if (g->n_bits > 1) {  // multi-allelic: always from the cached per-allele counts
        if (!g->have_counts) ensure_multi_counts_locked(g);
        return run_multi_diversity(g, v_lo, v_hi, pi_form == FM_PIFORM_COMPONENTS ? FM_MULTI_SPARSE : FM_MULTI_DENSE,
                                   d_pi, d_theta, d_mask, n_mask, d_filt, n_filt);
    }
    const fm::PassGeom G = batch_range(v_lo, v_hi);
    DivResult r{0.0, 0, 0};
    if (G.n_batches == 0) return r;
    DevBuf<double> part_pi(G.n_batches);
    DevBuf<uint32_t> part_u((size_t)G.n_batches * 2);
    fm::DivEpilogue e{};
    e.pi_out = d_pi;
    e.theta_out = d_theta;
    set_tables(e, g);
    DevBuf<uint32_t> flags;
    Timer tm;
    tm.start();
    if (d_pi && (d_mask || d_filt)) {  // K5a: mask / filtered-position bits, one word per batch
        flags.alloc(G.n_batches);
        launch_site_flags(g->m, v_lo, v_hi, G.b_lo, G.n_batches, d_mask, n_mask, d_filt, n_filt, flags.p);
        e.site_flags = flags.p;
    }
    e.pi_form = pi_form;
    e.part_pi = part_pi.p;
    e.part_u = part_u.p;
    if (g->have_counts) {
        const uint32_t blocks = std::min<uint32_t>((G.n_batches + 7) / 8, 8u * sm_count(g->m->device));
        fm::fm_k_div_from_counts<<<blocks, 256, 0, stream()>>>(g->d_alt, g->d_cnt, e, v_lo, v_hi,
                                                                G.b_lo, G.n_batches);
        CK(cudaGetLastError());
        g_launches++;
    } else {
        if (store_counts) {
            e.alt_out = g->d_alt;
            e.called_out = called_cache(g);
        }
        if (g->count_only) fail(FM_ERR_INVALID_ARG, "internal: a count-only group has no bitplanes to stream");
        std::vector<fm::RowSeg> segs{div_seg(g, e, v_lo, v_hi)};
        RowPlan plan;
        if (row_lanes_log2(g->wq) < 5 && plan_rows(segs, nullptr, plan))
            launch_rows(plan, g->m->device);
        else
            launch_chunked(fm::ChunkParams{planes_of(g), make_geom(g, v_lo, v_hi), e}, g->m->device);
    }
    tm.stop();
    double od[1];
    uint64_t ou[2];
    Timer tr;
    tr.start();
    finish_partials(part_pi.p, 1, part_u.p, 2, G, od, ou);
    r.pi_sum = od[0];
    r.seg = ou[0];
    r.unc = ou[1];
    tr.stop();
    t_tim.stats_ms += tm.ms();
    t_tim.reduce_ms += tr.ms();
    return r;
}

// Diversity statistics of several groups of one matrix over [v_lo, v_hi).  Groups whose counts are not cached yet
// and whose rows fit the row pass share ONE launch of it (fm_k_plane_pass_seq); everything else goes group by group
// through run_diversity.
bool run_diversity_multi(fm_group *const *gs, size_t n, uint32_t v_lo, uint32_t v_hi, int pi_form,
                         double *const *d_pi, double *const *d_theta, const int64_t *d_mask, uint32_t n_mask,
                         const int64_t *d_filt, uint32_t n_filt, DivResult *out, bool store_counts = false,
                         Timer *ext_tm = nullptr) {
    auto per_group = [&]() {
        for (size_t i = 0; i < n; ++i) {
            DivResult r = run_diversity(gs[i], v_lo, v_hi, pi_form, d_pi ? d_pi[i] : nullptr, d_theta ? d_theta[i] : nullptr,
                                        d_mask, n_mask, d_filt, n_filt, store_counts);
            if (out) out[i] = r;
        }
        return false;
    };
    bool fuse = v_hi > v_lo;
    for (size_t i = 0; i < n && fuse; ++i)
        fuse = !gs[i]->have_counts && gs[i]->m == gs[0]->m && gs[i]->n_bits == 1 && !gs[i]->count_only &&
               row_lanes_log2(gs[i]->wq) < 5;
    if (!fuse) return per_group();
    const fm::PassGeom G = batch_range(v_lo, v_hi);
    const bool tracks = d_pi != nullptr;
    const bool use_flags = tracks && (d_mask || d_filt);
    DevBuf<uint32_t> flags;
    if (use_flags) flags.alloc(G.n_batches);
    std::vector<DevBuf<double>> part_pi(n);
    std::vector<DevBuf<uint32_t>> part_u(n);
    std::vector<fm::RowSeg> segs(n);
    for (size_t i = 0; i < n; ++i) {
        part_pi[i].alloc(G.n_batches);
        part_u[i].alloc((size_t)G.n_batches * 2);
        fm::DivEpilogue e{};
        e.pi_out = tracks ? d_pi[i] : nullptr;
        e.theta_out = tracks ? d_theta[i] : nullptr;
        set_tables(e, gs[i]);
        e.site_flags = flags.p;
        e.pi_form = pi_form;
        e.part_pi = part_pi[i].p;
        e.part_u = part_u[i].p;
        if (store_counts) {  // cache the DensePopulationSummary arrays while the planes stream by
            e.alt_out = gs[i]->d_alt;
            e.called_out = called_cache(gs[i]);
        }
        segs[i] = div_seg(gs[i], e, v_lo, v_hi);
    }
    RowPlan plan;
    if (!plan_rows(segs, nullptr, plan)) return per_group();
    Timer own_tm;
    Timer &tm = ext_tm ? *ext_tm : own_tm;
    tm.start();
    if (use_flags) launch_site_flags(gs[0]->m, v_lo, v_hi, G.b_lo, G.n_batches, d_mask, n_mask, d_filt, n_filt, flags.p);
    launch_rows(plan, gs[0]->m->device);
    tm.stop();
    for (size_t i = 0; i < n && out; ++i) {  // out == nullptr: the caller only wants the tracks
        double od[1];
        uint64_t ou[2];
        finish_partials(part_pi[i].p, 1, part_u[i].p, 2, G, od, ou);
        out[i] = DivResult{od[0], ou[0], ou[1]};
    }
    if (out) t_tim.stats_ms += tm.ms();  // out == nullptr: the caller reads `ext_tm` after its own synchronise
    return true;  // one fused launch, timed by `tm`
}

void ensure_counts(fm_group *g) {
    std::lock_guard<std::mutex> lk(g->mu);
    if (g->have_counts) return;
    if (g->n_bits > 1) {
        ensure_multi_counts_locked(g);
        return;
    }
    set_dev(g->m);
    const size_t V = g->m->V;
    alloc_counts(g);
    DivResult r = run_diversity(g, 0, (uint32_t)V, FM_PIFORM_COUNTS, nullptr, nullptr, nullptr, 0,
                                nullptr, 0, /*store_counts=*/true);
    g->seg = r.seg;
    g->unc = r.unc;
    g->pi_sum = r.pi_sum;
    g->have_counts = true;
}

struct HudsonTotals {
    double num, den, dxy, pi1, pi2;
    uint64_t skipped, unc1, unc2;
};

// Hudson sums (and optional per-site outputs) for [v_lo, v_hi) from cached counts.
HudsonTotals run_hudson_counts(fm_group *g1, fm_group *g2, uint32_t v_lo, uint32_t v_hi, int variant,
                               fm::HudsonEpilogue e) {
    const fm::PassGeom G = batch_range(v_lo, v_hi);
    HudsonTotals t{0, 0, 0, 0, 0, 0, 0, 0};
    if (G.n_batches == 0) return t;
    DevBuf<double> pd((size_t)G.n_batches * 5);
    DevBuf<uint32_t> pu((size_t)G.n_batches * 3);
    e.variant = variant;
    e.part_d = pd.p;
    e.part_u = pu.p;
    Timer tm;
    tm.start();
    const uint32_t blocks = std::min<uint32_t>((G.n_batches + 7) / 8, 8u * sm_count(g1->m->device));
    if (g1->n_bits > 1) {
        if (variant < 0)
            fail(FM_ERR_UNSUPPORTED, "the summaries path does not exist for multi-allelic matrices (lib.rs:779)");
        if (g2->n_bits != g1->n_bits) fail(FM_ERR_INVALID_ARG, "groups of one pass must share a matrix");
        fm::fm_k_multi_hudson_from_counts<<<blocks, 256, 0, stream()>>>(
            g1->d_acount, g1->d_cnt, g2->d_acount, g2->d_cnt, 1u << g1->n_bits,
            variant == FM_HV_SPARSE ? FM_MULTI_SPARSE : FM_MULTI_DENSE, e, v_lo, v_hi, G.b_lo, G.n_batches);
    } else
        fm::fm_k_hudson_from_counts<<<blocks, 256, 0, stream()>>>(g1->d_alt, g1->d_cnt, g2->d_alt, g2->d_cnt,
                                                                   e, v_lo, v_hi, G.b_lo, G.n_batches);
    CK(cudaGetLastError());
    g_launches++;
    tm.stop();
    double od[5];
    uint64_t ou[3];
    finish_partials(pd.p, 5, pu.p, 3, G, od, ou);
    t_tim.stats_ms += tm.ms();
    t = HudsonTotals{od[0], od[1], od[2], od[3], od[4], ou[0], ou[1], ou[2]};
    return t;
}

void merge_intervals(const int64_t *iv, size_t n, std::vector<int64_t> &out) {
    std::vector<std::pair<int64_t, int64_t>> v;
    v.reserve(n);
    for (size_t i = 0; i < n; ++i)
        if (iv[2 * i + 1] > iv[2 * i]) v.emplace_back(iv[2 * i], iv[2 * i + 1]);
    std::sort(v.begin(), v.end());
    out.clear();
    for (auto &p : v) {
        if (!out.empty() && p.first <= out[out.size() - 1]) {
            if (p.second > out[out.size() - 1]) out[out.size() - 1] = p.second;
        } else {
            out.push_back(p.first);
            out.push_back(p.second);
        }
    }
}

int dense_variant(const fm_matrix *m) { return m->has_missing ? FM_HV_DENSE_MISSING : FM_HV_DENSE_NOMISSING; }

// 1-based output positions of sites [lo, lo + n) (stats.rs:747, 3004, 4746): small ranges are written by the host,
// large ones come from the device copy of the positions (one kernel + one D2H instead of a million-element host
// loop).  pos_out == NULL: the caller already knows the positions.  The copy is ordered on stream().
__global__ void fm_k_pos_plus1(const int64_t *__restrict__ pos, uint32_t lo, uint32_t n, int64_t *__restrict__ out) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) out[i] = pos[lo + i] + 1;
}
void download_positions_plus1(const fm_matrix *m, uint32_t lo, size_t n, int64_t *pos_out, DevBuf<int64_t> &scratch) {
    if (!pos_out || !n) return;
    if (n < 65536) {
        for (size_t i = 0; i < n; ++i) pos_out[i] = m->pos[lo + i] + 1;
        return;
    }
    scratch.alloc(n);
    fm_k_pos_plus1<<<(uint32_t)std::min<size_t>((n + 255) / 256, 2048), 256, 0, stream()>>>(m->d_pos, lo, (uint32_t)n, scratch.p);
    CK(cudaGetLastError());
    g_launches++;
    scratch.download(pos_out, n);
}

}  // namespace

// ------------------------------------------------------------------------------------ library
extern "C" {

const char *fm_last_error(void) { return t_err.c_str(); }
const char *fm_version(void) { return "ferromic_gpu 0.1.0 (sm_100a)"; }

fm_status fm_device_count(int *count) {
    return guarded([&] {
        if (!count) fail(FM_ERR_INVALID_ARG, "count is NULL");
        int n = 0;
        cudaError_t e = cudaGetDeviceCount(&n);
        if (e != cudaSuccess) {
            cudaGetLastError();
            n = 0;
        }
        *count = n;
    });
}

fm_status fm_set_device(int device) {
    return guarded([&] {
        require_device();
        if (!device_allowed(device))
            fail(FM_ERR_INVALID_ARG, "device is not in the allowed list (fm_set_devices / FERROMIC_GPU_DEVICES)");
        CK(cudaSetDevice(device));
        t_device_sel = device;
    });
}

fm_status fm_set_devices(const int *devices, size_t n) {
    return guarded([&] {
        if (n && !devices) fail(FM_ERR_INVALID_ARG, "devices is NULL");
        require_device();
        int count = 0;
        CK(cudaGetDeviceCount(&count));
        std::vector<int> v;
        for (size_t i = 0; i < n; ++i) {
            if (devices[i] < 0 || devices[i] >= count) fail(FM_ERR_INVALID_ARG, "device ordinal out of range");
            if (std::find(v.begin(), v.end(), devices[i]) == v.end()) v.push_back(devices[i]);
        }
        std::lock_guard<std::mutex> lk(g_dev_mu);
        g_devices_init = true;  // an explicit list overrides FERROMIC_GPU_DEVICES
        g_devices = v;          // n == 0: every visible device again
    });
}

fm_status fm_get_devices(int *devices_out, size_t capacity, size_t *n_out) {
    return guarded([&] {
        if (!n_out) fail(FM_ERR_INVALID_ARG, "n_out is NULL");
        int count = 0;
        if (cudaGetDeviceCount(&count) != cudaSuccess) {
            cudaGetLastError();
            count = 0;
        }
        std::lock_guard<std::mutex> lk(g_dev_mu);
        devices_init_locked();
        std::vector<int> v = g_devices;
        if (v.empty())
            for (int d = 0; d < count; ++d) v.push_back(d);
        *n_out = v.size();
        for (size_t i = 0; i < v.size() && i < capacity && devices_out; ++i) devices_out[i] = v[i];
    });
}

fm_status fm_synchronize(void) {
    return guarded([&] {
        require_device();
        CK(cudaStreamSynchronize(stream()));
    });
}

fm_status fm_trim_pool(void) {
    return guarded([&] {
        require_device();
        CK(cudaSetDevice(t_device));
        CK(cudaStreamSynchronize(stream()));
        cache_release_all(t_device);
    });
}

fm_status fm_timings_reset(void) {
    t_tim = fm_timings{};
    g_launches = 0;
    return FM_OK;
}
fm_status fm_timings_get(fm_timings *out) {
    if (!out) return FM_ERR_INVALID_ARG;
    *out = t_tim;
    out->kernel_launches = g_launches.load();
    return FM_OK;
}

// ------------------------------------------------------------------------------------ matrix
// Host position buffers of released matrices, kept for the next matrix: a fresh page-locked 8 MB buffer costs
// milliseconds (cudaHostAlloc), a fresh pageable one ~1.5 ms of page faults per 1M sites -- more than every kernel
// of a per-site call.
struct PosPool {
    std::mutex mu;
    std::vector<HostPos> free_list;
    HostPos take(size_t n) {
        std::lock_guard<std::mutex> lk(mu);
        size_t best = free_list.size();
        for (size_t i = 0; i < free_list.size(); ++i)
            if (free_list[i].cap >= n && (best == free_list.size() || free_list[i].cap < free_list[best].cap)) best = i;
        if (best == free_list.size()) return {};
        HostPos v = std::move(free_list[best]);
        free_list.erase(free_list.begin() + best);
        if (v.cap > 2 * n + ((size_t)1 << 18)) return {};  // far too large for this matrix: let it go
        return v;
    }
    void give(HostPos &&v) {
        if (!v.p || v.cap > ((size_t)1 << 28)) return;
        std::lock_guard<std::mutex> lk(mu);
        if (free_list.size() < 4) free_list.emplace_back(std::move(v));
    }
};
static PosPool g_pos_pool;

static fm_matrix *matrix_common(size_t V, size_t S, size_t ploidy, uint8_t max_allele,
                                const int64_t *positions) {
    if (ploidy != 0 && S != 0 && V > std::numeric_limits<size_t>::max() / S / ploidy)
        fail(FM_ERR_INVALID_ARG, "dense genotype matrix dimensions overflow");  // stats.rs:276-279
    if (V >= (1ull << 32) - 64) fail(FM_ERR_UNSUPPORTED, "more than 2^32 variants per matrix handle");
    if (S * ploidy >= (1ull << 32)) fail(FM_ERR_UNSUPPORTED, "row stride exceeds 2^32 entries");
    fm_matrix *m = new fm_matrix();
    m->device = t_device;
    m->V = V;
    m->S = S;
    m->ploidy = ploidy;
    m->stride = S * ploidy;
    m->max_allele = max_allele;
    m->plane_max_allele = max_allele;
    // copy the caller's positions and check that they ascend.  The vector comes from a small pool of buffers
    // handed back by released matrices (a fresh 8 MB vector costs ~1.5 ms of page faults per 1M sites, more than
    // every kernel of a per-site call); large copies are split over a few host threads.
    bool sorted = true;
    m->pos = g_pos_pool.take(V);
    if (positions) {
        m->pos.resize(V);
        int64_t *dst = m->pos.data();
        auto copy_check = [dst, positions](size_t lo, size_t hi) -> unsigned {
            std::memcpy(dst + lo, positions + lo, (hi - lo) * sizeof(int64_t));
            unsigned bad = 0;
            for (size_t i = std::max<size_t>(lo, 1); i < hi; ++i) bad |= (unsigned)(dst[i] < positions[i - 1]);
            return bad;
        };
        const size_t T = V >= ((size_t)1 << 18) ? 4 : 1;
        if (T == 1) {
            sorted = copy_check(0, V) == 0;
        } else {
            unsigned bad[4] = {0, 0, 0, 0};
            std::vector<std::thread> pool;
            const size_t slice = (V + T - 1) / T;
            for (size_t t = 1; t < T; ++t)
                pool.emplace_back([&, t] { bad[t] = copy_check(std::min(V, slice * t), std::min(V, slice * (t + 1))); });
            bad[0] = copy_check(0, std::min(V, slice));
            for (auto &th : pool) th.join();
            sorted = (bad[0] | bad[1] | bad[2] | bad[3]) == 0;
        }
    } else {
        m->pos.resize(V);
        for (size_t i = 0; i < V; ++i) m->pos[i] = (int64_t)i;
    }
    m->sorted = sorted;
    return m;
}

// max_allele > 15 on a resident u8 matrix: find the allele values that occur (called cells), rank them in ascending
// order (0 always first) and keep the value -> rank table on the device; K1 applies it while it bit-slices.  Real VCF
// cohorts have at most 8 distinct values (the parser's 7-ALT limit); more than 16 stay unsupported.
static void build_allele_remap(fm_matrix *m) {
    if (m->max_allele <= 15 || !m->d_data) return;
    const uint64_t total = (uint64_t)m->V * m->stride;
    DevBuf<uint32_t> d_present(8);
    CK(cudaMemsetAsync(d_present.p, 0, 32, stream()));
    if (total) {
        const uint32_t blocks = (uint32_t)std::min<uint64_t>((total + 255) / 256, 32ull * sm_count(m->device));
        fm::fm_k_allele_presence<<<blocks, 256, 0, stream()>>>(m->d_data, m->d_missing, total, m->in_band ? 1u : 0u,
                                                               d_present.p);
        CK(cudaGetLastError());
        g_launches++;
    }
    uint32_t present[8] = {};
    d_present.download(present, 8);
    CK(cudaStreamSynchronize(stream()));
    present[0] |= 1u;  // the reference allele keeps rank 0 whether it occurs or not
    uint8_t lut[256] = {};
    uint32_t rank = 0;
    for (uint32_t v = 0; v < 256; ++v)
        if ((present[v >> 5] >> (v & 31u)) & 1u) {
            lut[v] = (uint8_t)std::min<uint32_t>(rank, 255u);
            ++rank;
        }
    if (rank > 16) return;  // alloc_group reports the limit when a group is asked for
    m->plane_max_allele = (uint8_t)std::max<uint32_t>(rank - 1, 2u);  // max_allele > 1 keeps the general (multi-allelic) forms
    m->d_lut = static_cast<uint8_t *>(dev_alloc(256));
    CK(cudaMemcpyAsync(m->d_lut, lut, 256, cudaMemcpyHostToDevice, stream()));
    CK(cudaStreamSynchronize(stream()));
}

fm_status fm_matrix_create(const uint8_t *data, const uint64_t *missing, size_t V, size_t S,
                           size_t ploidy, uint8_t max_allele, const int64_t *positions,
                           fm_matrix **out) {
    return guarded([&] {
        FM_NVTX("fm_matrix_create (H2D u8)");
        if (!out) fail(FM_ERR_INVALID_ARG, "out is NULL");
        *out = nullptr;
        require_device();
        CK(cudaSetDevice(t_device));
        fm_matrix *m = matrix_common(V, S, ploidy, max_allele, positions);
        try {
            const size_t total = V * m->stride;
            if (total && !data) fail(FM_ERR_INVALID_ARG, "data is NULL");
            Timer tm;
            tm.start();
            uint8_t *dd = static_cast<uint8_t *>(dev_alloc(std::max<size_t>(total, 16)));
            m->d_data = dd;
            h2d(dd, data, total, stream());
            if (missing) {
                const size_t words = (total + 63) / 64;
                uint64_t *dm = static_cast<uint64_t *>(dev_alloc(std::max<size_t>(words, 2) * 8));
                m->d_missing = dm;
                m->has_missing = true;
                h2d(dm, missing, words * 8, stream());
            }
            m->d_pos = static_cast<int64_t *>(dev_alloc(std::max<size_t>(V, 1) * 8));
            if (V) CK(cudaMemcpyAsync(m->d_pos, m->pos.data(), V * 8, cudaMemcpyHostToDevice, stream()));
            tm.stop();
            t_tim.h2d_ms += tm.ms();
            build_allele_remap(m);
        } catch (...) {
            fm_matrix_release(m);
            throw;
        }
        *out = m;
    });
}

fm_status fm_matrix_create_inband(const uint8_t *data, size_t V, size_t S, size_t ploidy, uint8_t max_allele,
                                  const int64_t *positions, fm_matrix **out) {
    return guarded([&] {
        if (!out) fail(FM_ERR_INVALID_ARG, "out is NULL");
        *out = nullptr;
        if (max_allele > 127) fail(FM_ERR_INVALID_ARG, "in-band missingness needs allele indices <= 127");
        require_device();
        CK(cudaSetDevice(t_device));
        fm_matrix *m = matrix_common(V, S, ploidy, max_allele, positions);
        m->has_missing = true;
        m->in_band = true;
        try {
            const size_t total = V * m->stride;
            if (total && !data) fail(FM_ERR_INVALID_ARG, "data is NULL");
            Timer tm;
            tm.start();
            uint8_t *dd = static_cast<uint8_t *>(dev_alloc(std::max<size_t>(total, 16)));
            m->d_data = dd;
            h2d(dd, data, total, stream());
            m->d_pos = static_cast<int64_t *>(dev_alloc(std::max<size_t>(V, 1) * 8));
            if (V) CK(cudaMemcpyAsync(m->d_pos, m->pos.data(), V * 8, cudaMemcpyHostToDevice, stream()));
            tm.stop();
            t_tim.h2d_ms += tm.ms();
            build_allele_remap(m);
        } catch (...) {
            fm_matrix_release(m);
            throw;
        }
        *out = m;
    });
}

fm_status fm_matrix_create_device(const uint8_t *d_data, const uint64_t *d_missing, size_t V, size_t S,
                                  size_t ploidy, uint8_t max_allele, const int64_t *positions,
                                  fm_matrix **out) {
    return guarded([&] {
        if (!out) fail(FM_ERR_INVALID_ARG, "out is NULL");
        *out = nullptr;
        require_device();
        CK(cudaSetDevice(t_device));
        if ((reinterpret_cast<uintptr_t>(d_data) & 15u) || (reinterpret_cast<uintptr_t>(d_missing) & 7u))
            fail(FM_ERR_INVALID_ARG, "device matrix must be 16-byte aligned (bitmap 8-byte aligned)");
        fm_matrix *m = matrix_common(V, S, ploidy, max_allele, positions);
        m->owns = false;
        m->d_data = d_data;
        m->d_missing = d_missing;
        m->has_missing = d_missing != nullptr;
        try {
            m->d_pos = static_cast<int64_t *>(dev_alloc(std::max<size_t>(V, 1) * 8));
            if (V) CK(cudaMemcpyAsync(m->d_pos, m->pos.data(), V * 8, cudaMemcpyHostToDevice, stream()));
            CK(cudaStreamSynchronize(stream()));
            build_allele_remap(m);
        } catch (...) {
            fm_matrix_release(m);
            throw;
        }
        *out = m;
    });
}

fm_status fm_matrix_retain(fm_matrix *m) {
    if (!m) return FM_ERR_INVALID_ARG;
    m->refs++;
    return FM_OK;
}

fm_status fm_matrix_release(fm_matrix *m) {
    if (!m) return FM_OK;
    if (--m->refs == 0) {
        cudaSetDevice(m->device);
        if (m->owns) {
            dev_free(m->d_data);
            dev_free(m->d_missing);
        }
        dev_free(m->d_abits);
        dev_free(m->d_cbits);
        dev_free(m->d_lut);
        dev_free(m->d_pos);
        g_pos_pool.give(std::move(m->pos));
        delete m;
    }
    return FM_OK;
}

fm_status fm_matrix_info(const fm_matrix *m, size_t *V, size_t *S, size_t *ploidy, uint8_t *max_allele,
                         int *has_missing) {
    if (!m) return FM_ERR_INVALID_ARG;
    if (V) *V = m->V;
    if (S) *S = m->S;
    if (ploidy) *ploidy = m->ploidy;
    if (max_allele) *max_allele = m->max_allele;
    if (has_missing) *has_missing = m->has_missing;
    return FM_OK;
}

// ------------------------------------------------------------------------------------ group
// Allocate a group's bitplanes and lookup tables for the columns listed in `off` (sorted, unique).
// Can a warp stage one u8 row (+ its bitmap slice) in shared memory?  (row-staged K1 v2)
static size_t repack_warp_smem(const fm_matrix *m, uint32_t *row_buf_out, uint32_t *bit_buf_out) {
    // packed rows arrive as bit words: neither the u8 row nor the bitmap slice is staged
    const size_t row_buf = m->packed ? 0 : ((m->stride + 15) & ~(size_t)15) + 32;
    const size_t bit_buf = (!m->packed && m->has_missing && !m->in_band) ? ((m->stride + 63) / 64 + 2) * 8 : 0;
    // full-row allele / called bit words + one group's allele plane row while it is assembled
    // (+ 4 padding words: the compress fragments or a zero into the word after the last one)
    const size_t cnt_buf = 2 * ((m->stride + 31) / 32 + 1) * 4 + (((m->stride + 127) / 128) * 4 + 4) * 4;
    if (row_buf_out) *row_buf_out = (uint32_t)row_buf;
    if (bit_buf_out) *bit_buf_out = (uint32_t)bit_buf;
    return (row_buf + bit_buf + cnt_buf + 15) & ~(size_t)15;
}
static size_t repack_smem_limit(const fm_matrix *m) { return m->packed ? 100 * 1024 : 24 * 1024; }
static bool row_fits_smem(const fm_matrix *m) { return repack_warp_smem(m, nullptr, nullptr) <= repack_smem_limit(m); }

// counts_slab: when non-null, a count-only group takes its alt / called arrays from the caller's slab (a W&C
// partition allocates ONE block for all its groups: 54 separate cudaMallocs of 40 MB were 0.3 s of a cold
// fm_partition_create over 10M sites, two orders of magnitude more than the count kernel itself)
static fm_group *alloc_group(fm_matrix *m, std::vector<uint32_t> &&off, bool count_only = false,
                             uint32_t *counts_slab = nullptr) {
    uint32_t n_bits = 1;
    while ((1u << n_bits) <= m->plane_max_allele) ++n_bits;
    if (n_bits > 4)
        fail(FM_ERR_UNSUPPORTED,
             "more than 16 distinct allele values (or allele indices above 15 on a streamed / device-owned matrix) are "
             "not supported on the GPU path");
    set_dev(m);
    fm_group *g = new fm_group();
    g->m = m;
    fm_matrix_retain(m);
    try {
        g->off = std::move(off);
        g->n = (uint32_t)g->off.size();
        g->wq = std::max<uint32_t>(1, (g->n + 127) / 128);
        g->n_bits = n_bits;
        g->count_only = count_only && n_bits == 1 && row_fits_smem(m);
        {
            // tail layout when the padded last word would waste more than a quarter of itself and the group is
            // certain to be written by the compress plans (the only writer that knows the layout)
            static const uint32_t no_tail = env_u32("FM_NO_TAIL", 0);
            const uint32_t tail_bits = g->n % 128;
            const uint32_t tw = (tail_bits + 31) / 32;
            // worth it when the row shrinks by at least 2 % (the tail words cost tw extra loads per site in the
            // epilogue: 2504 haplotypes = 19 words + 72 bits would save 4 of 320 bytes and ran 3 % slower)
            if (!no_tail && n_bits == 1 && !g->count_only && row_fits_smem(m) && g->n >= 128 &&
                tail_bits != 0 && tail_bits <= 96 && (16u - 4u * tw) * 50u >= 16u * g->wq) {
                g->wq = g->n / 128;
                g->tw = tw;
            }
        }
        const size_t plane_u4 = std::max<size_t>(m->V, 1) * g->wq;
        if (g->count_only && counts_slab) {
            g->d_alt = counts_slab;  // interior pointers: dev_free ignores them, the partition frees the slab
            g->d_cnt = counts_slab + std::max<size_t>(m->V, 1);
        } else if (g->count_only) {
            g->d_alt = static_cast<uint32_t *>(dev_alloc(std::max<size_t>(m->V, 1) * sizeof(uint32_t)));
            g->d_cnt = static_cast<uint32_t *>(dev_alloc(std::max<size_t>(m->V, 1) * sizeof(uint32_t)));
        } else {
            g->d_allele = static_cast<uint4 *>(dev_alloc(plane_u4 * 16 * n_bits));
            // biallelic groups keep the called count per site instead of a called plane (K1 fills it)
            g->cnt_in = m->has_missing && n_bits == 1;
            if (g->cnt_in) g->d_cnt = static_cast<uint32_t *>(dev_alloc(std::max<size_t>(m->V, 1) * sizeof(uint32_t)));
            else if (m->has_missing) g->d_called = static_cast<uint4 *>(dev_alloc(plane_u4 * 16));
            if (g->tw) g->d_tail_a = static_cast<uint32_t *>(dev_alloc(std::max<size_t>(m->V, 1) * g->tw * 4));
        }
        // per-n tables: 1/n, n/(n-1) (stats.rs:2728-2732) and 1/H_{n-1} with the harmonic number
        // by forward summation exactly like stats.rs:4234-4240 / 4718-4719
        const size_t tn = (size_t)g->n + 1;
        std::vector<double> T(3 * tn, 0.0);
        double hsum = 0.0;  // H_{k-1} while visiting k
        for (size_t k = 1; k < tn; ++k) {
            const double kd = (double)k;
            T[k] = 1.0 / kd;
            T[tn + k] = kd / (kd - 1.0);
            T[2 * tn + k] = hsum > 0.0 ? 1.0 / hsum : 0.0;
            hsum += 1.0 / kd;
        }
        g->d_tab = static_cast<double *>(dev_alloc(T.size() * 8));
        CK(cudaMemcpyAsync(g->d_tab, T.data(), T.size() * 8, cudaMemcpyHostToDevice, stream()));
        g->d_off = static_cast<uint32_t *>(dev_alloc(std::max<size_t>(g->n, 1) * 4));
        if (g->n) CK(cudaMemcpyAsync(g->d_off, g->off.data(), (size_t)g->n * 4, cudaMemcpyHostToDevice, stream()));
        CK(cudaStreamSynchronize(stream()));  // T and off are host temporaries / may be moved
    } catch (...) {
        fm_group_release(g);
        throw;
    }
    return g;
}

// K1 for rows [v_lo, v_hi) of a set of groups of one matrix: `data` / `missing` point at the u8 row
// v_base and at the bitmap word word_base (resident matrix: v_base = word_base = 0; streaming
// ingest: the staged chunk).  Rows that fit a warp's shared-memory slice take the row-staged
// multi-group kernel (the u8 matrix is read once for all groups); wider rows (biobank cohorts)
// fall back to the per-group gather kernel.
struct RepackSet {  // device-resident descriptor tables of the groups one launch repacks / counts
    std::vector<fm_group *> gs;        // every group
    std::vector<fm_group *> plane_gs;  // groups that keep bitplanes
    fm::RepackGroup *d_desc = nullptr;
    // count-only groups: sparse (row word, mask) membership lists
    fm::CountTable ct{};
    uint32_t *d_ent = nullptr;         // ent_start | ent_word | ent_mask
    uint32_t **d_outs = nullptr;       // alt_out[n] | cnt_out[n]
    uint4 *d_plan = nullptr;           // compress plans of the biallelic plane groups (two uint4 per touched row word)
    bool need_row_bits = false;
    void build(const std::vector<fm_group *> &groups) {
        gs = groups;
        if (gs.empty()) return;
        const fm_matrix *m = gs[0]->m;
        std::vector<fm::RepackGroup> h;
        std::vector<uint32_t> ent_start{0}, ent_word, ent_mask;
        std::vector<uint32_t *> outs_a, outs_c;
        std::vector<uint32_t> plan;            // 8 words per entry
        std::vector<size_t> plan_at, plan_len;  // per plane group: first entry, entries (0 = no plan)
        const bool staged = row_fits_smem(m);
        for (fm_group *g : gs) {
            if (g->count_only) {
                for (size_t k = 0; k < g->off.size();) {  // offsets are sorted: one entry per row word
                    const uint32_t w = g->off[k] >> 5;
                    uint32_t mask = 0;
                    while (k < g->off.size() && (g->off[k] >> 5) == w) mask |= 1u << (g->off[k++] & 31u);
                    ent_word.push_back(w);
                    ent_mask.push_back(mask);
                }
                ent_start.push_back((uint32_t)ent_word.size());
                outs_a.push_back(g->d_alt);
                outs_c.push_back(g->d_cnt);
            } else {
                plane_gs.push_back(g);
                h.push_back(fm::RepackGroup{g->d_off, g->n, g->wq, g->n_bits, reinterpret_cast<uint32_t *>(g->d_allele),
                                            reinterpret_cast<uint32_t *>(g->d_called),
                                            std::max<size_t>(m->V, 1) * g->wq * 4, nullptr, nullptr, nullptr, 0,
                                            g->d_tail_a, g->tw, g->cnt_in ? g->d_cnt : nullptr});
                plan_at.push_back(plan.size() / 8);
                size_t ne = 0;
                if (g->n_bits == 1 && (staged || m->packed)) {
                    uint32_t pos = 0;
                    for (size_t k = 0; k < g->off.size(); ++ne) {  // offsets are sorted: one entry per row word
                        const uint32_t w = g->off[k] >> 5;
                        uint32_t mask = 0;
                        while (k < g->off.size() && (g->off[k] >> 5) == w) mask |= 1u << (g->off[k++] & 31u);
                        uint32_t mv[5], mm = mask, mk = ~mask << 1;  // Hacker's Delight 7-4: compress move masks
                        for (int i = 0; i < 5; ++i) {
                            uint32_t mp = mk ^ (mk << 1);
                            mp ^= mp << 2;
                            mp ^= mp << 4;
                            mp ^= mp << 8;
                            mp ^= mp << 16;
                            mv[i] = mp & mm;
                            mm = (mm ^ mv[i]) | (mv[i] >> (1u << i));
                            mk &= ~mp;
                        }
                        const uint32_t ent[8] = {w, mask, pos, mv[0], mv[1], mv[2], mv[3], mv[4]};
                        plan.insert(plan.end(), ent, ent + 8);
                        pos += (uint32_t)__builtin_popcount(mask);
                    }
                }
                plan_len.push_back(ne);
            }
        }
        // every biallelic plane group takes the plan path when plans are in use -- also an empty group (no entries):
        // the direct and packed kernels compile without the ballot gathers
        const bool plans_on = staged || m->packed;
        bool any_bial = false;
        for (const fm::RepackGroup &rg : h) any_bial = any_bial || rg.n_bits == 1;
        if (plans_on && any_bial && plan.empty()) plan.resize(8, 0u);
        if (!plan.empty()) {
            d_plan = static_cast<uint4 *>(dev_alloc(plan.size() * 4));
            CK(cudaMemcpyAsync(d_plan, plan.data(), plan.size() * 4, cudaMemcpyHostToDevice, stream()));
            for (size_t i = 0; i < h.size(); ++i)
                if (plan_len[i] || (plans_on && h[i].n_bits == 1)) {
                    h[i].plan = d_plan + 2 * plan_at[i];
                    h[i].n_ent = (uint32_t)plan_len[i];
                }
            need_row_bits = true;
        }
        if (!h.empty()) {
            d_desc = static_cast<fm::RepackGroup *>(dev_alloc(h.size() * sizeof(fm::RepackGroup)));
            CK(cudaMemcpyAsync(d_desc, h.data(), h.size() * sizeof(fm::RepackGroup), cudaMemcpyHostToDevice, stream()));
        }
        const uint32_t ncg = (uint32_t)outs_a.size();
        if (ncg) need_row_bits = true;
        if (ncg) {
            const size_t ne = ent_word.size();
            std::vector<uint32_t> packed;
            packed.insert(packed.end(), ent_start.begin(), ent_start.end());
            packed.insert(packed.end(), ent_word.begin(), ent_word.end());
            packed.insert(packed.end(), ent_mask.begin(), ent_mask.end());
            d_ent = static_cast<uint32_t *>(dev_alloc(packed.size() * 4));
            CK(cudaMemcpyAsync(d_ent, packed.data(), packed.size() * 4, cudaMemcpyHostToDevice, stream()));
            std::vector<uint32_t *> outs(outs_a);
            outs.insert(outs.end(), outs_c.begin(), outs_c.end());
            d_outs = static_cast<uint32_t **>(dev_alloc(outs.size() * sizeof(uint32_t *)));
            CK(cudaMemcpyAsync(d_outs, outs.data(), outs.size() * sizeof(uint32_t *), cudaMemcpyHostToDevice, stream()));
            ct.ent_start = d_ent;
            ct.ent_word = d_ent + ncg + 1;
            ct.ent_mask = d_ent + ncg + 1 + ne;
            ct.alt_out = d_outs;
            ct.cnt_out = d_outs + ncg;
            ct.n_groups = ncg;
            CK(cudaStreamSynchronize(stream()));
            return;
        }
        CK(cudaStreamSynchronize(stream()));
    }
    void release() {
        dev_free(d_desc);
        dev_free(d_ent);
        dev_free(d_outs);
        dev_free(d_plan);
        d_plan = nullptr;
        need_row_bits = false;
        d_desc = nullptr;
        d_ent = nullptr;
        d_outs = nullptr;
        ct = fm::CountTable{};
        gs.clear();
        plane_gs.clear();
    }
};

static void launch_repack(const RepackSet &set, const uint8_t *data, size_t data_bytes, const uint64_t *missing,
                          uint32_t v_base, uint64_t word_base, uint32_t v_lo, uint32_t v_hi, cudaStream_t st) {
    const std::vector<fm_group *> &gs = set.gs;
    if (gs.empty() || v_hi <= v_lo) return;
    const fm_matrix *m = gs[0]->m;
    uint32_t row_buf = 0, bit_buf = 0;
    uint32_t warp_smem = (uint32_t)repack_warp_smem(m, &row_buf, &bit_buf);
    if (m->packed) {  // K1p: groups from the resident packed rows (data / missing are unused)
        if (warp_smem > repack_smem_limit(m))
            fail(FM_ERR_UNSUPPORTED, "packed rows wider than the repack kernel's shared-memory slice");
        for (const fm_group *g : set.plane_gs)
            if (g->n_bits != 1 || !set.d_plan) fail(FM_ERR_INVALID_ARG, "internal: packed rows need compress plans");
        (void)row_buf;
        (void)bit_buf;
        const uint32_t warps = std::max(1u, std::min(8u, (200u * 1024u) / warp_smem));
        const size_t smem = (size_t)warps * warp_smem;
        static std::once_flag attr_once_p;
        std::call_once(attr_once_p, [] {
            cudaFuncSetAttribute(fm::fm_k_repack_rows<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        });
        const uint32_t rows = v_hi - v_lo;
        const uint32_t per_sm = std::max(1u, std::min(8u, (uint32_t)((220u * 1024u) / smem)));
        const uint32_t blocks = std::max(1u, std::min<uint32_t>((rows + warps - 1) / warps,
                                                                per_sm * (uint32_t)sm_count(m->device)));
        const fm::PackedRows pk{m->d_abits, m->d_cbits, m->rw};
        fm::fm_k_repack_rows<2, true><<<blocks, warps * 32, smem, st>>>(nullptr, 0, nullptr, m->stride, 0, 0, v_lo, v_hi,
                                                               set.d_desc, (uint32_t)set.plane_gs.size(), warp_smem, 0, 0,
                                                               set.ct, 0u, 1u, 0u, pk, nullptr);
        CK(cudaGetLastError());
        g_launches++;
        return;
    }
    if (warp_smem <= 24 * 1024) {
        // direct mode: nothing reads the raw bytes of the row after the full-row bit words are built
        static const uint32_t no_direct = env_u32("FM_REPACK_STAGED", 0);
        bool direct = !no_direct && set.need_row_bits && m->stride % 16 == 0 &&
                      (reinterpret_cast<uintptr_t>(data) & 15u) == 0;
        for (const fm_group *g : set.plane_gs) direct = direct && g->n_bits == 1;  // ballot gathers read the staged row
        if (direct && !set.plane_gs.empty() && !set.d_plan) direct = false;
        if (direct) {
            warp_smem -= row_buf;
            row_buf = 0;
        }
        const uint32_t warps = std::max(1u, std::min(8u, (200u * 1024u) / warp_smem));
        const size_t smem = (size_t)warps * warp_smem;
        static std::once_flag attr_once;
        std::call_once(attr_once, [] {
            cudaFuncSetAttribute(fm::fm_k_repack_rows<0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
            cudaFuncSetAttribute(fm::fm_k_repack_rows<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
            cudaFuncSetAttribute(fm::fm_k_repack_rows<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
            cudaFuncSetAttribute(fm::fm_k_repack_rows<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        });
        const uint32_t rows = v_hi - v_lo;
        const uint32_t per_sm = std::max(1u, std::min(8u, (uint32_t)((220u * 1024u) / smem)));
        const uint32_t blocks = std::max(1u, std::min<uint32_t>((rows + warps - 1) / warps,
                                                                per_sm * (uint32_t)sm_count(m->device)));
        const bool bial = m->plane_max_allele <= 1;
        auto go = [&](auto kern) {
            kern<<<blocks, warps * 32, smem, st>>>(data, data_bytes, missing, m->stride, v_base, word_base, v_lo, v_hi,
                                                   set.d_desc, (uint32_t)set.plane_gs.size(), warp_smem, row_buf, bit_buf,
                                                   set.ct, m->in_band ? 1u : 0u, set.need_row_bits ? 1u : 0u,
                                                   direct ? 1u : 0u, fm::PackedRows{nullptr, nullptr, 0}, m->d_lut);
        };
        if (direct) {
            if (bial) go(fm::fm_k_repack_rows<1, true>);
            else go(fm::fm_k_repack_rows<1, false>);
        } else {
            if (bial) go(fm::fm_k_repack_rows<0, true>);
            else go(fm::fm_k_repack_rows<0, false>);
        }
        CK(cudaGetLastError());
        g_launches++;
        return;
    }
    if (set.ct.n_groups) fail(FM_ERR_INVALID_ARG, "internal: count-only groups need the row-staged repack");
    for (const fm_group *g : set.plane_gs)
        if (g->tw) fail(FM_ERR_INVALID_ARG, "internal: a tail-layout group needs the plan path of the row-staged repack");
    for (const fm_group *g : set.plane_gs) {
        // the kernel adds the called members of every row slice to d_cnt
        if (g->cnt_in) CK(cudaMemsetAsync(g->d_cnt + v_lo, 0, (size_t)(v_hi - v_lo) * sizeof(uint32_t), st));
        const uint32_t blocks = (uint32_t)std::min<uint64_t>(
            (uint64_t)sm_count(m->device) * 8,
            std::max<uint64_t>(1, ((uint64_t)(v_hi - v_lo) * ((g->wq * 4 + 31) / 32) + 7) / 8));
        fm::fm_k_repack<<<blocks, 256, 0, st>>>(data, missing, m->stride, g->d_off, g->n, g->wq, v_base, word_base, v_lo,
                                                v_hi, reinterpret_cast<uint32_t *>(g->d_allele),
                                                reinterpret_cast<uint32_t *>(g->d_called),
                                                g->cnt_in ? g->d_cnt : nullptr, g->n_bits,
                                                std::max<size_t>(m->V, 1) * g->wq * 4, m->in_band ? 1u : 0u, m->d_lut);
        CK(cudaGetLastError());
        g_launches++;
    }
}

// Repack the resident matrix into freshly allocated groups (one pass over the u8 rows for all).
static void repack_resident(fm_matrix *m, const std::vector<fm_group *> &gs) {
    if (!m->V || gs.empty()) return;
    RepackSet set;
    set.build(gs);
    Timer tm;
    tm.start();
    try {
        launch_repack(set, m->d_data, m->V * m->stride, m->d_missing, 0, 0, 0, (uint32_t)m->V, stream());
        tm.stop();
        t_tim.repack_ms += tm.ms();
        CK(cudaStreamSynchronize(stream()));
        for (fm_group *g : gs)
            if (g->count_only) g->have_counts = true;
    } catch (...) {
        set.release();
        throw;
    }
    set.release();
}

// Repack the resident matrix columns listed in `off` into a new group's bitplanes.
static fm_group *make_group(fm_matrix *m, std::vector<uint32_t> &&off) {
    if (m->streamed && !m->packed)
        fail(FM_ERR_UNSUPPORTED,
             "this matrix was ingested in streaming mode (its u8 rows are not resident): declare groups "
             "with fm_ingest_add_group / fm_ingest_add_partition before fm_ingest_rows");
    fm_group *g = alloc_group(m, std::move(off));
    try {
        repack_resident(m, {g});
    } catch (...) {
        fm_group_release(g);
        throw;
    }
    return g;
}

// DenseMembership::build (stats.rs:1251-1284): sorted, de-duplicated offsets
static std::vector<uint32_t> membership_offsets(const fm_matrix *m, const uint64_t *sample_idx, const uint8_t *side,
                                                size_t n) {
    std::vector<uint8_t> left(m->S, 0), right(m->S, 0);
    std::vector<uint32_t> off;
    off.reserve(n);
    for (size_t i = 0; i < n; ++i) {
        const uint64_t s = sample_idx[i];
        if (s >= m->S) continue;
        if (side[i] == 0) {
            if (!left[s]) {
                left[s] = 1;
                off.push_back((uint32_t)(s * m->ploidy));
            }
        } else {
            if (m->ploidy <= 1) continue;
            if (!right[s]) {
                right[s] = 1;
                off.push_back((uint32_t)(s * m->ploidy + 1));
            }
        }
    }
    std::sort(off.begin(), off.end());
    return off;
}

// SubpopulationMembership (stats.rs:1093-1150): Left -> genotype[0], Right -> genotype[1];
// slot n_groups collects the haplotypes without a group
static std::vector<std::vector<uint32_t>> partition_columns(const fm_matrix *m, const uint16_t *left,
                                                            const uint16_t *right, size_t n_samples,
                                                            size_t n_groups) {
    std::vector<std::vector<uint32_t>> cols(n_groups + 1);
    const size_t P = m->ploidy;
    for (size_t s = 0; s < m->S; ++s) {
        for (size_t k = 0; k < P; ++k) {
            uint16_t g = 0xFFFF;
            if (s < n_samples) {
                if (k == 0) g = left[s];
                else if (k == 1) g = right[s];
            }
            const size_t slot = (g != 0xFFFF && g < n_groups) ? g : n_groups;
            cols[slot].push_back((uint32_t)(s * P + k));
        }
    }
    return cols;
}

fm_status fm_group_create(fm_matrix *m, const uint64_t *sample_idx, const uint8_t *side, size_t n,
                          fm_group **out) {
    return guarded([&] {
        FM_NVTX("fm_group_create (K1 repack)");
        if (!out || !m) fail(FM_ERR_INVALID_ARG, "NULL argument");
        *out = nullptr;
        if (n && (!sample_idx || !side)) fail(FM_ERR_INVALID_ARG, "haplotype arrays are NULL");
        require_device();
        std::vector<uint32_t> off = membership_offsets(m, sample_idx, side, n);
        *out = make_group(m, std::move(off));
    });
}

fm_status fm_groups_create(fm_matrix *m, const uint64_t *sample_idx, const uint8_t *side, const size_t *group_sizes,
                           size_t n_groups, fm_group **out) {
    return guarded([&] {
        FM_NVTX("fm_groups_create (K1 repack)");
        if (!out || !m) fail(FM_ERR_INVALID_ARG, "NULL argument");
        for (size_t g = 0; g < n_groups; ++g) out[g] = nullptr;
        if (n_groups && !group_sizes) fail(FM_ERR_INVALID_ARG, "group_sizes is NULL");
        require_device();
        if (m->streamed && !m->packed)
            fail(FM_ERR_UNSUPPORTED, "this matrix was ingested in streaming mode: declare groups with fm_ingest_add_group");
        std::vector<fm_group *> gs;
        try {
            size_t at = 0;
            for (size_t g = 0; g < n_groups; ++g) {
                const size_t n = group_sizes[g];
                if (n && (!sample_idx || !side)) fail(FM_ERR_INVALID_ARG, "haplotype arrays are NULL");
                gs.push_back(alloc_group(m, membership_offsets(m, sample_idx + at, side + at, n)));
                at += n;
            }
            repack_resident(m, gs);  // ONE pass over the u8 rows for all groups
        } catch (...) {
            for (fm_group *g : gs) fm_group_release(g);
            throw;
        }
        for (size_t g = 0; g < n_groups; ++g) out[g] = gs[g];
    });
}

fm_status fm_group_release(fm_group *g) {
    if (!g) return FM_OK;
    if (g->m) cudaSetDevice(g->m->device);
    dev_free(g->d_allele);
    dev_free(g->d_called);
    dev_free(g->d_tail_a);
    dev_free(g->d_tab);
    dev_free(g->d_off);
    dev_free(g->d_alt);
    dev_free(g->d_cnt);
    dev_free(g->d_acount);
    fm_matrix_release(g->m);
    delete g;
    return FM_OK;
}

fm_status fm_group_capacity(const fm_group *g, size_t *cap) {
    if (!g || !cap) return FM_ERR_INVALID_ARG;
    *cap = g->n;
    return FM_OK;
}

fm_status fm_group_summary(fm_group *g, uint32_t *alt_out, uint32_t *called_out, uint64_t *seg,
                           double *pi_sum, uint64_t *unc) {
    return guarded([&] {
        FM_NVTX("fm_group_summary (K2 plane pass)");
        if (!g) fail(FM_ERR_INVALID_ARG, "group is NULL");
        require_device();
        if (g->n_bits > 1 && alt_out)
            fail(FM_ERR_UNSUPPORTED,
                 "alt counts are undefined for a multi-allelic matrix (the reference builds no summary when "
                 "max_allele > 1, lib.rs:779)");
        ensure_counts(g);
        set_dev(g->m);
        Timer tm;
        tm.start();
        if (alt_out && g->m->V)
            CK(cudaMemcpyAsync(alt_out, g->d_alt, g->m->V * 4, cudaMemcpyDeviceToHost, stream()));
        if (called_out && g->m->V)
            CK(cudaMemcpyAsync(called_out, g->d_cnt, g->m->V * 4, cudaMemcpyDeviceToHost, stream()));
        tm.stop();
        CK(cudaStreamSynchronize(stream()));
        t_tim.d2h_ms += tm.ms();
        if (seg) *seg = g->seg;
        if (pi_sum) *pi_sum = g->pi_sum;
        if (unc) *unc = g->unc;
    });
}

// build_dense_population_summary for MANY groups -- normally one per region-sized matrix, the shape of the CLI's
// loop over config entries (process.rs:2169 -> stats.rs:1367-1470) -- in one persistent launch: groups whose counts
// are not cached yet become the units of one fm_k_plane_pass_seq launch, their partials
// are folded by one kernel and come back in one copy.  Each group ends up exactly as after fm_group_summary.
static void summarize_groups(fm_group *const *groups, size_t n_groups) {
    {
        if (n_groups && !groups) fail(FM_ERR_INVALID_ARG, "groups is NULL");
        require_device();
        if (!n_groups) return;
        for (size_t i = 0; i < n_groups; ++i) {
            if (!groups[i]) fail(FM_ERR_INVALID_ARG, "group is NULL");
            if (groups[i]->m->device != groups[0]->m->device) fail(FM_ERR_INVALID_ARG, "groups must live on one device");
        }
        const int device = groups[0]->m->device;
        CK(cudaSetDevice(device));
        std::vector<fm_group *> order(groups, groups + n_groups);
        std::sort(order.begin(), order.end());
        order.erase(std::unique(order.begin(), order.end()), order.end());
        std::vector<std::unique_lock<std::mutex>> locks;
        for (fm_group *g : order) locks.emplace_back(g->mu);  // address order: no lock inversion
        // the groups that share a launch: biallelic planes whose counts are not cached yet
        std::vector<fm_group *> gs;
        for (fm_group *g : order)
            if (!g->have_counts && g->n_bits == 1 && !g->count_only && g->m->V > 0) gs.push_back(g);
        if (!gs.empty()) {
            std::vector<fm::RowSeg> segs(gs.size());
            std::vector<size_t> part_off(gs.size());
            size_t total_b = 0;
            for (size_t i = 0; i < gs.size(); ++i) {
                const uint32_t V = (uint32_t)gs[i]->m->V;
                part_off[i] = total_b;
                total_b += (V + 31) / 32;
            }
            DevBuf<double> ppi(total_b);
            DevBuf<uint32_t> ppu(total_b * 2);
            std::vector<uint4> ents;
            for (size_t i = 0; i < gs.size(); ++i) {
                fm_group *g = gs[i];
                const uint32_t V = (uint32_t)g->m->V;
                alloc_counts(g);
                fm::DivEpilogue de{};
                set_tables(de, g);
                de.pi_form = FM_PIFORM_COUNTS;
                de.part_pi = ppi.p + part_off[i];
                de.part_u = ppu.p + 2 * part_off[i];
                de.alt_out = g->d_alt;
                de.called_out = called_cache(g);
                segs[i] = div_seg(g, de, 0, V);
                const uint32_t nb = (V + 31) / 32;
                for (uint32_t sb = 0; sb * fm::kSuperBatches < nb; ++sb)
                    ents.push_back(make_uint4((uint32_t)part_off[i], 0u, nb, sb));
            }
            if (total_b >= (1ull << 31)) fail(FM_ERR_UNSUPPORTED, "too many sites for one batched summary call");
            RowPlan plan;
            Timer tm;
            tm.start();
            if (!plan_rows(segs, nullptr, plan)) {
                // rows wider than the row pass handles (column-chunked): one pass per group
                locks.clear();
                for (fm_group *g : gs) ensure_counts(g);
                for (fm_group *g : order) locks.emplace_back(g->mu);
            } else {
                launch_rows(plan, device);
                DevBuf<uint4> d_ents(ents.size());
                d_ents.upload(ents.data(), ents.size());
                DevBuf<double> sd(ents.size());
                DevBuf<uint64_t> su(ents.size() * 2);
                fm::fm_k_reduce_partials_tab<<<(uint32_t)((ents.size() + 3) / 4), 128, 0, stream()>>>(
                    ppi.p, 1, ppu.p, 2, d_ents.p, (uint32_t)ents.size(), sd.p, su.p);
                CK(cudaGetLastError());
                g_launches++;
                tm.stop();
                std::vector<double> hd(ents.size());
                std::vector<uint64_t> hu(ents.size() * 2);
                sd.download(hd.data(), ents.size());
                su.download(hu.data(), ents.size() * 2);
                CK(cudaStreamSynchronize(stream()));
                t_tim.stats_ms += tm.ms();
                size_t e = 0;
                for (size_t i = 0; i < gs.size(); ++i) {
                    const uint32_t nb = ((uint32_t)gs[i]->m->V + 31) / 32;
                    double pi = 0.0;
                    uint64_t sg = 0, un = 0;
                    for (uint32_t sb = 0; sb * fm::kSuperBatches < nb; ++sb, ++e) {  // fixed order, like finish_partials
                        pi += hd[e];
                        sg += hu[2 * e];
                        un += hu[2 * e + 1];
                    }
                    gs[i]->pi_sum = pi;
                    gs[i]->seg = sg;
                    gs[i]->unc = un;
                    gs[i]->have_counts = true;
                }
            }
        }
        locks.clear();
        for (size_t i = 0; i < n_groups; ++i)
            if (!groups[i]->have_counts) ensure_counts(groups[i]);  // multi-allelic / empty matrices / leftovers
    }
}

fm_status fm_groups_summary_batch(fm_group *const *groups, size_t n_groups, uint64_t *seg_out, double *pi_sum_out,
                                  uint64_t *unc_out) {
    return guarded([&] {
        FM_NVTX("fm_groups_summary_batch (row plane pass)");
        summarize_groups(groups, n_groups);
        for (size_t i = 0; i < n_groups; ++i) {
            const fm_group *g = groups[i];
            if (seg_out) seg_out[i] = g->seg;
            if (pi_sum_out) pi_sum_out[i] = g->pi_sum;
            if (unc_out) unc_out[i] = g->unc;
        }
    });
}

// summaries of the two groups of a pair: one launch when neither is cached yet
static void ensure_counts_pair(fm_group *g1, fm_group *g2) {
    if (g1 != g2 && !g1->have_counts && !g2->have_counts && g1->m->device == g2->m->device) {
        fm_group *gs[2] = {g1, g2};
        summarize_groups(gs, 2);
        return;
    }
    ensure_counts(g1);
    ensure_counts(g2);
}

fm_status fm_group_segregating_sites(fm_group *g, uint64_t *out) {
    return guarded([&] {
        if (!g || !out) fail(FM_ERR_INVALID_ARG, "NULL argument");
        require_device();
        // stats.rs:3835-3842 / 4033-4035: membership.len() <= 1 -> 0
        if (g->n <= 1) {
            *out = 0;
            return;
        }
        ensure_counts(g);
        *out = g->seg;
    });
}

fm_status fm_group_pi(fm_group *g, int64_t L, int path, size_t raw_n, double *out) {
    return guarded([&] {
        if (!g || !out) fail(FM_ERR_INVALID_ARG, "NULL argument");
        require_device();
        const double NaN = std::numeric_limits<double>::quiet_NaN();
        const double Inf = std::numeric_limits<double>::infinity();
        if (path == FM_PI_SPARSE) {
            if (raw_n <= 1) { *out = NaN; return; }          // stats.rs:4322-4331
        } else if (g->n <= 1) { *out = NaN; return; }        // :1485 / :4539
        if (L < 0) { *out = 0.0; return; }
        if (L == 0) { *out = Inf; return; }
        if (path == FM_PI_SPARSE && g->n <= 1) { *out = NaN; return; }  // :4365
        if (g->n_bits > 1 && path == FM_PI_SUMMARY)
            fail(FM_ERR_UNSUPPORTED, "no dense summary exists for a multi-allelic matrix (lib.rs:779)");
        ensure_counts(g);
        set_dev(g->m);
        double pi_sum;
        uint64_t skipped;
        if (path == FM_PI_SUMMARY || (path == FM_PI_DENSE && g->m->has_missing)) {
            pi_sum = g->pi_sum;  // dense_pi_from_counts form
            skipped = g->unc;
        } else {
            const int form = path == FM_PI_DENSE ? FM_PIFORM_NOMISSING : FM_PIFORM_COMPONENTS;
            DivResult r = run_diversity(g, 0, (uint32_t)g->m->V, form, nullptr, nullptr, nullptr, 0,
                                        nullptr, 0, false);
            pi_sum = r.pi_sum;
            skipped = path == FM_PI_DENSE ? 0 : r.unc;  // stats.rs:4523: (sum_pi, 0usize)
        }
        const int64_t eff = sat_sub(L, (int64_t)skipped);
        if (eff == 0) { *out = NaN; return; }
        *out = pi_sum / (double)eff;
    });
}

fm_status fm_harmonic(size_t n, double *out) {
    if (!out) return FM_ERR_INVALID_ARG;
    double s = 0.0;
    for (size_t k = 1; k <= n; ++k) s += 1.0 / (double)k;
    *out = s;
    return FM_OK;
}

fm_status fm_watterson_theta(size_t seg, size_t n, int64_t L, double *out) {
    if (!out) return FM_ERR_INVALID_ARG;
    const double NaN = std::numeric_limits<double>::quiet_NaN();
    const double Inf = std::numeric_limits<double>::infinity();
    if (n <= 1 || L <= 0) {  // stats.rs:4246-4279
        *out = seg == 0 ? NaN : Inf;
        return FM_OK;
    }
    double h;
    fm_harmonic(n - 1, &h);
    *out = h > 0.0 ? (double)seg / h / (double)L : (seg == 0 ? NaN : Inf);
    return FM_OK;
}

fm_status fm_per_site_diversity_multi(fm_group *const *groups, const size_t *raw_n, size_t n_groups, int64_t rs,
                                      int64_t re, const int64_t *mask_iv, size_t n_mask, const int64_t *filtered,
                                      size_t n_filt, int64_t *pos_out, double *pi_out, double *theta_out,
                                      size_t capacity, size_t *n_out);

fm_status fm_per_site_diversity(fm_group *g, size_t raw_n, int64_t rs, int64_t re, const int64_t *mask_iv,
                                size_t n_mask, const int64_t *filtered, size_t n_filt, int64_t *pos_out,
                                double *pi_out, double *theta_out, size_t capacity, size_t *n_out) {
    fm_status st = guarded([&] {
        if (!g || !n_out) fail(FM_ERR_INVALID_ARG, "NULL argument");
        *n_out = 0;
        require_device();
    });
    if (st != FM_OK) return st;
    if (raw_n < 2) return FM_OK;  // stats.rs:4675-4681: no sites at all (the multi-group call reports NaN rows)
    return fm_per_site_diversity_multi(&g, &raw_n, 1, rs, re, mask_iv, n_mask, filtered, n_filt, pos_out, pi_out, theta_out,
                                       capacity, n_out);
}

fm_status fm_per_site_diversity_multi(fm_group *const *groups, const size_t *raw_n, size_t n_groups, int64_t rs,
                                      int64_t re, const int64_t *mask_iv, size_t n_mask, const int64_t *filtered,
                                      size_t n_filt, int64_t *pos_out, double *pi_out, double *theta_out,
                                      size_t capacity, size_t *n_out) {
    return guarded([&] {
        FM_NVTX("fm_per_site_diversity_multi (fused plane pass + tracks)");
        if (!groups || !n_groups || !n_out || !raw_n) fail(FM_ERR_INVALID_ARG, "NULL argument");
        *n_out = 0;
        require_device();
        fm_matrix *m = groups[0]->m;
        for (size_t i = 0; i < n_groups; ++i)
            if (!groups[i] || groups[i]->m != m) fail(FM_ERR_INVALID_ARG, "groups must share one matrix");
        if (region_len(rs, re) <= 0) return;  // stats.rs:4656-4666
        set_dev(m);
        uint32_t lo, hi;
        site_range(m, rs, re, lo, hi);
        const size_t n = hi - lo;
        if (n == 0) return;
        if (n > capacity) fail(FM_ERR_INVALID_ARG, "output capacity too small");
        if (!pi_out || !theta_out) fail(FM_ERR_INVALID_ARG, "output arrays are NULL");
        std::vector<int64_t> merged, fs;
        DevBuf<int64_t> d_mask, d_filt;
        if (mask_iv) {
            merge_intervals(mask_iv, n_mask, merged);
            d_mask.alloc(std::max<size_t>(merged.size(), 2));
            d_mask.upload(merged.data(), merged.size());
        }
        if (filtered && n_filt) {
            fs.assign(filtered, filtered + n_filt);
            std::sort(fs.begin(), fs.end());
            d_filt.alloc(fs.size());
            d_filt.upload(fs.data(), fs.size());
        }
        // groups with fewer than two listed haplotypes yield no sites in the reference
        // (stats.rs:4675-4681): their rows are NaN here
        std::vector<fm_group *> act;
        std::vector<size_t> act_idx;
        for (size_t i = 0; i < n_groups; ++i)
            if (raw_n[i] >= 2) {
                act.push_back(groups[i]);
                act_idx.push_back(i);
            }
        // Page-locked output arrays take the tracks straight from the kernel's epilogue (coalesced 256-byte stores
        // over PCIe, no HBM round trip and no copy after the pass); pageable ones get device buffers + D2H copies.
        std::vector<DevBuf<double>> d_pi(act.size()), d_th(act.size());
        std::vector<double *> ppi(act.size()), pth(act.size());
        std::vector<char> direct(act.size(), 0);
        for (size_t i = 0; i < act.size(); ++i) {
            double *mp = static_cast<double *>(mapped_host_range(pi_out + act_idx[i] * capacity, n * 8));
            double *mt = static_cast<double *>(mapped_host_range(theta_out + act_idx[i] * capacity, n * 8));
            if (mp && mt) {
                direct[i] = 1;
                ppi[i] = mp;
                pth[i] = mt;
            } else {
                d_pi[i].alloc(n);
                d_th[i].alloc(n);
                ppi[i] = d_pi[i].p;
                pth[i] = d_th[i].p;
            }
        }
        // positions + 1 (stats.rs:4746): a small kernel on a side stream underneath the pass
        DevBuf<int64_t> d_p1;
        int64_t *pos_direct = (pos_out && n >= 65536) ? static_cast<int64_t *>(mapped_host_range(pos_out, n * 8)) : nullptr;
        cudaStream_t side = nullptr;
        struct SideJoin {  // an early exit must not leave the side kernel writing into the caller's buffer
            cudaStream_t *s;
            ~SideJoin() {
                if (*s) cudaStreamSynchronize(*s);
            }
        } side_join{&side};
        EventPairs evs;
        if (pos_direct) {
            side = t_side_streams.get(m->device);
            cudaEvent_t e0 = evs.next();
            CK(cudaEventRecord(e0, stream()));
            CK(cudaStreamWaitEvent(side, e0, 0));
            fm_k_pos_plus1<<<(uint32_t)std::min<size_t>((n + 255) / 256, 2048), 256, 0, side>>>(m->d_pos, lo, (uint32_t)n, pos_direct);
            CK(cudaGetLastError());
            g_launches++;
        }
        Timer pass_tm;
        bool fused = false;
        {
            std::vector<std::unique_lock<std::mutex>> locks;
            std::vector<fm_group *> order(act);
            std::sort(order.begin(), order.end());
            order.erase(std::unique(order.begin(), order.end()), order.end());
            for (fm_group *g : order) locks.emplace_back(g->mu);  // address order: no lock inversion
            if (!act.empty())
                fused = run_diversity_multi(act.data(), act.size(), lo, hi, FM_PIFORM_COMPONENTS, ppi.data(), pth.data(),
                                            mask_iv ? d_mask.p : nullptr, (uint32_t)(merged.size() / 2),
                                            fs.empty() ? nullptr : d_filt.p, (uint32_t)fs.size(), /*out=*/nullptr, false,
                                            &pass_tm);
        }
        Timer tm;
        tm.start();
        for (size_t i = 0; i < act.size(); ++i)
            if (!direct[i]) {
                d_pi[i].download(pi_out + act_idx[i] * capacity, n);
                d_th[i].download(theta_out + act_idx[i] * capacity, n);
            }
        if (pos_direct) {
            cudaEvent_t e1 = evs.next();
            CK(cudaEventRecord(e1, side));
            CK(cudaStreamWaitEvent(stream(), e1, 0));
        } else {
            download_positions_plus1(m, lo, n, pos_out, d_p1);
        }
        tm.stop();
        CK(cudaStreamSynchronize(stream()));
        t_tim.d2h_ms += tm.ms();
        if (fused) t_tim.stats_ms += pass_tm.ms();
        const double NaN = std::numeric_limits<double>::quiet_NaN();
        for (size_t i = 0; i < n_groups; ++i)
            if (raw_n[i] < 2)
                for (size_t k = 0; k < n; ++k) pi_out[i * capacity + k] = theta_out[i * capacity + k] = NaN;
        *n_out = n;
    });
}

// ------------------------------------------------------------------------------------ streaming ingest
// SURVEY §8(f1): the u8 matrix is handed over in row chunks, staged in two device buffers and
// repacked straight into the bitplanes of every declared group while the next chunk is still
// on the PCIe bus.  The u8 rows are never resident (1.125 B/genotype of HBM and the separate
// repack pass are saved).
// Per-site pi / theta tracks requested for the matrix being ingested (fm_ingest_request_tracks): every chunk's
// tracks are computed right after its repack and stored while the next chunks are still on the bus.
struct IngestTracks {
    std::vector<fm_group *> act;        // groups with >= 2 listed haplotypes
    std::vector<size_t> act_idx;        // their row in the caller's arrays
    std::vector<size_t> nan_rows;       // rows of groups with < 2 listed haplotypes: NaN (stats.rs:4675-4681)
    uint32_t lo = 0, hi = 0;            // site range of the region
    size_t capacity = 0;
    DevBuf<int64_t> d_mask, d_filt;
    uint32_t n_mask = 0, n_filt = 0;
    bool has_mask = false;
    std::vector<double *> ppi, pth;     // device-visible destinations (the caller's page-locked rows or own buffers)
    std::vector<DevBuf<double>> own_pi, own_th;
    std::vector<char> direct;
    int64_t *pos_out = nullptr, *pos_direct = nullptr;
    double *pi_out = nullptr, *theta_out = nullptr;
    bool pos_done = false;
};

struct fm_ingest {
    fm_matrix *m = nullptr;
    std::unique_ptr<IngestTracks> tracks;
    cudaEvent_t pos_up = nullptr;         // the positions are on the device (recorded on copy_s)
    std::vector<fm_group *> groups;       // declared with fm_ingest_add_group (owned until finish)
    std::vector<fm_partition *> parts;    // declared with fm_ingest_add_partition
    std::vector<fm_group *> all;          // every group that receives rows
    size_t chunk_rows = 0, rows_done = 0;
    uint8_t *stage[2] = {nullptr, nullptr};
    uint64_t *stage_m[2] = {nullptr, nullptr};
    size_t stage_words = 0;
    cudaStream_t copy_s = nullptr, comp_s = nullptr;
    cudaEvent_t copied[2] = {nullptr, nullptr}, consumed[2] = {nullptr, nullptr};
    cudaEvent_t t_copy0 = nullptr, t_copy1 = nullptr, t_comp0 = nullptr, t_comp1 = nullptr;
    bool used[2] = {false, false};
    bool timing_started = false;
    RepackSet set;                        // descriptor table of `all`, built at the first fm_ingest_rows
    int next = 0;
    uint8_t *pin[2] = {nullptr, nullptr};  // fm_ingest_rows_pack: pinned staging of packed chunks
    cudaEvent_t pin_free[2] = {nullptr, nullptr};
    bool pin_used[2] = {false, false};
    float pack_ms = 0.f;                   // host time spent in the packer (fm_ingest_rows_pack)
    bool pos_uploaded = false;
};

// Host work that does not depend on the rows -- the upload of the (pageable) position vector -- is done once,
// after a rows call has queued its asynchronous copies, so it hides under the DMA instead of preceding it.
// Page-locked positions (large matrices) are a true asynchronous copy: they go first on the copy stream of the first
// rows call, 0.15 ms per 1M sites ahead of the row chunks.
static void ingest_early_setup(fm_ingest *h) {
    if (h->pos_uploaded || !h->m->pos.pinned) return;
    fm_matrix *m = h->m;
    if (m->V) CK(cudaMemcpyAsync(m->d_pos, m->pos.data(), m->V * 8, cudaMemcpyHostToDevice, h->copy_s));
    h->pos_uploaded = true;
    if (h->tracks) {  // the track kernels read the positions (mask lookup, positions + 1)
        if (!h->pos_up) CK(cudaEventCreateWithFlags(&h->pos_up, cudaEventDisableTiming));
        CK(cudaEventRecord(h->pos_up, h->copy_s));
        CK(cudaStreamWaitEvent(h->comp_s, h->pos_up, 0));
    }
}

// Tracks of the freshly repacked rows [r0, r1) on the ingest's compute stream (after launch_repack).
static void ingest_tracks_chunk(fm_ingest *h, size_t r0, size_t r1) {
    IngestTracks *T = h->tracks.get();
    if (!T || T->act.empty()) return;
    const uint32_t lo = (uint32_t)std::max<size_t>(r0, T->lo), hi = (uint32_t)std::min<size_t>(r1, T->hi);
    if (lo >= hi) return;
    fm_matrix *m = h->m;
    if (!h->pos_uploaded) {  // pageable positions (small matrices): put them on the device now, ordered before the pass
        if (m->V) CK(cudaMemcpyAsync(m->d_pos, m->pos.data(), m->V * 8, cudaMemcpyHostToDevice, h->comp_s));
        h->pos_uploaded = true;
    }
    StreamScope on_comp(h->comp_s);
    if (!T->pos_done && T->pos_direct) {
        const size_t n = T->hi - T->lo;
        fm_k_pos_plus1<<<(uint32_t)std::min<size_t>((n + 255) / 256, 2048), 256, 0, h->comp_s>>>(m->d_pos, T->lo, (uint32_t)n,
                                                                                                    T->pos_direct);
        CK(cudaGetLastError());
        g_launches++;
        T->pos_done = true;
    }
    std::vector<double *> ppi(T->act.size()), pth(T->act.size());
    for (size_t i = 0; i < T->act.size(); ++i) {
        ppi[i] = T->ppi[i] + (lo - T->lo);
        pth[i] = T->pth[i] + (lo - T->lo);
    }
    run_diversity_multi(T->act.data(), T->act.size(), lo, hi, FM_PIFORM_COMPONENTS, ppi.data(), pth.data(),
                        T->has_mask ? T->d_mask.p : nullptr, T->n_mask, T->n_filt ? T->d_filt.p : nullptr, T->n_filt,
                        /*out=*/nullptr);
}

static size_t tapered_chunk(size_t rows_left, size_t chunk);

static void ingest_late_setup(fm_ingest *h) {
    if (h->pos_uploaded) return;
    fm_matrix *m = h->m;
    if (m->V) CK(cudaMemcpyAsync(m->d_pos, m->pos.data(), m->V * 8, cudaMemcpyHostToDevice, stream()));
    CK(cudaStreamSynchronize(stream()));
    h->pos_uploaded = true;
}

static void ingest_destroy(fm_ingest *h, bool release_handles) {
    if (!h) return;
    if (h->m) cudaSetDevice(h->m->device);
    if (h->copy_s) cudaStreamSynchronize(h->copy_s);
    if (h->comp_s) cudaStreamSynchronize(h->comp_s);
    h->set.release();
    for (int i = 0; i < 2; ++i) {
        dev_free(h->stage[i]);
        dev_free(h->stage_m[i]);
        if (h->copied[i]) cudaEventDestroy(h->copied[i]);
        if (h->consumed[i]) cudaEventDestroy(h->consumed[i]);
    }
    for (cudaEvent_t e : {h->t_copy0, h->t_copy1, h->t_comp0, h->t_comp1, h->pin_free[0], h->pin_free[1], h->pos_up})
        if (e) cudaEventDestroy(e);
    for (int i = 0; i < 2; ++i) g_pinned.give(h->pin[i]);  // the copy stream was synchronised above
    const int pool_dev = h->m ? h->m->device : t_device;  // both streams were synchronised above
    g_stream_pool.give(pool_dev, h->copy_s);
    g_stream_pool.give(pool_dev, h->comp_s);
    if (release_handles) {
        for (fm_group *g : h->groups) fm_group_release(g);
        for (fm_partition *p : h->parts) fm_partition_release(p);
        fm_matrix_release(h->m);
    }
    delete h;
}

fm_status fm_ingest_begin(size_t V, size_t S, size_t ploidy, int has_missing, uint8_t max_allele,
                          const int64_t *positions, size_t chunk_rows, fm_ingest **out) {
    return guarded([&] {
        if (!out) fail(FM_ERR_INVALID_ARG, "out is NULL");
        *out = nullptr;
        require_device();
        CK(cudaSetDevice(t_device));
        fm_ingest *h = new fm_ingest();
        static const uint32_t trace = env_u32("FM_INGEST_TRACE", 0);
        const auto tb0 = std::chrono::steady_clock::now();
        auto since = [&] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tb0).count(); };
        double tb_pos = 0, tb_ev = 0, tb_st = 0;
        try {
            h->m = matrix_common(V, S, ploidy, max_allele, positions);
            tb_pos = since();
            h->m->has_missing = has_missing != 0;
            h->m->in_band = has_missing == FM_MISSING_IN_BAND;
            if (h->m->in_band && max_allele > 127)
                fail(FM_ERR_INVALID_ARG, "in-band missingness needs allele indices <= 127");
            h->m->streamed = true;
            h->m->d_pos = static_cast<int64_t *>(dev_alloc(std::max<size_t>(V, 1) * 8));
            // the positions are uploaded by the first rows call, while its DMA is in flight (ingest_late_setup)
            const size_t stride = std::max<size_t>(h->m->stride, 1);
            if (chunk_rows == 0) chunk_rows = std::max<size_t>(32, ((size_t)64 << 20) / stride);
            chunk_rows = std::min(std::max<size_t>(chunk_rows, 1), std::max<size_t>(V, 1));
            h->chunk_rows = chunk_rows;
            h->stage_words = (chunk_rows * stride + 63) / 64 + 2;
            for (int i = 0; i < 2; ++i) {  // the u8 staging buffers are allocated by the first fm_ingest_rows
                CK(cudaEventCreateWithFlags(&h->copied[i], cudaEventDisableTiming));
                CK(cudaEventCreateWithFlags(&h->consumed[i], cudaEventDisableTiming));
            }
            CK(cudaEventCreate(&h->t_copy0));
            CK(cudaEventCreate(&h->t_copy1));
            CK(cudaEventCreate(&h->t_comp0));
            CK(cudaEventCreate(&h->t_comp1));
            tb_ev = since();
            h->copy_s = g_stream_pool.take(h->m->device);
            h->comp_s = g_stream_pool.take(h->m->device);
            tb_st = since();
            CK(cudaStreamSynchronize(stream()));  // staging buffers are now usable from any stream
            if (trace)
                fprintf(stderr, "[ingest begin] positions %.3f ms, alloc + events %.3f ms, streams %.3f ms, sync %.3f ms\n", tb_pos,
                        tb_ev - tb_pos, tb_st - tb_ev, since() - tb_st);
        } catch (...) {
            ingest_destroy(h, true);
            throw;
        }
        *out = h;
    });
}

fm_status fm_ingest_add_group(fm_ingest *h, const uint64_t *sample_idx, const uint8_t *side, size_t n,
                              size_t *group_index) {
    return guarded([&] {
        if (!h) fail(FM_ERR_INVALID_ARG, "ingest handle is NULL");
        if (n && (!sample_idx || !side)) fail(FM_ERR_INVALID_ARG, "haplotype arrays are NULL");
        if (h->rows_done) fail(FM_ERR_INVALID_ARG, "groups must be declared before the first fm_ingest_rows");
        fm_group *g = alloc_group(h->m, membership_offsets(h->m, sample_idx, side, n));
        h->groups.push_back(g);
        h->all.push_back(g);
        if (group_index) *group_index = h->groups.size() - 1;
    });
}

fm_status fm_ingest_add_partition(fm_ingest *h, const uint16_t *left, const uint16_t *right, size_t n_samples,
                                  size_t n_groups, size_t *partition_index) {
    return guarded([&] {
        if (!h) fail(FM_ERR_INVALID_ARG, "ingest handle is NULL");
        if (n_samples && (!left || !right)) fail(FM_ERR_INVALID_ARG, "membership arrays are NULL");
        if (n_groups >= 0xFFFF) fail(FM_ERR_INVALID_ARG, "too many groups");
        if (h->rows_done) fail(FM_ERR_INVALID_ARG, "partitions must be declared before the first fm_ingest_rows");
        fm_partition *p = new fm_partition();
        p->m = h->m;
        p->G = n_groups;
        fm_matrix_retain(h->m);
        try {
            std::vector<std::vector<uint32_t>> cols = partition_columns(h->m, left, right, n_samples, n_groups);
            set_dev(h->m);
            const size_t per = 2 * std::max<size_t>(h->m->V, 1);
            p->d_counts_slab = static_cast<uint32_t *>(dev_alloc((n_groups + 1) * per * sizeof(uint32_t)));
            for (size_t g = 0; g <= n_groups; ++g)
                p->groups.push_back(alloc_group(h->m, std::move(cols[g]), true, p->d_counts_slab + g * per));
        } catch (...) {
            fm_partition_release(p);
            throw;
        }
        h->parts.push_back(p);
        for (fm_group *g : p->groups) h->all.push_back(g);
        if (partition_index) *partition_index = h->parts.size() - 1;
    });
}

fm_status fm_ingest_request_tracks(fm_ingest *h, const size_t *group_index, const size_t *raw_n, size_t n_groups,
                                   int64_t rs, int64_t re, const int64_t *mask_iv, size_t n_mask, const int64_t *filtered,
                                   size_t n_filt, int64_t *pos_out, double *pi_out, double *theta_out, size_t capacity,
                                   size_t *n_out) {
    return guarded([&] {
        if (!h || !group_index || !raw_n || !n_groups || !n_out) fail(FM_ERR_INVALID_ARG, "NULL argument");
        *n_out = 0;
        if (h->rows_done) fail(FM_ERR_INVALID_ARG, "tracks must be requested before the first rows call");
        if (h->tracks) fail(FM_ERR_INVALID_ARG, "tracks were already requested for this ingest");
        fm_matrix *m = h->m;
        set_dev(m);
        auto T = std::make_unique<IngestTracks>();
        for (size_t i = 0; i < n_groups; ++i) {
            if (group_index[i] >= h->groups.size()) fail(FM_ERR_INVALID_ARG, "group index out of range");
            fm_group *g = h->groups[group_index[i]];
            if (g->n_bits != 1 || g->count_only)
                fail(FM_ERR_UNSUPPORTED, "streamed tracks need biallelic bitplane groups (use fm_per_site_diversity after finish)");
            if (raw_n[i] >= 2) {
                T->act.push_back(g);
                T->act_idx.push_back(i);
            } else {
                T->nan_rows.push_back(i);
            }
        }
        if (region_len(rs, re) <= 0) {  // stats.rs:4656-4666: no sites; nothing to compute while the rows arrive
            h->tracks = std::move(T);
            h->tracks->act.clear();
            h->tracks->nan_rows.clear();
            return;
        }
        uint32_t lo, hi;
        site_range(m, rs, re, lo, hi);
        const size_t n = hi - lo;
        T->lo = lo;
        T->hi = hi;
        T->capacity = capacity;
        T->pos_out = pos_out;
        T->pi_out = pi_out;
        T->theta_out = theta_out;
        if (n) {
            if (n > capacity) fail(FM_ERR_INVALID_ARG, "output capacity too small");
            if (!pi_out || !theta_out) fail(FM_ERR_INVALID_ARG, "output arrays are NULL");
            std::vector<int64_t> merged, fs;
            if (mask_iv) {
                merge_intervals(mask_iv, n_mask, merged);
                T->d_mask.alloc(std::max<size_t>(merged.size(), 2));
                T->d_mask.upload(merged.data(), merged.size());
                T->n_mask = (uint32_t)(merged.size() / 2);
                T->has_mask = true;
            }
            if (filtered && n_filt) {
                fs.assign(filtered, filtered + n_filt);
                std::sort(fs.begin(), fs.end());
                T->d_filt.alloc(fs.size());
                T->d_filt.upload(fs.data(), fs.size());
                T->n_filt = (uint32_t)fs.size();
            }
            const size_t na = T->act.size();
            T->ppi.resize(na);
            T->pth.resize(na);
            T->own_pi = std::vector<DevBuf<double>>(na);
            T->own_th = std::vector<DevBuf<double>>(na);
            T->direct.assign(na, 0);
            for (size_t i = 0; i < na; ++i) {
                double *mp = static_cast<double *>(mapped_host_range(pi_out + T->act_idx[i] * capacity, n * 8));
                double *mt = static_cast<double *>(mapped_host_range(theta_out + T->act_idx[i] * capacity, n * 8));
                if (mp && mt) {
                    T->direct[i] = 1;
                    T->ppi[i] = mp;
                    T->pth[i] = mt;
                } else {
                    T->own_pi[i].alloc(n);
                    T->own_th[i].alloc(n);
                    T->ppi[i] = T->own_pi[i].p;
                    T->pth[i] = T->own_th[i].p;
                }
            }
            if (pos_out) T->pos_direct = static_cast<int64_t *>(mapped_host_range(pos_out, n * 8));
            CK(cudaStreamSynchronize(stream()));  // the interval lists are host temporaries; buffers usable on comp_s
        } else {
            T->act.clear();
            T->nan_rows.clear();
        }
        *n_out = n;
        h->tracks = std::move(T);
    });
}

fm_status fm_ingest_rows(fm_ingest *h, const uint8_t *rows, const uint64_t *missing_whole, size_t first_row,
                         size_t n_rows) {
    return guarded([&] {
        FM_NVTX("fm_ingest_rows (H2D u8 + K1 repack)");
        if (!h) fail(FM_ERR_INVALID_ARG, "ingest handle is NULL");
        fm_matrix *m = h->m;
        if (first_row > m->V || n_rows > m->V - first_row) fail(FM_ERR_INVALID_ARG, "row range outside the matrix");
        if (n_rows && m->stride && !rows) fail(FM_ERR_INVALID_ARG, "rows is NULL");
        const bool bitmap = m->has_missing && !m->in_band;
        if (bitmap && !missing_whole) fail(FM_ERR_INVALID_ARG, "matrix was declared with a missing bitmap");
        if (m->packed) fail(FM_ERR_INVALID_ARG, "this ingest already received packed rows (fm_ingest_rows_packed)");
        set_dev(m);
        const size_t stride = m->stride;
        if (!h->stage[0]) {
            for (int i = 0; i < 2; ++i) {
                h->stage[i] = static_cast<uint8_t *>(dev_alloc(std::max<size_t>(h->chunk_rows * std::max<size_t>(stride, 1), 16)));
                if (bitmap) h->stage_m[i] = static_cast<uint64_t *>(dev_alloc(h->stage_words * 8));
            }
            CK(cudaStreamSynchronize(stream()));  // staging buffers are now usable from any stream
        }
        if (!h->set.d_desc && !h->all.empty()) h->set.build(h->all);  // groups are final from here on
        if (!h->timing_started && n_rows) {
            CK(cudaEventRecord(h->t_copy0, h->copy_s));
            ingest_early_setup(h);
            CK(cudaEventRecord(h->t_comp0, h->comp_s));
            h->timing_started = true;
        }
        for (size_t r0 = first_row; r0 < first_row + n_rows; r0 += h->chunk_rows) {
            const size_t r1 = std::min(first_row + n_rows, r0 + h->chunk_rows);
            const int b = h->next;
            h->next ^= 1;
            if (h->used[b]) CK(cudaStreamWaitEvent(h->copy_s, h->consumed[b], 0));
            if (stride)
                h2d(h->stage[b], rows + (r0 - first_row) * stride, (r1 - r0) * stride, h->copy_s);
            uint64_t w0 = 0;
            if (bitmap && stride) {
                w0 = (uint64_t)(r0 * stride) >> 6;
                const uint64_t w1 = ((uint64_t)(r1 * stride) + 63) >> 6;
                h2d(h->stage_m[b], missing_whole + w0, (w1 - w0) * 8, h->copy_s);
            }
            CK(cudaEventRecord(h->copied[b], h->copy_s));
            CK(cudaStreamWaitEvent(h->comp_s, h->copied[b], 0));
            launch_repack(h->set, h->stage[b], (r1 - r0) * stride, bitmap ? h->stage_m[b] : nullptr,
                          (uint32_t)r0, w0, (uint32_t)r0, (uint32_t)r1, h->comp_s);
            ingest_tracks_chunk(h, r0, r1);
            CK(cudaEventRecord(h->consumed[b], h->comp_s));
            h->used[b] = true;
        }
        h->rows_done += n_rows;
        CK(cudaEventRecord(h->t_copy1, h->copy_s));
        CK(cudaEventRecord(h->t_comp1, h->comp_s));
        ingest_late_setup(h);
        CK(cudaStreamSynchronize(h->copy_s));  // the caller's buffers are free again on return
    });
}

// Packed rows (2 bits per genotype, SURVEY 8 f1): the host hands over the full-row bit words a parser or the
// library's own packer (fm_pack_rows) produced.  They are copied straight into the resident packed matrix --
// no staging, no u8 on PCIe -- and every declared group is compressed out of them chunk by chunk (K1p) while
// the next chunk is on the bus.
static void ensure_packed_storage(fm_matrix *m, bool with_called) {
    if (m->max_allele > 1)
        fail(FM_ERR_UNSUPPORTED, "packed rows carry one allele bit per cell: max_allele must be <= 1 (use the u8 ingest)");
    if (m->d_abits) return;
    m->rw = (uint32_t)((m->stride + 31) / 32);
    const size_t words = std::max<size_t>(m->V * (size_t)m->rw, 4);
    m->d_abits = static_cast<uint32_t *>(dev_alloc(words * 4));
    if (with_called) m->d_cbits = static_cast<uint32_t *>(dev_alloc(words * 4));
    m->packed = true;
}

fm_status fm_packed_row_words(size_t n_samples, size_t ploidy, size_t *row_words) {
    if (!row_words) return FM_ERR_INVALID_ARG;
    *row_words = (n_samples * ploidy + 31) / 32;
    return FM_OK;
}

fm_status fm_pack_rows(const uint8_t *rows, const uint64_t *missing_whole, int missing_mode, size_t first_row,
                       size_t n_rows, size_t n_total_rows, size_t stride, uint32_t *allele_bits, uint32_t *called_bits,
                       int n_threads) {
    return guarded([&] {  // host only: works without a CUDA device
        const char *err = fm_host_pack_rows(rows, missing_whole, missing_mode, first_row, n_rows, n_total_rows, stride,
                                            allele_bits, called_bits, n_threads);
        if (err) fail(FM_ERR_INVALID_ARG, err);
    });
}

fm_status fm_pack_rows_generic(const uint8_t *rows, const uint64_t *missing_whole, int missing_mode, size_t first_row,
                               size_t n_rows, size_t n_total_rows, size_t stride, uint32_t *allele_bits,
                               uint32_t *called_bits) {
    return guarded([&] {
        const char *err = fm_host_pack_rows_generic(rows, missing_whole, missing_mode, first_row, n_rows, n_total_rows,
                                                    stride, allele_bits, called_bits);
        if (err) fail(FM_ERR_INVALID_ARG, err);
    });
}

fm_status fm_ingest_rows_packed(fm_ingest *h, const uint32_t *allele_bits, const uint32_t *called_bits,
                                size_t first_row, size_t n_rows) {
    return guarded([&] {
        FM_NVTX("fm_ingest_rows_packed (H2D packed + K1p compress)");
        if (!h) fail(FM_ERR_INVALID_ARG, "ingest handle is NULL");
        fm_matrix *m = h->m;
        if (first_row > m->V || n_rows > m->V - first_row) fail(FM_ERR_INVALID_ARG, "row range outside the matrix");
        if (h->stage[0]) fail(FM_ERR_INVALID_ARG, "this ingest already received u8 rows (fm_ingest_rows)");
        if (m->in_band) fail(FM_ERR_INVALID_ARG, "packed rows carry their own called bits: begin with FM_MISSING_BITMAP or _NONE");
        if (n_rows && m->stride && !allele_bits) fail(FM_ERR_INVALID_ARG, "allele_bits is NULL");
        if (m->has_missing && n_rows && m->stride && !called_bits)
            fail(FM_ERR_INVALID_ARG, "matrix was declared with missing data: called_bits is required");
        if (!m->has_missing && called_bits)
            fail(FM_ERR_INVALID_ARG, "matrix was declared without missing data: called_bits must be NULL");
        set_dev(m);
        const bool first_call = !m->d_abits;
        ensure_packed_storage(m, m->has_missing);
        if (first_call) CK(cudaStreamSynchronize(stream()));  // storage (and a cached block's previous owner) is settled
        if (!h->set.d_desc && !h->all.empty()) h->set.build(h->all);  // groups are final from here on
        if (!h->timing_started && n_rows) {
            CK(cudaEventRecord(h->t_copy0, h->copy_s));
            ingest_early_setup(h);
            CK(cudaEventRecord(h->t_comp0, h->comp_s));
            h->timing_started = true;
        }
        const size_t rw = m->rw;
        // chunk = ~32 MB of bit words: small enough that the last chunk's compress pass is short
        const size_t per_row = std::max<size_t>(rw * 4 * (m->has_missing ? 2 : 1), 1);
        const size_t chunk = std::max<size_t>(32, ((size_t)32 << 20) / per_row);
        for (size_t r0 = first_row, step = 0; r0 < first_row + n_rows; r0 += step) {
            step = tapered_chunk(first_row + n_rows - r0, chunk);
            const size_t r1 = r0 + step;
            if (rw) {
                h2d(m->d_abits + r0 * rw, allele_bits + (r0 - first_row) * rw, (r1 - r0) * rw * 4, h->copy_s);
                if (m->has_missing)
                    h2d(m->d_cbits + r0 * rw, called_bits + (r0 - first_row) * rw, (r1 - r0) * rw * 4, h->copy_s);
            }
            const int b = h->next;
            h->next ^= 1;
            CK(cudaEventRecord(h->copied[b], h->copy_s));
            CK(cudaStreamWaitEvent(h->comp_s, h->copied[b], 0));
            launch_repack(h->set, nullptr, 0, nullptr, 0, 0, (uint32_t)r0, (uint32_t)r1, h->comp_s);
            ingest_tracks_chunk(h, r0, r1);
        }
        h->rows_done += n_rows;
        CK(cudaEventRecord(h->t_copy1, h->copy_s));
        CK(cudaEventRecord(h->t_comp1, h->comp_s));
        ingest_late_setup(h);
        CK(cudaStreamSynchronize(h->copy_s));  // the caller's buffers are free again on return
    });
}

// ---- packed rows with a sparse missing list
// Shared by the streaming and the one-shot entry points: rows [first_row, first_row + n_rows) arrive as allele bit
// words + a CSR list of missing cells (row_start relative to this call).  Chunks of rows are copied on copy_s; on
// comp_s every chunk's called words are rebuilt on the device (fm_k_expand_called) and -- when groups are declared --
// compressed into their planes (K1p), while the next chunk is on the bus.
static void expand_called_launch(fm_matrix *m, const uint64_t *d_start, const void *d_cols, int col_bytes, uint64_t cols_base,
                                 uint32_t r_base, uint32_t v_lo, uint32_t v_hi, cudaStream_t st) {
    if (v_hi <= v_lo || !m->rw) return;
    const size_t warp_bytes = (size_t)m->rw * 4;
    if (warp_bytes > 200 * 1024) fail(FM_ERR_UNSUPPORTED, "packed rows wider than the expand kernel's shared memory");
    const uint32_t warps = (uint32_t)std::max<size_t>(1, std::min<size_t>(8, (200 * 1024) / warp_bytes));
    const size_t smem = warps * warp_bytes;
    const uint32_t rows = v_hi - v_lo;
    const uint32_t per_sm = (uint32_t)std::max<size_t>(1, std::min<size_t>(8, (220 * 1024) / std::max<size_t>(smem, 1)));
    const uint32_t blocks = std::max(1u, std::min<uint32_t>((rows + warps - 1) / warps, per_sm * (uint32_t)sm_count(m->device)));
    static std::once_flag once2, once4;
    if (col_bytes == 1) {
        static std::once_flag once1;
        std::call_once(once1, [] {
            cudaFuncSetAttribute(fm::fm_k_expand_called<uint8_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        });
        fm::fm_k_expand_called<uint8_t><<<blocks, warps * 32, smem, st>>>(d_start, static_cast<const uint8_t *>(d_cols),
                                                                           cols_base, r_base, v_lo, v_hi, m->rw,
                                                                           (uint32_t)m->stride, m->d_cbits);
    } else if (col_bytes == 2) {
        std::call_once(once2, [] {
            cudaFuncSetAttribute(fm::fm_k_expand_called<uint16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        });
        fm::fm_k_expand_called<uint16_t><<<blocks, warps * 32, smem, st>>>(d_start, static_cast<const uint16_t *>(d_cols),
                                                                            cols_base, r_base, v_lo, v_hi, m->rw,
                                                                            (uint32_t)m->stride, m->d_cbits);
    } else {
        std::call_once(once4, [] {
            cudaFuncSetAttribute(fm::fm_k_expand_called<uint32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        });
        fm::fm_k_expand_called<uint32_t><<<blocks, warps * 32, smem, st>>>(d_start, static_cast<const uint32_t *>(d_cols),
                                                                            cols_base, r_base, v_lo, v_hi, m->rw,
                                                                            (uint32_t)m->stride, m->d_cbits);
    }
    CK(cudaGetLastError());
    g_launches++;
}

// Chunk sizes of a chunked upload: full chunks, then halves of what is left down to a quarter chunk -- the kernels of the LAST chunk are the only work
// that is not hidden under the DMA of a following one, so the last chunk is a quarter of the others.
static size_t tapered_chunk(size_t rows_left, size_t chunk) {
    if (chunk < 128 || rows_left > 2 * chunk) return std::min(rows_left, chunk);
    if (rows_left <= chunk / 4) return rows_left;
    return std::min(rows_left, std::min(chunk, std::max(chunk / 4, (rows_left + 1) / 2)));
}

static void packed_sparse_rows(fm_matrix *m, const RepackSet *set, const uint32_t *allele_bits, const uint64_t *row_start,
                               const void *missing_cols, int col_bytes, size_t first_row, size_t n_rows, cudaStream_t copy_s,
                               cudaStream_t comp_s, cudaEvent_t ev[2], fm_ingest *tracks_of = nullptr) {
    if (col_bytes != 1 && col_bytes != 2 && col_bytes != 4) fail(FM_ERR_INVALID_ARG, "col_bytes must be 1 (gap code), 2 or 4");
    if (col_bytes == 2 && m->stride > 65536) fail(FM_ERR_INVALID_ARG, "16-bit columns need a row stride <= 65536");
    if (n_rows && !row_start) fail(FM_ERR_INVALID_ARG, "row_start is NULL");
    const size_t rw = m->rw;
    if (!n_rows || !rw) return;
    if (row_start[0] != 0) fail(FM_ERR_INVALID_ARG, "row_start[0] must be 0 (offsets are relative to the call)");
    const uint64_t total = row_start[n_rows];
    if (total && !missing_cols) fail(FM_ERR_INVALID_ARG, "missing_cols is NULL");
    DevBuf<uint64_t> d_start(n_rows + 1);
    DevBuf<uint8_t> d_cols(std::max<uint64_t>(total * col_bytes, 16));
    CK(cudaStreamSynchronize(stream()));  // fresh (or recycled) scratch is settled before other streams touch it
    static const uint32_t chunk_mb = std::max(1u, env_u32("FM_PACKED_CHUNK_MB", 32));
    const size_t chunk = std::max<size_t>(32, ((size_t)chunk_mb << 20) / (rw * 4));
    int b = 0;
    for (size_t r0 = 0, step = 0; r0 < n_rows; r0 += step, b ^= 1) {
        step = tapered_chunk(n_rows - r0, chunk);
        const size_t r1 = r0 + step;
        if (row_start[r1] < row_start[r0] || row_start[r1] > total) fail(FM_ERR_INVALID_ARG, "row_start is not ascending");
        h2d(m->d_abits + (first_row + r0) * rw, allele_bits + r0 * rw, (r1 - r0) * rw * 4, copy_s);
        h2d(d_start.p + r0, row_start + r0, (r1 - r0 + 1) * 8, copy_s);
        const uint64_t c0 = row_start[r0], c1 = row_start[r1];
        if (c1 > c0)
            h2d(d_cols.p + c0 * col_bytes, static_cast<const uint8_t *>(missing_cols) + c0 * col_bytes, (c1 - c0) * col_bytes,
                copy_s);
        CK(cudaEventRecord(ev[b], copy_s));
        CK(cudaStreamWaitEvent(comp_s, ev[b], 0));
        expand_called_launch(m, d_start.p, d_cols.p, col_bytes, 0, (uint32_t)first_row, (uint32_t)(first_row + r0),
                             (uint32_t)(first_row + r1), comp_s);
        if (set) launch_repack(*set, nullptr, 0, nullptr, 0, 0, (uint32_t)(first_row + r0), (uint32_t)(first_row + r1), comp_s);
        if (tracks_of) ingest_tracks_chunk(tracks_of, first_row + r0, first_row + r1);
    }
    // the scratch lists go back to the allocator ordered after the last kernel that reads them
    CK(cudaEventRecord(ev[b], comp_s));
    CK(cudaStreamWaitEvent(stream(), ev[b], 0));
}

fm_status fm_pack_rows_sparse(const uint8_t *rows, const uint64_t *missing_whole, int missing_mode, size_t first_row,
                              size_t n_rows, size_t n_total_rows, size_t stride, uint32_t *allele_bits,
                              uint64_t *row_missing_start, void *missing_cols, size_t capacity, int col_bytes,
                              int n_threads, size_t *needed) {
    return guarded([&] {  // host only
        const char *err = fm_host_pack_rows_sparse(rows, missing_whole, missing_mode, first_row, n_rows, n_total_rows, stride,
                                                   allele_bits, row_missing_start, missing_cols, capacity, col_bytes,
                                                   n_threads, needed);
        if (err) fail(FM_ERR_INVALID_ARG, err);
    });
}

fm_status fm_ingest_rows_packed_sparse(fm_ingest *h, const uint32_t *allele_bits, const uint64_t *row_missing_start,
                                       const void *missing_cols, int col_bytes, size_t first_row, size_t n_rows) {
    return guarded([&] {
        FM_NVTX("fm_ingest_rows_packed_sparse (H2D packed + expand + K1p compress)");
        if (!h) fail(FM_ERR_INVALID_ARG, "ingest handle is NULL");
        fm_matrix *m = h->m;
        if (first_row > m->V || n_rows > m->V - first_row) fail(FM_ERR_INVALID_ARG, "row range outside the matrix");
        if (h->stage[0]) fail(FM_ERR_INVALID_ARG, "this ingest already received u8 rows (fm_ingest_rows)");
        if (m->in_band) fail(FM_ERR_INVALID_ARG, "packed rows carry their own missingness: begin with FM_MISSING_BITMAP");
        if (!m->has_missing) fail(FM_ERR_INVALID_ARG, "matrix was declared without missing data: use fm_ingest_rows_packed");
        if (n_rows && m->stride && !allele_bits) fail(FM_ERR_INVALID_ARG, "allele_bits is NULL");
        set_dev(m);
        static const uint32_t trace = env_u32("FM_INGEST_TRACE", 0);
        std::vector<std::pair<const char *, std::chrono::steady_clock::time_point>> tr;
        auto mark = [&](const char *what) {
            if (trace) tr.emplace_back(what, std::chrono::steady_clock::now());
        };
        mark("start");
        const bool first_call = !m->d_abits;
        ensure_packed_storage(m, true);
        if (first_call) CK(cudaStreamSynchronize(stream()));
        mark("storage");
        if (!h->set.d_desc && !h->all.empty()) h->set.build(h->all);
        mark("plans");
        if (!h->timing_started && n_rows) {
            CK(cudaEventRecord(h->t_copy0, h->copy_s));
            ingest_early_setup(h);
            CK(cudaEventRecord(h->t_comp0, h->comp_s));
            h->timing_started = true;
        }
        packed_sparse_rows(m, h->all.empty() ? nullptr : &h->set, allele_bits, row_missing_start, missing_cols, col_bytes,
                           first_row, n_rows, h->copy_s, h->comp_s, h->copied, h);
        mark("queued");
        h->rows_done += n_rows;
        CK(cudaEventRecord(h->t_copy1, h->copy_s));
        CK(cudaEventRecord(h->t_comp1, h->comp_s));
        ingest_late_setup(h);
        mark("positions");
        CK(cudaStreamSynchronize(h->copy_s));  // the caller's buffers are free again on return
        mark("copies done");
        if (trace) {
            for (size_t i = 1; i < tr.size(); ++i)
                fprintf(stderr, "[ingest] %-12s +%.3f ms\n", tr[i].first,
                        std::chrono::duration<double, std::milli>(tr[i].second - tr[i - 1].second).count());
        }
    });
}

fm_status fm_matrix_create_packed_sparse(const uint32_t *allele_bits, const uint64_t *row_missing_start,
                                         const void *missing_cols, int col_bytes, size_t V, size_t S, size_t ploidy,
                                         const int64_t *positions, fm_matrix **out) {
    return guarded([&] {
        FM_NVTX("fm_matrix_create_packed_sparse (H2D packed + expand)");
        if (!out) fail(FM_ERR_INVALID_ARG, "out is NULL");
        *out = nullptr;
        require_device();
        CK(cudaSetDevice(t_device));
        fm_matrix *m = matrix_common(V, S, ploidy, 1, positions);
        try {
            m->has_missing = true;
            m->streamed = true;
            ensure_packed_storage(m, true);
            if ((V * (size_t)m->rw) != 0 && !allele_bits) fail(FM_ERR_INVALID_ARG, "allele_bits is NULL");
            Timer tm;
            tm.start();
            EventPairs evs;
            cudaEvent_t ev[2] = {evs.next(), evs.next()};
            packed_sparse_rows(m, nullptr, allele_bits, row_missing_start, missing_cols, col_bytes, 0, V, stream(), stream(), ev);
            m->d_pos = static_cast<int64_t *>(dev_alloc(std::max<size_t>(V, 1) * 8));
            if (V) CK(cudaMemcpyAsync(m->d_pos, m->pos.data(), V * 8, cudaMemcpyHostToDevice, stream()));
            tm.stop();
            CK(cudaStreamSynchronize(stream()));
            t_tim.h2d_ms += tm.ms();
        } catch (...) {
            fm_matrix_release(m);
            throw;
        }
        *out = m;
    });
}

// u8 rows in, 2 bits per genotype over PCIe: the library packs chunk i+1 on the host (fm_pack_rows, several
// threads, reading the caller's buffer where it lies -- pageable memory needs no bounce copy) while the DMA of
// chunk i and the compress pass of chunk i-1 run.  Same arguments and semantics as fm_ingest_rows.
fm_status fm_ingest_rows_pack(fm_ingest *h, const uint8_t *rows, const uint64_t *missing_whole, size_t first_row,
                              size_t n_rows, int n_threads) {
    return guarded([&] {
        FM_NVTX("fm_ingest_rows_pack (host pack + H2D + K1p)");
        if (!h) fail(FM_ERR_INVALID_ARG, "ingest handle is NULL");
        fm_matrix *m = h->m;
        if (first_row > m->V || n_rows > m->V - first_row) fail(FM_ERR_INVALID_ARG, "row range outside the matrix");
        if (h->stage[0]) fail(FM_ERR_INVALID_ARG, "this ingest already received u8 rows (fm_ingest_rows)");
        if (n_rows && m->stride && !rows) fail(FM_ERR_INVALID_ARG, "rows is NULL");
        const int mode = m->in_band ? FM_MISSING_IN_BAND : (m->has_missing ? FM_MISSING_BITMAP : FM_MISSING_NONE);
        if (mode == FM_MISSING_BITMAP && !missing_whole) fail(FM_ERR_INVALID_ARG, "matrix was declared with a missing bitmap");
        set_dev(m);
        const bool first_call = !m->d_abits;
        ensure_packed_storage(m, m->has_missing);
        if (first_call) CK(cudaStreamSynchronize(stream()));
        if (!h->set.d_desc && !h->all.empty()) h->set.build(h->all);
        if (!h->timing_started && n_rows) {
            CK(cudaEventRecord(h->t_copy0, h->copy_s));
            ingest_early_setup(h);
            CK(cudaEventRecord(h->t_comp0, h->comp_s));
            h->timing_started = true;
        }
        const size_t rw = m->rw, stride = m->stride;
        if (!rw) {
            h->rows_done += n_rows;
            return;
        }
        const size_t planes = m->has_missing ? 2 : 1;
        const size_t chunk = std::max<size_t>(1, PinnedPool::kBytes / (rw * 4 * planes));
        for (int i = 0; i < 2; ++i)
            if (!h->pin[i]) {
                h->pin[i] = g_pinned.take();
                CK(cudaEventCreateWithFlags(&h->pin_free[i], cudaEventDisableTiming));
            }
        int b = 0;
        for (size_t r0 = first_row; r0 < first_row + n_rows; r0 += chunk, b ^= 1) {
            const size_t r1 = std::min(first_row + n_rows, r0 + chunk), nr = r1 - r0;
            if (h->pin_used[b]) CK(cudaEventSynchronize(h->pin_free[b]));  // its previous DMA has drained
            uint32_t *pa = reinterpret_cast<uint32_t *>(h->pin[b]);
            uint32_t *pc = m->has_missing ? pa + nr * rw : nullptr;
            const auto t0 = std::chrono::steady_clock::now();
            const char *err = fm_host_pack_rows(rows + (r0 - first_row) * stride, missing_whole, mode, r0, nr, m->V, stride,
                                                pa, pc, n_threads);
            if (err) fail(FM_ERR_INVALID_ARG, err);
            h->pack_ms += std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
            CK(cudaMemcpyAsync(m->d_abits + r0 * rw, pa, nr * rw * 4, cudaMemcpyHostToDevice, h->copy_s));
            if (pc) CK(cudaMemcpyAsync(m->d_cbits + r0 * rw, pc, nr * rw * 4, cudaMemcpyHostToDevice, h->copy_s));
            CK(cudaEventRecord(h->pin_free[b], h->copy_s));
            h->pin_used[b] = true;
            CK(cudaStreamWaitEvent(h->comp_s, h->pin_free[b], 0));
            launch_repack(h->set, nullptr, 0, nullptr, 0, 0, (uint32_t)r0, (uint32_t)r1, h->comp_s);
            ingest_tracks_chunk(h, r0, r1);
        }
        h->rows_done += n_rows;
        CK(cudaEventRecord(h->t_copy1, h->copy_s));
        CK(cudaEventRecord(h->t_comp1, h->comp_s));
        ingest_late_setup(h);
        CK(cudaStreamSynchronize(h->copy_s));
    });
}

fm_status fm_matrix_create_packed(const uint32_t *allele_bits, const uint32_t *called_bits, size_t V, size_t S,
                                  size_t ploidy, const int64_t *positions, fm_matrix **out) {
    return guarded([&] {
        FM_NVTX("fm_matrix_create_packed (H2D packed rows)");
        if (!out) fail(FM_ERR_INVALID_ARG, "out is NULL");
        *out = nullptr;
        require_device();
        CK(cudaSetDevice(t_device));
        fm_matrix *m = matrix_common(V, S, ploidy, 1, positions);
        try {
            m->has_missing = called_bits != nullptr;
            m->streamed = true;  // no u8 rows: groups come from the packed rows
            ensure_packed_storage(m, m->has_missing);
            const size_t words = V * (size_t)m->rw;
            if (words && !allele_bits) fail(FM_ERR_INVALID_ARG, "allele_bits is NULL");
            Timer tm;
            tm.start();
            h2d(m->d_abits, allele_bits, words * 4, stream());
            if (called_bits) h2d(m->d_cbits, called_bits, words * 4, stream());
            m->d_pos = static_cast<int64_t *>(dev_alloc(std::max<size_t>(V, 1) * 8));
            if (V) CK(cudaMemcpyAsync(m->d_pos, m->pos.data(), V * 8, cudaMemcpyHostToDevice, stream()));
            tm.stop();
            t_tim.h2d_ms += tm.ms();
        } catch (...) {
            fm_matrix_release(m);
            throw;
        }
        *out = m;
    });
}

fm_status fm_ingest_finish(fm_ingest *h, fm_matrix **matrix_out, fm_group **groups_out, fm_partition **parts_out) {
    return guarded([&] {
        if (!h) fail(FM_ERR_INVALID_ARG, "ingest handle is NULL");
        if (h->rows_done != h->m->V)
            fail(FM_ERR_INVALID_ARG, "fm_ingest_finish before every row was ingested");
        if ((!groups_out && !h->groups.empty()) || (!parts_out && !h->parts.empty()) || !matrix_out)
            fail(FM_ERR_INVALID_ARG, "output arrays are NULL");
        set_dev(h->m);
        ingest_late_setup(h);
        CK(cudaStreamSynchronize(h->comp_s));
        if (IngestTracks *T = h->tracks.get()) {  // requested tracks: everything was computed as the rows arrived
            const size_t n = T->hi - T->lo;
            DevBuf<int64_t> d_p1;
            if (n) {
                for (size_t i = 0; i < T->act.size(); ++i)
                    if (!T->direct[i]) {  // pageable output rows: copy them out now
                        T->own_pi[i].download(T->pi_out + T->act_idx[i] * T->capacity, n);
                        T->own_th[i].download(T->theta_out + T->act_idx[i] * T->capacity, n);
                    }
                if (!T->pos_done) download_positions_plus1(h->m, T->lo, n, T->pos_out, d_p1);  // stats.rs:4746
                CK(cudaStreamSynchronize(stream()));
                const double NaN = std::numeric_limits<double>::quiet_NaN();
                for (size_t row : T->nan_rows)
                    for (size_t k = 0; k < n; ++k) T->pi_out[row * T->capacity + k] = T->theta_out[row * T->capacity + k] = NaN;
            }
        }
        if (h->timing_started) {
            float a = 0.f, b = 0.f;
            CK(cudaEventElapsedTime(&a, h->t_copy0, h->t_copy1));
            CK(cudaEventElapsedTime(&b, h->t_comp0, h->t_comp1));
            t_tim.h2d_ms += a;      // span of the copy stream
            t_tim.repack_ms += b;   // span of the repack stream (overlaps the copies)
            t_tim.pack_ms += h->pack_ms;  // host packer (fm_ingest_rows_pack), overlaps both
        }
        for (fm_group *g : h->all)
            if (g->count_only) g->have_counts = true;
        *matrix_out = h->m;
        for (size_t i = 0; i < h->groups.size(); ++i) groups_out[i] = h->groups[i];
        for (size_t i = 0; i < h->parts.size(); ++i) parts_out[i] = h->parts[i];
        ingest_destroy(h, false);
    });
}

fm_status fm_ingest_abort(fm_ingest *h) {
    ingest_destroy(h, true);
    return FM_OK;
}

// ------------------------------------------------------------------------------------ Hudson
static void check_pair(fm_group *g1, fm_group *g2, bool allow_distinct_matrices = false) {
    if (!g1 || !g2) fail(FM_ERR_INVALID_ARG, "group is NULL");
    if (g1->m == g2->m) return;
    // Two contexts with their own matrices are only meaningful on the summaries path, which
    // works on the per-group count arrays (stats.rs:1554-1623); variants_compatible
    // (stats.rs:3399-3401) still has to hold.
    if (!allow_distinct_matrices || g1->m->device != g2->m->device || g1->m->pos != g2->m->pos)
        fail(FM_ERR_PARSE, "Variant slices differ in positions/length.");  // stats.rs:3451-3455
}

// regional Dxy of calculate_d_xy_hudson (stats.rs:2403-2524) given totals of the matching variant
static void dxy_outcome(int path, fm_group *g1, fm_group *g2, int64_t L, size_t raw_n1, size_t raw_n2,
                        const HudsonTotals &t, double *d, bool *some) {
    *some = false;
    *d = 0.0;
    if (raw_n1 == 0 || raw_n2 == 0) return;                                 // :2434-2446
    if (path == FM_HUDSON_DENSE && (g1->n == 0 || g2->n == 0)) return;      // :2532-2534
    const int64_t eff = sat_sub(L, (int64_t)t.skipped);
    if (eff > 0) {
        *d = t.dxy / (double)eff;
        *some = true;
    }
}

fm_status fm_hudson_dxy(fm_group *g1, fm_group *g2, int64_t L1, int64_t L2, int path, size_t raw_n1,
                        size_t raw_n2, double *d_xy, int *is_some) {
    return guarded([&] {
        if (!d_xy || !is_some) fail(FM_ERR_INVALID_ARG, "NULL argument");
        *is_some = 0;
        *d_xy = 0.0;
        if (L1 <= 0) fail(FM_ERR_INVALID_REGION, "Sequence length must be positive for Dxy calculation");
        if (L1 != L2) fail(FM_ERR_PARSE, "Sequence length mismatch in Dxy calculation");
        check_pair(g1, g2, path == FM_HUDSON_SUMMARIES);
        require_device();
        if (raw_n1 == 0 || raw_n2 == 0) return;
        ensure_counts_pair(g1, g2);
        set_dev(g1->m);
        const int variant = path == FM_HUDSON_SUMMARIES ? -1
                            : path == FM_HUDSON_DENSE   ? dense_variant(g1->m)
                                                        : FM_HV_SPARSE;
        HudsonTotals t = run_hudson_counts(g1, g2, 0, (uint32_t)g1->m->V, variant, fm::HudsonEpilogue{});
        bool some;
        dxy_outcome(path, g1, g2, L1, raw_n1, raw_n2, t, d_xy, &some);
        *is_some = some;
    });
}

// calculate_pi_for_population for one side of a Hudson call, given the matching totals
static double pi_outcome(int path, fm_group *g, int64_t L, size_t raw_n, double pi_sum, uint64_t unc) {
    const double NaN = std::numeric_limits<double>::quiet_NaN();
    if (path == FM_HUDSON_SPARSE) {
        if (raw_n <= 1) return NaN;
    } else if (g->n <= 1)
        return NaN;
    if (L < 0) return 0.0;
    if (L == 0) return std::numeric_limits<double>::infinity();
    if (path == FM_HUDSON_SPARSE && g->n <= 1) return NaN;
    const uint64_t skipped = (path == FM_HUDSON_DENSE && !g->m->has_missing) ? 0 : unc;
    const int64_t eff = sat_sub(L, (int64_t)skipped);
    if (eff == 0) return NaN;
    return pi_sum / (double)eff;
}

fm_status fm_hudson_pair(fm_group *g1, fm_group *g2, int64_t L1, int64_t L2, int path, int has_region,
                         int64_t rs, int64_t re, size_t raw_n1, size_t raw_n2, fm_hudson_outcome *out,
                         fm_hudson_sites *sites, size_t *n_sites) {
    return guarded([&] {
        FM_NVTX("fm_hudson_pair (K3 fused pass / light kernel)");
        if (!out) fail(FM_ERR_INVALID_ARG, "out is NULL");
        std::memset(out, 0, sizeof(*out));
        if (n_sites) *n_sites = 0;
        if (L1 <= 0)
            fail(FM_ERR_INVALID_REGION, "Sequence length must be positive for Hudson FST calculation.");
        if (L1 != L2)
            fail(FM_ERR_PARSE,
                 "Sequence length mismatch between population contexts for Hudson FST calculation.");
        check_pair(g1, g2, path == FM_HUDSON_SUMMARIES && !has_region);
        require_device();
        fm_matrix *m = g1->m;
        set_dev(m);
        const uint32_t V = (uint32_t)m->V;
        const int aux_variant = path == FM_HUDSON_SUMMARIES ? -1
                                : path == FM_HUDSON_DENSE   ? dense_variant(m)
                                                            : FM_HV_SPARSE;
        HudsonTotals main_t{0, 0, 0, 0, 0, 0, 0, 0}, aux_t{0, 0, 0, 0, 0, 0, 0, 0};
        bool aux_done = false;

        // --- per-site outputs (region => sparse per-site path; else the path's own per-site form)
        uint32_t lo = 0, hi = V;
        int site_variant = aux_variant;
        if (has_region) {
            site_range(m, rs, re, lo, hi);
            site_variant = FM_HV_SPARSE;  // stats.rs:3473-3475
        }
        const bool emit_sites = sites && site_variant >= 0;
        const size_t ns = hi - lo;
        DevBuf<double> sd;
        DevBuf<uint32_t> su;
        fm::HudsonEpilogue e{};
        if (emit_sites && ns) {
            if (ns > sites->capacity) fail(FM_ERR_INVALID_ARG, "per-site output capacity too small");
            sd.alloc(ns * 6);
            su.alloc(ns * 2);
            e.fst = sd.p;
            e.dxy = sd.p + ns;
            e.pi1 = sd.p + 2 * ns;
            e.pi2 = sd.p + 3 * ns;
            e.num = sd.p + 4 * ns;
            e.den = sd.p + 5 * ns;
            e.n1_out = su.p;
            e.n2_out = su.p + ns;
        }
        // counts: fused two-group sweep when nothing is cached yet and the main pass covers the
        // whole matrix; otherwise per-group plane passes (cached) + light kernels on the counts.
        bool fused = false;
        if (g1 != g2 && g1->m == g2->m && lo == 0 && hi == V && V > 0 && g1->n_bits == 1) {
            std::unique_lock<std::mutex> l1(g1->mu, std::defer_lock), l2(g2->mu, std::defer_lock);
            std::lock(l1, l2);
            if (!g1->have_counts && !g2->have_counts) {
                for (fm_group *g : {g1, g2}) alloc_counts(g);
                // ONE sweep of both groups' planes (fm_k_plane_pass_seq, pair units): every warp streams a batch of
                // group 1, then the same batch of group 2, and evaluates the Hudson components in place -- the
                // groups' counts and summary scalars are cached for later calls AND the Hudson partials (plus the
                // optional per-site values) come out of the same pass (stats.rs:3179-3278).
                fm_group *pair[2] = {g1, g2};
                const uint32_t nb = (V + 31) / 32;
                DevBuf<double> ppi[2], pd((size_t)nb * 5);
                DevBuf<uint32_t> ppu[2], pu((size_t)nb * 3);
                std::vector<fm::RowSeg> segs(2);
                for (int k = 0; k < 2; ++k) {
                    ppi[k].alloc(nb);
                    ppu[k].alloc((size_t)nb * 2);
                    fm::DivEpilogue de{};
                    set_tables(de, pair[k]);
                    de.pi_form = FM_PIFORM_COUNTS;
                    de.part_pi = ppi[k].p;
                    de.part_u = ppu[k].p;
                    de.alt_out = pair[k]->d_alt;
                    de.called_out = called_cache(pair[k]);
                    segs[k] = div_seg(pair[k], de, 0, V);
                }
                fm::HudsonEpilogue he = e;
                he.variant = site_variant;
                he.part_d = pd.p;
                he.part_u = pu.p;
                std::vector<fm::HudsonEpilogue> hv{he};
                RowPlan plan;
                Timer tm;
                tm.start();
                const bool ok = plan_rows(segs, &hv, plan);
                if (ok) launch_rows(plan, m->device);
                tm.stop();
                if (ok) {
                    const fm::PassGeom G = batch_range(0, V);
                    for (int k = 0; k < 2; ++k) {
                        double od[1];
                        uint64_t ou[2];
                        finish_partials(ppi[k].p, 1, ppu[k].p, 2, G, od, ou);
                        pair[k]->pi_sum = od[0];
                        pair[k]->seg = ou[0];
                        pair[k]->unc = ou[1];
                        pair[k]->have_counts = true;
                    }
                    double od[5];
                    uint64_t ou[3];
                    finish_partials(pd.p, 5, pu.p, 3, G, od, ou);
                    main_t = HudsonTotals{od[0], od[1], od[2], od[3], od[4], ou[0], ou[1], ou[2]};
                    t_tim.stats_ms += tm.ms();
                } else {  // rows too wide for the row pass: two chunked passes, then the light kernel
                    DivResult r[2];
                    run_diversity_multi(pair, 2, 0, V, FM_PIFORM_COUNTS, nullptr, nullptr, nullptr, 0, nullptr, 0, r, true);
                    for (int k = 0; k < 2; ++k) {
                        pair[k]->seg = r[k].seg;
                        pair[k]->unc = r[k].unc;
                        pair[k]->pi_sum = r[k].pi_sum;
                        pair[k]->have_counts = true;
                    }
                    main_t = run_hudson_counts(g1, g2, lo, hi, site_variant, e);
                }
                fused = true;
            }
        }
        if (!fused) {
            ensure_counts_pair(g1, g2);
            main_t = run_hudson_counts(g1, g2, lo, hi, site_variant, e);
        }
        if (!has_region || (lo == 0 && hi == V && site_variant == aux_variant)) {
            aux_t = main_t;
            aux_done = true;
        }
        if (!aux_done) aux_t = run_hudson_counts(g1, g2, 0, V, aux_variant, fm::HudsonEpilogue{});

        // --- regional FST (stats.rs:3505-3509); DENSE/SPARSE with no variants -> (0,0)
        const double num_sum = main_t.num, den_sum = main_t.den;
        if (den_sum > FM_FST_EPSILON) {
            out->fst = num_sum / den_sum;
            out->some |= 1u;
        }
        // --- auxiliary pi / Dxy (stats.rs:3512-3566)
        double pi1_raw, pi2_raw;
        bool dsome = false;
        double dval = 0.0;
        if (path == FM_HUDSON_SUMMARIES && !has_region) {
            // calculate_pi_from_summary_with_precomputed(Some(totals.piX_sum))
            pi1_raw = pi_outcome(path, g1, L1, raw_n1, aux_t.pi1, g1->unc);
            pi2_raw = pi_outcome(path, g2, L2, raw_n2, aux_t.pi2, g2->unc);
            if (raw_n1 != 0 && raw_n2 != 0) {
                const int64_t eff = sat_sub(L1, (int64_t)aux_t.skipped);
                if (eff > 0) {
                    dval = aux_t.dxy / (double)eff;
                    dsome = true;
                }
            }
        } else if (path == FM_HUDSON_SUMMARIES) {
            // calculate_pi_for_population -> calculate_pi_from_summary (cached pi_sum)
            pi1_raw = pi_outcome(path, g1, L1, raw_n1, g1->pi_sum, g1->unc);
            pi2_raw = pi_outcome(path, g2, L2, raw_n2, g2->pi_sum, g2->unc);
            dxy_outcome(path, g1, g2, L1, raw_n1, raw_n2, aux_t, &dval, &dsome);
        } else {
            pi1_raw = pi_outcome(path, g1, L1, raw_n1, aux_t.pi1, aux_t.unc1);
            pi2_raw = pi_outcome(path, g2, L2, raw_n2, aux_t.pi2, aux_t.unc2);
            dxy_outcome(path, g1, g2, L1, raw_n1, raw_n2, aux_t, &dval, &dsome);
        }
        if (std::isfinite(pi1_raw)) { out->pi_pop1 = pi1_raw; out->some |= 4u; }
        if (std::isfinite(pi2_raw)) { out->pi_pop2 = pi2_raw; out->some |= 8u; }
        if (dsome) { out->d_xy = dval; out->some |= 2u; }
        if ((out->some & 12u) == 12u) {
            out->pi_xy_avg = 0.5 * (out->pi_pop1 + out->pi_pop2);
            out->some |= 16u;
        }
        // --- copy per-site outputs
        if (emit_sites && ns) {
            Timer tm;
            tm.start();
            double *dst[6] = {sites->fst, sites->d_xy, sites->pi_pop1, sites->pi_pop2,
                              sites->num_component, sites->den_component};
            for (int i = 0; i < 6; ++i)
                if (dst[i]) CK(cudaMemcpyAsync(dst[i], sd.p + (size_t)i * ns, ns * 8, cudaMemcpyDeviceToHost, stream()));
            if (sites->n1_called) CK(cudaMemcpyAsync(sites->n1_called, su.p, ns * 4, cudaMemcpyDeviceToHost, stream()));
            if (sites->n2_called) CK(cudaMemcpyAsync(sites->n2_called, su.p + ns, ns * 4, cudaMemcpyDeviceToHost, stream()));
            tm.stop();
            CK(cudaStreamSynchronize(stream()));
            t_tim.d2h_ms += tm.ms();
            if (sites->position)
                for (size_t i = 0; i < ns; ++i) sites->position[i] = m->pos[lo + i] + 1;
        }
        if (n_sites) *n_sites = (site_variant >= 0) ? ns : 0;
    });
}

// ------------------------------------------------------------------------------------ W&C (fm_wc.cuh)
fm_status fm_partition_create(fm_matrix *m, const uint16_t *left, const uint16_t *right, size_t n_samples,
                              size_t n_groups, fm_partition **out) {
    return guarded([&] {
        FM_NVTX("fm_partition_create (K1 count pass)");
        if (!out || !m) fail(FM_ERR_INVALID_ARG, "NULL argument");
        *out = nullptr;
        if (n_samples && (!left || !right)) fail(FM_ERR_INVALID_ARG, "membership arrays are NULL");
        if (n_groups >= 0xFFFF) fail(FM_ERR_INVALID_ARG, "too many groups");
        require_device();
        fm_partition *p = new fm_partition();
        p->m = m;
        p->G = n_groups;
        fm_matrix_retain(m);
        try {
            if (m->streamed && !m->packed)
                fail(FM_ERR_UNSUPPORTED,
                     "this matrix was ingested in streaming mode: declare partitions with fm_ingest_add_partition");
            std::vector<std::vector<uint32_t>> cols = partition_columns(m, left, right, n_samples, n_groups);
            set_dev(m);
            const size_t per = 2 * std::max<size_t>(m->V, 1);
            p->d_counts_slab = static_cast<uint32_t *>(dev_alloc((n_groups + 1) * per * sizeof(uint32_t)));
            for (size_t g = 0; g <= n_groups; ++g)
                p->groups.push_back(alloc_group(m, std::move(cols[g]), true, p->d_counts_slab + g * per));
            repack_resident(m, p->groups);  // the u8 matrix is read once for all G + 1 groups
        } catch (...) {
            fm_partition_release(p);
            throw;
        }
        *out = p;
    });
}

fm_status fm_partition_release(fm_partition *p) {
    if (!p) return FM_OK;
    if (p->m) cudaSetDevice(p->m->device);
    dev_free(p->d_wc_tab);
    for (fm_group *g : p->groups) fm_group_release(g);
    dev_free(p->d_counts_slab);
    fm_matrix_release(p->m);
    delete p;
    return FM_OK;
}

static void window_ranges(const fm_matrix *m, const int64_t *windows, size_t n, std::vector<uint32_t> &lo,
                          std::vector<uint32_t> &hi);

static fm_fst_estimate classify_estimate(double a, double b, uint64_t sites) {
    // threshold ladder of stats.rs:2237-2270 / 2297-2328 (same as :1785-1811)
    fm_fst_estimate e;
    e.sum_a = a;
    e.sum_b = b;
    e.sites = sites;
    e.value = std::numeric_limits<double>::quiet_NaN();
    e.state = fm_fst_state(a, b);
    if (e.state == 0) e.value = a / (a + b);
    return e;
}

namespace {
struct WcSiteOut {
    int32_t *state = nullptr;
    double *a = nullptr, *b = nullptr;
    uint32_t *sizes = nullptr;
    double *pair_a = nullptr, *pair_b = nullptr;
};
struct WcWindowTotals {  // host copies, one entry per window
    std::vector<double> overall;     // [n_w][2]
    std::vector<uint64_t> sites;     // [n_w]
    std::vector<double> pair;        // [n_w][n_pairs][2]
    std::vector<uint64_t> pair_n;    // [n_w][n_pairs]
};

// Reciprocal tables of the biallelic W&C kernels (fm_wc.cuh): every divisor of the pair formulas that depends
// only on sample sizes is an integer n <= n_i + n_j (or n/2, n/2 - 1, 2 (n/2)^2), so its correctly rounded
// reciprocal comes from a table built once per partition with IEEE divisions on the host.
fm::WcTables wc_tables(fm_partition *p) {
    std::lock_guard<std::mutex> lk(p->mu);
    if (!p->d_wc_tab) {
        uint32_t top1 = 0, top2 = 0;  // the two largest group capacities
        for (size_t g = 0; g < p->G; ++g) {
            const uint32_t n = p->groups[g]->n;
            if (n > top1) { top2 = top1; top1 = n; }
            else if (n > top2) top2 = n;
        }
        const uint32_t n_max = std::max(top1 + top2, 2u);
        std::vector<double> T(2 * ((size_t)n_max + 1), 0.0);
        for (uint32_t n = 1; n <= n_max; ++n) {
            const double nd = (double)n, n_bar = nd / 2.0;
            T[n] = 1.0 / nd;
            T[(size_t)n_max + 1 + n] = 1.0 / (2.0 * n_bar * n_bar);
        }
        p->d_wc_tab = static_cast<double *>(dev_alloc(T.size() * 8));
        CK(cudaMemcpyAsync(p->d_wc_tab, T.data(), T.size() * 8, cudaMemcpyHostToDevice, stream()));
        CK(cudaStreamSynchronize(stream()));
        p->wc_n_max = n_max;
    }
    return fm::WcTables{p->d_wc_tab, p->d_wc_tab + p->wc_n_max + 1, p->wc_n_max};
}

// K4 over a list of windows given as site-index ranges: segments cut at multiples of
// kWcSegSites, one warp per segment, then the per-window fold.  Per-site outputs (host
// pointers, indexed v - out_base) are only meaningful for a single window.
void run_wc(fm_partition *p, const std::vector<uint32_t> &wlo, const std::vector<uint32_t> &whi,
            const WcSiteOut &so, uint32_t out_base, size_t n_out_sites, WcWindowTotals &tot) {
    fm_matrix *m = p->m;
    const uint32_t G = (uint32_t)p->G;
    const uint32_t n_pairs = G * (G > 0 ? G - 1 : 0) / 2;
    const size_t nw = wlo.size();
    tot.overall.assign(nw * 2, 0.0);
    tot.sites.assign(nw, 0);
    tot.pair.assign(nw * std::max(n_pairs, 1u) * 2, 0.0);
    tot.pair_n.assign(nw * std::max(n_pairs, 1u), 0);
    std::vector<uint32_t> seg_lo, seg_hi, wseg(nw + 1, 0);
    static const uint32_t seg_sites = env_u32("FM_WC_SEG", fm::kWcSegSites);  // tuning only: changes the association
    for (size_t w = 0; w < nw; ++w) {
        wseg[w] = (uint32_t)seg_lo.size();
        for (uint32_t v = wlo[w]; v < whi[w];) {
            const uint32_t e = std::min<uint64_t>(whi[w], ((uint64_t)v / seg_sites + 1) * seg_sites);
            seg_lo.push_back(v);
            seg_hi.push_back(e);
            v = e;
        }
    }
    wseg[nw] = (uint32_t)seg_lo.size();
    const uint32_t n_seg = (uint32_t)seg_lo.size();
    if (n_seg == 0) return;
    for (fm_group *g : p->groups) ensure_counts(g);
    set_dev(m);
    const bool multi = p->groups[0]->n_bits > 1;
    const uint32_t A = multi ? 1u << p->groups[0]->n_bits : 2u;
    std::vector<const uint32_t *> h_alt(G + 1), h_cnt(G + 1);
    for (uint32_t g = 0; g <= G; ++g) {
        h_alt[g] = multi ? p->groups[g]->d_acount : p->groups[g]->d_alt;
        h_cnt[g] = p->groups[g]->d_cnt;
    }
    DevBuf<const uint32_t *> d_alt(G + 1), d_cnt(G + 1);
    d_alt.upload(h_alt.data(), G + 1);
    d_cnt.upload(h_cnt.data(), G + 1);
    std::vector<uint16_t> pi(std::max(n_pairs, 1u)), pj(std::max(n_pairs, 1u));
    {
        uint32_t k = 0;
        for (uint32_t i = 0; i < G; ++i)
            for (uint32_t j = i + 1; j < G; ++j, ++k) {
                pi[k] = (uint16_t)i;
                pj[k] = (uint16_t)j;
            }
    }
    DevBuf<uint16_t> d_pi(pi.size()), d_pj(pj.size());
    d_pi.upload(pi.data(), pi.size());
    d_pj.upload(pj.data(), pj.size());
    DevBuf<uint32_t> d_slo(n_seg), d_shi(n_seg), d_wseg(nw + 1);
    d_slo.upload(seg_lo.data(), n_seg);
    d_shi.upload(seg_hi.data(), n_seg);
    d_wseg.upload(wseg.data(), nw + 1);

    fm::WcParams W{};
    W.alt = multi ? nullptr : d_alt.p;
    W.acount = multi ? d_alt.p : nullptr;
    W.A = A;
    W.cnt = d_cnt.p;
    W.G = G;
    W.n_pairs = n_pairs;
    W.pair_i = d_pi.p;
    W.pair_j = d_pj.p;
    W.seg_lo = d_slo.p;
    W.seg_hi = d_shi.p;
    W.n_seg = n_seg;
    W.out_base = out_base;
    const size_t ns = n_out_sites;
    DevBuf<int32_t> d_state;
    DevBuf<double> d_sa, d_sb, d_pa, d_pb;
    DevBuf<uint32_t> d_sizes;
    if (so.state && ns) { d_state.alloc(ns); W.site_state = d_state.p; }
    if (so.a && ns) { d_sa.alloc(ns); W.site_a = d_sa.p; }
    if (so.b && ns) { d_sb.alloc(ns); W.site_b = d_sb.p; }
    if (so.sizes && G && ns) { d_sizes.alloc(ns * G); W.site_sizes = d_sizes.p; }
    if (so.pair_a && so.pair_b && n_pairs && ns) {
        d_pa.alloc(ns * n_pairs);
        d_pb.alloc(ns * n_pairs);
        W.pair_a = d_pa.p;
        W.pair_b = d_pb.p;
    }
    DevBuf<double> d_po((size_t)n_seg * 2), d_pp((size_t)n_seg * std::max(n_pairs, 1u) * 2);
    DevBuf<uint32_t> d_pc((size_t)n_seg), d_pn((size_t)n_seg * std::max(n_pairs, 1u));
    W.part_overall = d_po.p;
    W.part_counts = d_pc.p;
    W.part_pair = d_pp.p;
    W.part_pair_n = d_pn.p;

    // multi-allelic kernel geometry: pair warps (lane = pair, KP pairs per lane in registers) + one overall warp per
    // CTA, one CTA per segment; the biallelic path has its own pairs / overall kernels (below)
    static const uint32_t kp_pref = env_u32("FM_WC_KP", 1);
    uint32_t n_pw = std::max(1u, std::min<uint32_t>(fm::kWcMaxPairWarps, (n_pairs + 32 * kp_pref - 1) / (32 * kp_pref)));
    const uint32_t kp_need = std::max(1u, (n_pairs + n_pw * 32 - 1) / (n_pw * 32));
    const size_t smem = multi ? fm::fm_wc_multi_cta_smem(G, A) : 0;
    if (multi) {
        if (kp_need > fm::kWcMaxKP) fail(FM_ERR_UNSUPPORTED, "too many populations for the W&C kernel (pairs per lane)");
        if (smem > 200 * 1024) fail(FM_ERR_UNSUPPORTED, "too many populations for the W&C kernel's staging");
    }
    W.n_pair_warps = n_pw;
    const uint32_t blocks = std::max<uint32_t>(1, std::min<uint32_t>(n_seg, 8u * sm_count(m->device)));
    Timer tm;
    tm.start();
    EventPairs wc_events;
    cudaEvent_t wc_ready = wc_events.next();
    if (multi) {
        const uint32_t threads = (n_pw + 1) * 32;
        auto launch = [&](auto kern) {
            CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            kern<<<blocks, threads, smem, stream()>>>(W);
        };
        if (kp_need <= 1) launch(fm::fm_k_wc_multi<1>);
        else if (kp_need <= 2) launch(fm::fm_k_wc_multi<2>);
        else if (kp_need <= 4) launch(fm::fm_k_wc_multi<4>);
        else launch(fm::fm_k_wc_multi<8>);
        CK(cudaGetLastError());
        g_launches++;
    } else {
        const fm::WcTables T = wc_tables(p);
        CK(cudaEventRecord(wc_ready, stream()));
        if (n_pairs) {
            // producer / consumer pairs kernel: task = (segment, chunk of 352 pair slots), grid-strided over a
            // persistent grid of two CTAs per SM
            const size_t psm = fm::fm_wc_pc_smem(G);
            if (psm > 200 * 1024) fail(FM_ERR_UNSUPPORTED, "too many populations for the W&C kernel's staging");
            const uint32_t n_chunks = (n_pairs + fm::kWcPcPairWarps * 32 - 1) / (fm::kWcPcPairWarps * 32);
            static const uint32_t su = env_u32("FM_WC_SITES_PER_STEP", 1);
            auto launch = [&](auto kern) {
                CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psm));
                int per_sm = 1;
                CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, (int)((fm::kWcPcPairWarps + 1) * 32), psm));
                const uint64_t tasks = (uint64_t)n_seg * n_chunks;
                const uint32_t grid = (uint32_t)std::max<uint64_t>(
                    1, std::min<uint64_t>(tasks, (uint64_t)std::max(per_sm, 1) * sm_count(m->device)));
                kern<<<grid, (fm::kWcPcPairWarps + 1) * 32, psm, stream()>>>(W, T, n_chunks);
            };
            if (su >= 2) launch(fm::fm_k_wc_pairs_pc<2>);
            else launch(fm::fm_k_wc_pairs_pc<1>);
            CK(cudaGetLastError());
            g_launches++;
        }
        // the overall components are one latency-bound warp per segment: they run on a side stream underneath the
        // pair kernel (both only read the cached counts; the fold below joins them)
        const uint32_t ob = std::max<uint32_t>(1, std::min<uint32_t>((n_seg + 3) / 4, 16u * sm_count(m->device)));
        cudaStream_t side = t_side_streams.get(m->device);
        CK(cudaStreamWaitEvent(side, wc_ready, 0));  // inputs and output buffers were set up before the pair launch
        fm::fm_k_wc_overall<<<ob, 128, 0, side>>>(W, T);
        CK(cudaGetLastError());
        g_launches++;
        cudaEvent_t join = wc_events.next();
        CK(cudaEventRecord(join, side));
        CK(cudaStreamWaitEvent(stream(), join, 0));
    }
    DevBuf<double> d_oo(nw * 2), d_op(nw * std::max(n_pairs, 1u) * 2);
    DevBuf<uint64_t> d_os(nw), d_on(nw * std::max(n_pairs, 1u));
    {
        // one CTA per (window, block of 32 slots); as many warps as the longest window has chunks (up to 16)
        uint32_t max_seg = 1;
        for (size_t w = 0; w < nw; ++w) max_seg = std::max(max_seg, wseg[w + 1] - wseg[w]);
        const uint32_t fw = std::max(1u, std::min<uint32_t>(fm::kWcFoldMaxWarps, (max_seg + fm::kWcFoldChunk - 1) / fm::kWcFoldChunk));
        const uint32_t n_pb = (n_pairs + 1 + 31) / 32;
        const uint32_t fb = (uint32_t)std::min<uint64_t>((uint64_t)nw * n_pb, 64ull * sm_count(m->device));
        fm::fm_k_wc_fold<<<std::max(fb, 1u), fw * 32, 0, stream()>>>(d_po.p, d_pc.p, d_pp.p, d_pn.p, d_wseg.p,
                                                                   (uint32_t)nw, n_pairs, n_pb, d_oo.p, d_os.p, d_op.p,
                                                                   d_on.p);
        CK(cudaGetLastError());
        g_launches++;
    }
    tm.stop();
    d_oo.download(tot.overall.data(), nw * 2);
    d_os.download(tot.sites.data(), nw);
    if (n_pairs) {
        d_op.download(tot.pair.data(), nw * n_pairs * 2);
        d_on.download(tot.pair_n.data(), nw * n_pairs);
    }
    if (W.site_state) d_state.download(so.state, ns);
    if (W.site_a) d_sa.download(so.a, ns);
    if (W.site_b) d_sb.download(so.b, ns);
    if (W.site_sizes) d_sizes.download(so.sizes, ns * G);
    if (W.pair_a) {
        d_pa.download(so.pair_a, ns * n_pairs);
        d_pb.download(so.pair_b, ns * n_pairs);
    }
    CK(cudaStreamSynchronize(stream()));
    t_tim.stats_ms += tm.ms();
}

fm_fst_estimate insufficient_estimate(uint64_t sites) {
    fm_fst_estimate e;
    e.state = 3;
    e.value = std::numeric_limits<double>::quiet_NaN();
    e.sum_a = 0.0;
    e.sum_b = 0.0;
    e.sites = sites;
    return e;
}
}  // namespace

// test hook for the FP64 building blocks of the W&C kernels (fm_wc.cuh): y[i] = fm_recip_rn(b[i]),
// q[i] = fm_div_recip(a[i], b[i], RN(1 / b[i])); host arrays
fm_status fm_wc_arith_probe(const double *a, const double *b, double *y, double *q, double *q_int, size_t n) {
    return guarded([&] {
        if (n && (!a || !b || !y || !q)) fail(FM_ERR_INVALID_ARG, "NULL argument");
        require_device();
        CK(cudaSetDevice(t_device));
        if (!n) return;
        DevBuf<double> da(n), db(n), dy(n), dq(n), dq3(n);
        da.upload(a, n);
        db.upload(b, n);
        fm::fm_k_wc_arith_probe<<<1024, 256, 0, stream()>>>(da.p, db.p, dy.p, dq.p, q_int ? dq3.p : nullptr, n);
        CK(cudaGetLastError());
        dy.download(y, n);
        dq.download(q, n);
        if (q_int) dq3.download(q_int, n);
        CK(cudaStreamSynchronize(stream()));
    });
}

fm_status fm_fst_estimate_from_sums(double sum_a, double sum_b, uint64_t informative_sites,
                                    uint64_t sites_attempted, fm_fst_estimate *out) {
    if (!out) return FM_ERR_INVALID_ARG;
    // stats.rs:2231-2270 (overall) / 2290-2356 (pairs)
    *out = informative_sites == 0 ? insufficient_estimate(sites_attempted)
                                  : classify_estimate(sum_a, sum_b, informative_sites);
    return FM_OK;
}

fm_status fm_wc_fst(fm_partition *p, int64_t rs, int64_t re, fm_fst_estimate *overall, fm_fst_estimate *pairs,
                    uint8_t *pair_present, int64_t *site_pos, int32_t *site_state, double *site_a, double *site_b,
                    uint32_t *site_pop_sizes, double *pair_a, double *pair_b, size_t capacity, size_t *n_sites_out) {
    return guarded([&] {
        FM_NVTX("fm_wc_fst (K4)");
        if (!p || !overall) fail(FM_ERR_INVALID_ARG, "NULL argument");
        if (n_sites_out) *n_sites_out = 0;
        require_device();
        fm_matrix *m = p->m;
        set_dev(m);
        const uint32_t G = (uint32_t)p->G;
        const uint32_t n_pairs = G * (G > 0 ? G - 1 : 0) / 2;
        if (n_pairs && !pairs) fail(FM_ERR_INVALID_ARG, "pairs is NULL");
        uint32_t lo = 0, hi = 0;
        site_range(m, rs, re, lo, hi);
        const size_t ns = hi - lo;
        if (ns == 0) {  // stats.rs:2152-2159
            *overall = insufficient_estimate(0);
            for (uint32_t i = 0; i < n_pairs; ++i) {
                pairs[i] = insufficient_estimate(0);
                if (pair_present) pair_present[i] = 0;
            }
            return;
        }
        const bool want_sites = site_state || site_a || site_b || site_pop_sizes || pair_a || pair_b || site_pos;
        if (want_sites && ns > capacity) fail(FM_ERR_INVALID_ARG, "per-site output capacity too small");
        WcSiteOut so;
        so.state = site_state;
        so.a = site_a;
        so.b = site_b;
        so.sizes = site_pop_sizes;
        so.pair_a = pair_a;
        so.pair_b = pair_b;
        WcWindowTotals t;
        run_wc(p, {lo}, {hi}, so, lo, ns, t);
        if (site_pos)
            for (size_t i = 0; i < ns; ++i) site_pos[i] = m->pos[lo + i] + 1;  // stats.rs:747
        // region aggregation (stats.rs:2145-2374)
        const uint64_t n_inf = t.sites[0];
        *overall = n_inf == 0 ? insufficient_estimate(ns) : classify_estimate(t.overall[0], t.overall[1], n_inf);
        for (uint32_t k = 0; k < n_pairs; ++k) {
            const uint64_t pn = t.pair_n[k];
            if (pair_present) pair_present[k] = n_inf > 0;
            if (n_inf == 0)
                pairs[k] = insufficient_estimate(0);
            else if (pn > 0)
                pairs[k] = classify_estimate(t.pair[2 * k], t.pair[2 * k + 1], pn);
            else
                pairs[k] = insufficient_estimate(n_inf);  // stats.rs:2342-2356
        }
        if (n_sites_out) *n_sites_out = ns;
    });
}

fm_status fm_wc_window_sums(fm_partition *p, const int64_t *windows, size_t n_windows, uint64_t *n_variants,
                            double *overall_a, double *overall_b, uint64_t *overall_sites, double *pair_a,
                            double *pair_b, uint64_t *pair_sites) {
    return guarded([&] {
        FM_NVTX("fm_wc_window_sums (K4)");
        if (!p || (n_windows && !windows)) fail(FM_ERR_INVALID_ARG, "NULL argument");
        require_device();
        if (!n_windows) return;
        fm_matrix *m = p->m;
        const uint32_t G = (uint32_t)p->G;
        const uint32_t n_pairs = G * (G > 0 ? G - 1 : 0) / 2;
        std::vector<uint32_t> lo, hi;
        window_ranges(m, windows, n_windows, lo, hi);
        WcWindowTotals t;
        run_wc(p, lo, hi, WcSiteOut{}, 0, 0, t);
        for (size_t w = 0; w < n_windows; ++w) {
            if (n_variants) n_variants[w] = hi[w] - lo[w];
            if (overall_a) overall_a[w] = t.overall[2 * w];
            if (overall_b) overall_b[w] = t.overall[2 * w + 1];
            if (overall_sites) overall_sites[w] = t.sites[w];
            for (uint32_t k = 0; k < n_pairs; ++k) {
                const size_t o = w * n_pairs + k;
                if (pair_a) pair_a[o] = t.pair[2 * o];
                if (pair_b) pair_b[o] = t.pair[2 * o + 1];
                if (pair_sites) pair_sites[o] = t.pair_n[o];
            }
        }
    });
}

// ------------------------------------------------------------------------------------ L_adj
fm_status fm_adjusted_sequence_length(int64_t region_start, int64_t region_end, const int64_t *allow,
                                      size_t n_allow, const int64_t *mask, size_t n_mask, int64_t *out) {
    return guarded([&] {
        if (!out) fail(FM_ERR_INVALID_ARG, "out is NULL");
        // stats.rs:3644-3736.  ZeroBasedHalfOpen::from_1based_inclusive (process.rs:193-206)
        auto hb = [](int64_t s, int64_t e, uint64_t &hs, uint64_t &he) {
            if (s < 1) s = 1;
            if (e < s) e = s;
            hs = (uint64_t)(s - 1);
            he = (uint64_t)e;
        };
        uint64_t rs, re;
        hb(region_start, region_end, rs, re);
        std::vector<std::pair<int64_t, int64_t>> allowed;
        if (allow) {
            for (size_t i = 0; i < n_allow; ++i) {
                const uint64_t as = (uint64_t)allow[2 * i], ae = (uint64_t)allow[2 * i + 1];
                const uint64_t s = std::max(rs, as), e = std::min(re, ae);
                if (s < e) allowed.emplace_back((int64_t)s + 1, (int64_t)e);
            }
        } else {
            allowed.emplace_back(region_start, region_end);
        }
        int64_t total = 0;
        std::vector<std::pair<int64_t, int64_t>> parts, next;
        for (auto &a : allowed) {  // subtract_regions (stats.rs:3739-3775): masks applied in order
            parts.assign(1, a);
            if (mask) {
                for (size_t mi = 0; mi < n_mask && !parts.empty(); ++mi) {
                    const int64_t m_start = (int64_t)((uint64_t)mask[2 * mi]) + 1;
                    const int64_t m_end = (int64_t)((uint64_t)mask[2 * mi + 1]);
                    next.clear();
                    for (auto &p : parts) {
                        const int64_t s = p.first, e = p.second;
                        if (m_end < s || m_start > e) {
                            next.push_back(p);
                            continue;
                        }
                        if (m_start > s && m_start - 1 >= s) next.emplace_back(s, m_start - 1);
                        if (m_end < e && m_end + 1 <= e) next.emplace_back(m_end + 1, e);
                    }
                    parts.swap(next);
                }
            }
            for (auto &p : parts) {
                uint64_t hs, he;
                hb(p.first, p.second, hs, he);
                total += he > hs ? (int64_t)(he - hs) : 0;
            }
        }
        *out = total;
    });
}

// ------------------------------------------------------------------------------------ windows (K5)
static void window_ranges(const fm_matrix *m, const int64_t *windows, size_t n, std::vector<uint32_t> &lo,
                          std::vector<uint32_t> &hi) {
    lo.resize(n);
    hi.resize(n);
    for (size_t i = 0; i < n; ++i) site_range(m, windows[2 * i], windows[2 * i + 1], lo[i], hi[i]);
}

fm_status fm_group_window_sums(fm_group *g, const int64_t *windows, size_t n_windows, uint64_t *n_variants,
                               uint64_t *seg, double *pi_sum, uint64_t *unc) {
    return guarded([&] {
        if (!g || (n_windows && !windows)) fail(FM_ERR_INVALID_ARG, "NULL argument");
        require_device();
        if (!n_windows) return;
        ensure_counts(g);
        set_dev(g->m);
        std::vector<uint32_t> lo, hi;
        window_ranges(g->m, windows, n_windows, lo, hi);
        DevBuf<uint32_t> dlo(n_windows), dhi(n_windows);
        dlo.upload(lo.data(), n_windows);
        dhi.upload(hi.data(), n_windows);
        DevBuf<uint64_t> dseg(n_windows), dunc(n_windows);
        DevBuf<double> dpi(n_windows);
        const uint32_t blocks = (uint32_t)std::min<size_t>((n_windows + 7) / 8, 8u * sm_count(g->m->device));
        if (g->n_bits > 1)  // multi-allelic: general dense forms over the cached per-allele counts
            fm::fm_k_window_div_multi<<<blocks, 256, 0, stream()>>>(g->d_acount, g->d_cnt, 1u << g->n_bits, FM_MULTI_DENSE,
                                                                     dlo.p, dhi.p, (uint32_t)n_windows, dseg.p, dpi.p,
                                                                     dunc.p);
        else
            fm::fm_k_window_div<<<blocks, 256, 0, stream()>>>(g->d_alt, g->d_cnt, dlo.p, dhi.p, (uint32_t)n_windows,
                                                               FM_PIFORM_COUNTS, dseg.p, dpi.p, dunc.p);
        CK(cudaGetLastError());
        g_launches++;
        if (seg) dseg.download(seg, n_windows);
        if (unc) dunc.download(unc, n_windows);
        if (pi_sum) dpi.download(pi_sum, n_windows);
        CK(cudaStreamSynchronize(stream()));
        if (n_variants)
            for (size_t i = 0; i < n_windows; ++i) n_variants[i] = hi[i] - lo[i];
    });
}

fm_status fm_hudson_window_sums(fm_group *g1, fm_group *g2, const int64_t *windows, size_t n_windows,
                                double *num_sum, double *den_sum, double *dxy_sum, uint64_t *dxy_unc,
                                double *pi1_sum, double *pi2_sum) {
    return guarded([&] {
        check_pair(g1, g2);
        if (n_windows && !windows) fail(FM_ERR_INVALID_ARG, "NULL argument");
        require_device();
        if (!n_windows) return;
        ensure_counts_pair(g1, g2);
        set_dev(g1->m);
        std::vector<uint32_t> lo, hi;
        window_ranges(g1->m, windows, n_windows, lo, hi);
        DevBuf<uint32_t> dlo(n_windows), dhi(n_windows);
        dlo.upload(lo.data(), n_windows);
        dhi.upload(hi.data(), n_windows);
        DevBuf<double> dd(n_windows * 5);
        DevBuf<uint64_t> ds(n_windows);
        const uint32_t blocks = (uint32_t)std::min<size_t>((n_windows + 7) / 8, 8u * sm_count(g1->m->device));
        if (g1->n_bits > 1)
            fm::fm_k_window_hudson_multi<<<blocks, 256, 0, stream()>>>(g1->d_acount, g1->d_cnt, g2->d_acount, g2->d_cnt,
                                                                        1u << g1->n_bits, FM_MULTI_DENSE, dlo.p, dhi.p,
                                                                        (uint32_t)n_windows, dd.p, ds.p);
        else
            fm::fm_k_window_hudson<<<blocks, 256, 0, stream()>>>(g1->d_alt, g1->d_cnt, g2->d_alt, g2->d_cnt, dlo.p,
                                                                  dhi.p, (uint32_t)n_windows, dd.p, ds.p);
        CK(cudaGetLastError());
        g_launches++;
        std::vector<double> h(n_windows * 5);
        dd.download(h.data(), n_windows * 5);
        if (dxy_unc) ds.download(dxy_unc, n_windows);
        CK(cudaStreamSynchronize(stream()));
        for (size_t i = 0; i < n_windows; ++i) {
            if (num_sum) num_sum[i] = h[i * 5 + 0];
            if (den_sum) den_sum[i] = h[i * 5 + 1];
            if (dxy_sum) dxy_sum[i] = h[i * 5 + 2];
            if (pi1_sum) pi1_sum[i] = h[i * 5 + 3];
            if (pi2_sum) pi2_sum[i] = h[i * 5 + 4];
        }
    });
}

// ------------------------------------------------------------------------------------ merged totals
fm_status fm_pi_from_sums(double pi_sum, uint64_t unc, int64_t L, size_t cap, double *out) {
    if (!out) return FM_ERR_INVALID_ARG;
    const double NaN = std::numeric_limits<double>::quiet_NaN();
    if (cap <= 1) *out = NaN;  // stats.rs:1485-1492
    else if (L < 0) *out = 0.0;
    else if (L == 0) *out = std::numeric_limits<double>::infinity();
    else {
        const int64_t eff = sat_sub(L, (int64_t)unc);  // :1512-1527
        *out = eff == 0 ? NaN : pi_sum / (double)eff;
    }
    return FM_OK;
}

fm_status fm_hudson_outcome_from_sums(const fm_hudson_sums *t, int64_t L, size_t cap1, size_t cap2,
                                      fm_hudson_outcome *out) {
    return guarded([&] {
        if (!t || !out) fail(FM_ERR_INVALID_ARG, "NULL argument");
        std::memset(out, 0, sizeof(*out));
        if (L <= 0)
            fail(FM_ERR_INVALID_REGION, "Sequence length must be positive for Hudson FST calculation.");
        if (t->den > FM_FST_EPSILON) {  // stats.rs:3505-3509
            out->fst = t->num / t->den;
            out->some |= 1u;
        }
        double p1, p2;
        fm_pi_from_sums(t->pi1, t->unc1, L, cap1, &p1);
        fm_pi_from_sums(t->pi2, t->unc2, L, cap2, &p2);
        if (std::isfinite(p1)) { out->pi_pop1 = p1; out->some |= 4u; }
        if (std::isfinite(p2)) { out->pi_pop2 = p2; out->some |= 8u; }
        if (cap1 != 0 && cap2 != 0) {  // dxy_from_summaries (stats.rs:1637-1662)
            const int64_t eff = sat_sub(L, (int64_t)t->dxy_uncallable);
            if (eff > 0) {
                out->d_xy = t->dxy / (double)eff;
                out->some |= 2u;
            }
        }
        if ((out->some & 12u) == 12u) {
            out->pi_xy_avg = 0.5 * (out->pi_pop1 + out->pi_pop2);
            out->some |= 16u;
        }
    });
}

// ------------------------------------------------------------------------------------ peer mailbox exchange
struct fm_comm {
    int rank = 0, world = 1, device = 0;
    fm::CommMailbox *mine = nullptr;
    fm::CommMailbox *peers[fm::kCommMaxRanks] = {};
    bool ipc_opened[fm::kCommMaxRanks] = {};
    bool connected = false;
    unsigned long long step = 0;
    uint32_t *d_status = nullptr;  // = d_merged + kCommMaxValues: merged words and status travel in one copy
    unsigned long long *d_local = nullptr, *d_gathered = nullptr, *d_merged = nullptr;
    unsigned long long *h_result = nullptr;  // pinned: [kCommMaxValues + 1], small results land here asynchronously
    // An exchange waits for the slowest rank like any collective; the timeout only exists so that a rank that
    // died cannot hang the GPU for ever (0 = no timeout).  Ranks may legitimately be far apart (unequal shard
    // work, host I/O between calls), hence minutes, not seconds.
    unsigned long long timeout_ns = 120000000000ull;
};

namespace {
// Enqueue one exchange on the calling thread's stream (asynchronous).
void comm_launch(fm_comm *c, const unsigned long long *d_local, uint32_t n_words, uint32_t n_double,
                 const fm::CommFold *folds, uint32_t n_fold, cudaStream_t st = nullptr) {
    if (!st) st = stream();
    if (!c->connected) fail(FM_ERR_INVALID_ARG, "fm_comm is not connected");
    if (n_words > fm::kCommMaxValues) fail(FM_ERR_INVALID_ARG, "too many values for one exchange");
    fm::CommParams P{};
    for (int r = 0; r < c->world; ++r) P.peers[r] = c->peers[r];
    P.rank = (uint32_t)c->rank;
    P.world = (uint32_t)c->world;
    P.step = ++c->step;
    P.n_words = n_words;
    P.n_double = n_double;
    P.local = d_local;
    P.n_fold = n_fold;
    for (uint32_t f = 0; f < n_fold; ++f) {
        if (folds[f].nd + folds[f].nu > 32) fail(FM_ERR_INVALID_ARG, "fold has more than 32 columns");
        if (folds[f].nd + folds[f].nu == 0) fail(FM_ERR_INVALID_ARG, "fold has no columns");
        P.fold[f] = folds[f];
    }
    P.gathered = c->d_gathered;
    P.merged = c->d_merged;
    P.status = c->d_status;
    P.timeout_ns = c->timeout_ns;
    fm::fm_k_comm_exchange<<<1, 128, 0, st>>>(P);
    CK(cudaGetLastError());
    g_launches++;
}
void comm_report_timeout(fm_comm *c);
// merged words [0, n_words) + the status word in ONE asynchronous copy into pinned memory, then one synchronise
const unsigned long long *comm_fetch_merged(fm_comm *c, uint32_t n_words) {
    // the kernel leaves a copy of the status word right behind the merged words: ONE asynchronous copy into pinned
    // memory and one synchronise (a pageable destination would make the copy a blocking driver round trip)
    if (n_words >= fm::kCommMaxValues) fail(FM_ERR_INVALID_ARG, "too many values for one fetch");
    CK(cudaMemcpyAsync(c->h_result, c->d_merged, ((size_t)n_words + 1) * 8, cudaMemcpyDeviceToHost, stream()));
    CK(cudaStreamSynchronize(stream()));
    if ((uint32_t)c->h_result[n_words] != 0) comm_report_timeout(c);
    return c->h_result;
}
void comm_report_timeout(fm_comm *c) {
    CK(cudaMemsetAsync(c->d_status, 0, 4, stream()));
    CK(cudaStreamSynchronize(stream()));
    fail(FM_ERR_CUDA, "peer exchange timed out waiting for another rank (fm_comm_set_timeout_ms raises the limit)");
}
void comm_check_status(fm_comm *c) {
    uint32_t st = 0;
    CK(cudaMemcpyAsync(&st, c->d_status, 4, cudaMemcpyDeviceToHost, stream()));
    CK(cudaStreamSynchronize(stream()));
    if (st != 0) {
        // report once: the word is cleared so that later exchanges on this communicator start clean.  The rank
        // that timed out had already published its own contribution, so its peers completed the step; the
        // step counters stay aligned and the next exchange is valid if the late rank has caught up.
        CK(cudaMemsetAsync(c->d_status, 0, 4, stream()));
        CK(cudaStreamSynchronize(stream()));
        fail(FM_ERR_CUDA, "peer exchange timed out waiting for another rank (fm_comm_set_timeout_ms raises the limit)");
    }
}
}  // namespace

fm_status fm_comm_create(int rank, int world, fm_comm **out) {
    return guarded([&] {
        if (!out) fail(FM_ERR_INVALID_ARG, "out is NULL");
        *out = nullptr;
        if (world < 1 || world > (int)fm::kCommMaxRanks || rank < 0 || rank >= world)
            fail(FM_ERR_INVALID_ARG, "bad rank / world size");
        require_device();
        CK(cudaSetDevice(t_device));
        fm_comm *c = new fm_comm();
        c->rank = rank;
        c->world = world;
        c->device = t_device;
        try {
            // plain cudaMalloc (not the cache): the allocation is exported through cudaIpc
            CK(cudaMalloc((void **)&c->mine, sizeof(fm::CommMailbox)));
            CK(cudaMemset(c->mine, 0, sizeof(fm::CommMailbox)));
            CK(cudaMalloc((void **)&c->d_local, fm::kCommMaxValues * 8));
            CK(cudaMalloc((void **)&c->d_merged, (fm::kCommMaxValues + 32) * 8));
            CK(cudaMemset(c->d_merged, 0, (fm::kCommMaxValues + 32) * 8));
            c->d_status = reinterpret_cast<uint32_t *>(c->d_merged + fm::kCommMaxValues);
            CK(cudaHostAlloc((void **)&c->h_result, (fm::kCommMaxValues + 32) * 8, cudaHostAllocDefault));
            CK(cudaMalloc((void **)&c->d_gathered, (size_t)world * fm::kCommMaxValues * 8));
            CK(cudaDeviceSynchronize());
            c->peers[rank] = c->mine;
            if (world == 1) c->connected = true;
        } catch (...) {
            fm_comm_destroy(c);
            throw;
        }
        *out = c;
    });
}

fm_status fm_comm_export(fm_comm *c, uint8_t *handle_out) {
    return guarded([&] {
        if (!c || !handle_out) fail(FM_ERR_INVALID_ARG, "NULL argument");
        static_assert(sizeof(cudaIpcMemHandle_t) == FM_COMM_HANDLE_BYTES, "handle size");
        CK(cudaSetDevice(c->device));
        cudaIpcMemHandle_t h;
        CK(cudaIpcGetMemHandle(&h, c->mine));
        std::memcpy(handle_out, &h, sizeof(h));
    });
}

fm_status fm_comm_connect(fm_comm *c, const uint8_t *handles) {
    return guarded([&] {
        if (!c || !handles) fail(FM_ERR_INVALID_ARG, "NULL argument");
        CK(cudaSetDevice(c->device));
        for (int r = 0; r < c->world; ++r) {
            if (r == c->rank) continue;
            cudaIpcMemHandle_t h;
            std::memcpy(&h, handles + (size_t)r * FM_COMM_HANDLE_BYTES, sizeof(h));
            void *p = nullptr;
            CK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
            c->peers[r] = static_cast<fm::CommMailbox *>(p);
            c->ipc_opened[r] = true;
        }
        c->connected = true;
    });
}

fm_status fm_comm_connect_local(fm_comm *c, fm_comm *const *all) {
    return guarded([&] {
        if (!c || !all) fail(FM_ERR_INVALID_ARG, "NULL argument");
        CK(cudaSetDevice(c->device));
        for (int r = 0; r < c->world; ++r) {
            if (!all[r] || all[r]->world != c->world || all[r]->rank != r)
                fail(FM_ERR_INVALID_ARG, "peer list does not match the communicator");
            if (all[r]->device != c->device) {
                cudaError_t e = cudaDeviceEnablePeerAccess(all[r]->device, 0);
                if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
                else CK(e);
            }
            c->peers[r] = all[r]->mine;
        }
        c->connected = true;
    });
}

fm_status fm_comm_allgather(fm_comm *c, const void *local, size_t n_words, size_t n_double, void *gathered_out,
                            void *merged_out) {
    return guarded([&] {
        FM_NVTX("fm_comm_allgather (NVLink mailbox exchange)");
        if (!c || (n_words && !local)) fail(FM_ERR_INVALID_ARG, "NULL argument");
        if (n_words > fm::kCommMaxValues) fail(FM_ERR_INVALID_ARG, "too many values for one exchange");
        CK(cudaSetDevice(c->device));
        if (n_words) CK(cudaMemcpyAsync(c->d_local, local, n_words * 8, cudaMemcpyHostToDevice, stream()));
        comm_launch(c, c->d_local, (uint32_t)n_words, (uint32_t)std::min(n_double, n_words), nullptr, 0);
        if (gathered_out && n_words)
            CK(cudaMemcpyAsync(gathered_out, c->d_gathered, (size_t)c->world * n_words * 8, cudaMemcpyDeviceToHost,
                               stream()));
        if (merged_out && n_words)
            CK(cudaMemcpyAsync(merged_out, c->d_merged, n_words * 8, cudaMemcpyDeviceToHost, stream()));
        comm_check_status(c);
    });
}

fm_status fm_comm_set_timeout_ms(fm_comm *c, uint64_t ms) {
    if (!c) return FM_ERR_INVALID_ARG;
    c->timeout_ns = ms * 1000000ull;
    return FM_OK;
}

fm_status fm_comm_destroy(fm_comm *c) {
    if (!c) return FM_OK;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();  // every exchange this rank launched (on any stream) has finished writing to its peers
    bool leak_mailbox = false;
    bool cross_process = false;
    for (int r = 0; r < c->world; ++r) cross_process = cross_process || c->ipc_opened[r];
    if (c->connected && c->world > 1 && cross_process) {
        // closing handshake between processes: nobody frees a mailbox a peer may still write into (ranks wired
        // inside one process with fm_comm_connect_local are torn down by their common owner, in any order)
        fm::CommParams P{};
        for (int r = 0; r < c->world; ++r) P.peers[r] = c->peers[r];
        P.rank = (uint32_t)c->rank;
        P.world = (uint32_t)c->world;
        P.status = c->d_status;
        // a peer that is more than 10 s late (or dead) is not waited for: the mailbox is then kept, not freed
        P.timeout_ns = c->timeout_ns ? std::min<unsigned long long>(c->timeout_ns, 10000000000ull) : 10000000000ull;
        cudaMemsetAsync(c->d_status, 0, 4, stream());
        fm::fm_k_comm_goodbye<<<1, 32, 0, stream()>>>(nullptr, P);
        uint32_t st = 1;
        if (cudaMemcpyAsync(&st, c->d_status, 4, cudaMemcpyDeviceToHost, stream()) != cudaSuccess ||
            cudaStreamSynchronize(stream()) != cudaSuccess) {
            cudaGetLastError();
            st = 1;
        }
        leak_mailbox = st != 0;  // a peer never closed: keep the memory rather than free it under a writer
    }
    for (int r = 0; r < c->world; ++r)
        if (c->ipc_opened[r]) cudaIpcCloseMemHandle(c->peers[r]);
    if (!leak_mailbox) cudaFree(c->mine);
    if (c->h_result) cudaFreeHost(c->h_result);
    cudaFree(c->d_local);
    cudaFree(c->d_merged);
    cudaFree(c->d_gathered);
    delete c;
    return FM_OK;
}

// ------------------------------------------------------------------------------------ sharded Hudson call
// One Hudson call over a cohort that is sharded by site range across the ranks of `comm` (SURVEY 8e, config 3):
// every rank sweeps its own shard once (pair units of fm_k_plane_pass_seq, nothing cached, nothing written but
// the per-batch partials), folds the partials per super-batch, and the fold into region totals is fused with
// the NVLink mailbox exchange; the rank-ordered merged totals come back in ONE small copy and are finished on
// the host exactly like the single-GPU summaries path (stats.rs:3476-3566).  Three launches, one host sync.
fm_status fm_hudson_pair_sharded(fm_group *g1, fm_group *g2, int64_t sequence_length, size_t raw_n1, size_t raw_n2,
                                 fm_comm *comm, fm_hudson_outcome *out, fm_hudson_sums *merged_out) {
    return guarded([&] {
        FM_NVTX("fm_hudson_pair_sharded (pass + fold + NVLink exchange)");
        if (!out) fail(FM_ERR_INVALID_ARG, "out is NULL");
        std::memset(out, 0, sizeof(*out));
        if (sequence_length <= 0)
            fail(FM_ERR_INVALID_REGION, "Sequence length must be positive for Hudson FST calculation.");
        check_pair(g1, g2);
        require_device();
        fm_matrix *m = g1->m;
        set_dev(m);
        if (comm && comm->device != m->device) fail(FM_ERR_INVALID_ARG, "communicator and groups live on different devices");
        if (g1->n_bits != 1) fail(FM_ERR_UNSUPPORTED, "the summaries path does not exist for multi-allelic matrices (lib.rs:779)");
        const uint32_t V = (uint32_t)m->V;
        const uint32_t nb = (V + 31) / 32;
        const uint32_t n_super = (nb + fm::kSuperBatches - 1) / fm::kSuperBatches;
        // one allocation for all four scratch arrays: every trip through the caching allocator costs a few driver
        // calls (event wait / create / record), and this call is only ~250 us long on an eighth of config 3
        const size_t nb1 = std::max(nb, 1u), ns1 = std::max(n_super, 1u);
        const size_t off_pd = 0, off_sd = off_pd + nb1 * 5 * 8, off_su = off_sd + ns1 * 5 * 8,
                     off_pu = off_su + ns1 * 3 * 8, total_scratch = off_pu + nb1 * 3 * 4;
        DevBuf<uint8_t> scratch(total_scratch);
        struct {
            double *p;
        } pd{reinterpret_cast<double *>(scratch.p + off_pd)}, sd{reinterpret_cast<double *>(scratch.p + off_sd)};
        struct {
            uint64_t *p;
        } su{reinterpret_cast<uint64_t *>(scratch.p + off_su)};
        struct {
            uint32_t *p;
        } pu{reinterpret_cast<uint32_t *>(scratch.p + off_pu)};
        fm::HudsonEpilogue he{};
        he.variant = -1;  // aggregate_hudson_components_from_summaries (stats.rs:1554-1623)
        he.part_d = pd.p;
        he.part_u = pu.p;
        Timer tm;
        static const uint32_t trace = env_u32("FM_SHARDED_TRACE", 0);  // stage timings on stderr (tuning)
        EventPairs tev;
        cudaEvent_t te[4] = {nullptr, nullptr, nullptr, nullptr};
        const auto th0 = std::chrono::steady_clock::now();
        if (trace) {
            for (auto &e : te) e = tev.next();
            CK(cudaEventRecord(te[0], stream()));
        }
        tm.start();
        if (V) {
            bool done = false;
            if (g1 != g2 && !g1->count_only && !g2->count_only && !(g1->have_counts && g2->have_counts)) {
                // no diversity epilogue (div.part_pi == nullptr): the Hudson partials are the only output
                std::vector<fm::RowSeg> segs{div_seg(g1, fm::DivEpilogue{}, 0, V), div_seg(g2, fm::DivEpilogue{}, 0, V)};
                std::vector<fm::HudsonEpilogue> hv{he};
                RowPlan plan;
                done = plan_rows(segs, &hv, plan);
                if (done) launch_rows(plan, m->device);
            }
            if (!done) {  // cached counts, count-only groups or rows wider than the row pass: from the counts
                ensure_counts_pair(g1, g2);
                const uint32_t blocks = std::min<uint32_t>((nb + 7) / 8, 8u * sm_count(m->device));
                fm::fm_k_hudson_from_counts<<<blocks, 256, 0, stream()>>>(g1->d_alt, g1->d_cnt, g2->d_alt, g2->d_cnt, he, 0,
                                                                           V, 0, nb);
                CK(cudaGetLastError());
                g_launches++;
            }
            if (trace) CK(cudaEventRecord(te[1], stream()));
            launch_reduce(pd.p, 5, pu.p, 3, batch_range(0, V), sd.p, su.p, stream());
            if (trace) CK(cudaEventRecord(te[2], stream()));
        }
        unsigned long long w[8] = {};
        if (comm) {
            fm::CommFold fold{sd.p, reinterpret_cast<const unsigned long long *>(su.p), n_super, 5u, 3u};
            comm_launch(comm, nullptr, 8, 0, &fold, 1, stream());
            if (trace) CK(cudaEventRecord(te[3], stream()));
            std::memcpy(w, comm_fetch_merged(comm, 8), sizeof(w));
            if (trace && V) {
                float a = 0, b = 0, c = 0;
                cudaEventElapsedTime(&a, te[0], te[1]);
                cudaEventElapsedTime(&b, te[1], te[2]);
                cudaEventElapsedTime(&c, te[2], te[3]);
                const double host_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - th0).count();
                fprintf(stderr, "[sharded rank %d] pass %.1f us, fold %.1f us, exchange %.1f us, host total %.1f us\n", comm->rank,
                        a * 1e3, b * 1e3, c * 1e3, host_ms * 1e3);
            }
        } else {
            std::vector<double> hd((size_t)n_super * 5);
            std::vector<uint64_t> hu((size_t)n_super * 3);
            if (!hd.empty()) CK(cudaMemcpyAsync(hd.data(), sd.p, hd.size() * 8, cudaMemcpyDeviceToHost, stream()));
            if (!hu.empty()) CK(cudaMemcpyAsync(hu.data(), su.p, hu.size() * 8, cudaMemcpyDeviceToHost, stream()));
            CK(cudaStreamSynchronize(stream()));
            double d[5];
            uint64_t u[3] = {0, 0, 0};
            for (int i = 0; i < 5; ++i) d[i] = fm::fm_comm_fold_host(hd.data(), n_super, 5, i);  // the exchange kernel's fold
            for (uint32_t sb = 0; sb < n_super; ++sb)
                for (int i = 0; i < 3; ++i) u[i] += hu[(size_t)sb * 3 + i];
            std::memcpy(w, d, sizeof(d));
            for (int i = 0; i < 3; ++i) w[5 + i] = u[i];
        }
        tm.stop();
        t_tim.stats_ms += tm.ms();
        fm_hudson_sums sums;
        std::memcpy(&sums.num, &w[0], 8);
        std::memcpy(&sums.den, &w[1], 8);
        std::memcpy(&sums.dxy, &w[2], 8);
        std::memcpy(&sums.pi1, &w[3], 8);
        std::memcpy(&sums.pi2, &w[4], 8);
        sums.dxy_uncallable = w[5];
        sums.unc1 = w[6];
        sums.unc2 = w[7];
        if (merged_out) *merged_out = sums;
        // calculate_hudson_fst_for_pair_core, summaries path (stats.rs:3476-3488, 3505-3566)
        fm_hudson_outcome o;
        fm_status st = fm_hudson_outcome_from_sums(&sums, sequence_length, g1->n, g2->n, &o);
        if (st != FM_OK) fail(st, t_err);
        if (raw_n1 == 0 || raw_n2 == 0) o.some &= ~2u;  // dxy_from_summaries needs both haplotype lists non-empty
        *out = o;
    });
}

// ------------------------------------------------------------------------------------ FALSTA track bodies
fm_status fm_falsta_format_value(double value, int mode, char *buf, size_t capacity, size_t *len_out) {
    if (!buf || !len_out || capacity < 56) return FM_ERR_INVALID_ARG;
    if (mode != FM_FALSTA_DIVERSITY && mode != FM_FALSTA_FST && mode != FM_FALSTA_TSV) return FM_ERR_INVALID_ARG;
    *len_out = fm::fm_falsta_token(value, mode, buf);  // the same __host__ __device__ routine the kernels run
    return FM_OK;
}

fm_status fm_falsta_tracks(const int64_t *pos1, const double *values, size_t n, size_t n_tracks, int64_t region_start,
                           int64_t region_end, int mode, char *out, size_t capacity, size_t *line_len,
                           size_t *len_out) {
    return guarded([&] {
        FM_NVTX("fm_falsta_tracks");
        if (!len_out) fail(FM_ERR_INVALID_ARG, "len_out is NULL");
        *len_out = 0;
        if (n_tracks == 0) return;
        if (n && (!pos1 || !values)) fail(FM_ERR_INVALID_ARG, "record arrays are NULL");
        if (mode != FM_FALSTA_DIVERSITY && mode != FM_FALSTA_FST) fail(FM_ERR_INVALID_ARG, "unknown track mode");
        if (n >= (1ull << 31)) fail(FM_ERR_UNSUPPORTED, "more than 2^31 records per track");
        if (n_tracks > 64) fail(FM_ERR_UNSUPPORTED, "more than 64 tracks per call");
        require_device();
        CK(cudaSetDevice(t_device));
        // ZeroBasedHalfOpen::from_1based_inclusive (process.rs:193-206)
        int64_t s1 = region_start < 1 ? 1 : region_start;
        int64_t e1 = region_end < s1 ? s1 : region_end;
        const uint64_t rs = (uint64_t)(s1 - 1), re = (uint64_t)e1;
        const uint64_t L = re - rs;  // >= 1 by construction
        const uint64_t T = L * n_tracks;
        DevBuf<int> d_idx(L);
        DevBuf<uint32_t> d_len(T);
        DevBuf<uint64_t> d_off(T);
        DevBuf<int64_t> d_pos(std::max<size_t>(n, 1));
        DevBuf<double> d_val(std::max<size_t>(n * n_tracks, 1));
        CK(cudaMemsetAsync(d_idx.p, 0xFF, L * sizeof(int), stream()));
        h2d(d_pos.p, pos1, n * 8, stream());
        h2d(d_val.p, values, n * n_tracks * 8, stream());
        const int dev_sms = sm_count(t_device);
        if (n) {
            const uint32_t b = (uint32_t)std::min<uint64_t>((n + 255) / 256, 8ull * dev_sms);
            fm::fm_k_falsta_scatter<<<b, 256, 0, stream()>>>(d_pos.p, (uint32_t)n, rs, re, d_idx.p);
            CK(cudaGetLastError());
            g_launches++;
        }
        const uint32_t blocks = (uint32_t)std::min<uint64_t>((T + 255) / 256, 16ull * dev_sms);
        // FM_FALSTA_TEST_INFLATE=k (length queries only) adds k bytes to every token length so that a test can push
        // the body past 4 GiB without a multi-gigabyte input
        const uint32_t inflate = env_u32("FM_FALSTA_TEST_INFLATE", 0);
        if (inflate && out) fail(FM_ERR_INVALID_ARG, "FM_FALSTA_TEST_INFLATE is for length queries (out == NULL) only");
        fm::fm_k_falsta_lengths<<<blocks, 256, 0, stream()>>>(d_idx.p, d_val.p, n, L, (uint32_t)n_tracks, mode,
                                                               d_len.p, inflate);
        CK(cudaGetLastError());
        g_launches++;
        // The prefix sum must run in 64 bits: a body can exceed 4 GiB (a 250 Mb region with a dozen tracks).  cub
        // derives the accumulator from the INPUT type, so the u32 lengths are widened by the input iterator and the
        // scan is given a u64 initial value.
        size_t tmp_bytes = 0;
        thrust::transform_iterator<fm::U32ToU64, const uint32_t *> len64(d_len.p, fm::U32ToU64());
        CK(cub::DeviceScan::ExclusiveScan(nullptr, tmp_bytes, len64, d_off.p, cuda::std::plus<>(), (uint64_t)0, (int64_t)T,
                                          stream()));
        DevBuf<uint8_t> d_tmp(std::max<size_t>(tmp_bytes, 16));
        CK(cub::DeviceScan::ExclusiveScan(d_tmp.p, tmp_bytes, len64, d_off.p, cuda::std::plus<>(), (uint64_t)0, (int64_t)T,
                                          stream()));
        // line t starts at off[t*L]; the call ends at off[T-1] + len[T-1]
        std::vector<uint64_t> starts(n_tracks + 1);
        for (size_t t = 0; t < n_tracks; ++t)
            CK(cudaMemcpyAsync(&starts[t], d_off.p + t * L, 8, cudaMemcpyDeviceToHost, stream()));
        uint32_t last_len = 0;
        CK(cudaMemcpyAsync(&starts[n_tracks], d_off.p + (T - 1), 8, cudaMemcpyDeviceToHost, stream()));
        CK(cudaMemcpyAsync(&last_len, d_len.p + (T - 1), 4, cudaMemcpyDeviceToHost, stream()));
        CK(cudaStreamSynchronize(stream()));
        const uint64_t total = starts[n_tracks] + last_len;
        starts[n_tracks] = total + 1;  // as if a separator followed the last line too
        if (line_len)
            for (size_t t = 0; t < n_tracks; ++t) line_len[t] = (size_t)(starts[t + 1] - starts[t] - 1);
        *len_out = (size_t)total;
        if (!out) return;  // length query
        if (total > capacity) fail(FM_ERR_INVALID_ARG, "output capacity too small for the track lines");
        DevBuf<char> d_out(std::max<uint64_t>(total, 1));
        fm::fm_k_falsta_write<<<blocks, 256, 0, stream()>>>(d_idx.p, d_val.p, n, L, (uint32_t)n_tracks, mode, d_off.p,
                                                             d_out.p);
        CK(cudaGetLastError());
        g_launches++;
        CK(cudaMemcpyAsync(out, d_out.p, total, cudaMemcpyDeviceToHost, stream()));
        CK(cudaStreamSynchronize(stream()));
    });
}

fm_status fm_falsta_track(const int64_t *pos1, const double *values, size_t n, int64_t region_start,
                          int64_t region_end, int mode, char *out, size_t capacity, size_t *len_out) {
    return fm_falsta_tracks(pos1, values, n, 1, region_start, region_end, mode, out, capacity, nullptr, len_out);
}

// ------------------------------------------------------------------------------------ VCF parse/filter stage
struct fm_vcf_batch {
    int device = 0;
    size_t n_lines = 0, S = 0, P = 0, n_rows = 0;
    uint8_t *d_gt = nullptr;       // [n_rows][S][P], rows in line order of the variant-producing lines
    uint32_t *d_order = nullptr;   // [n_variants] row index per output variant
    std::vector<fm::VcfLine> var;  // per output variant (output order)
    std::vector<uint32_t> order;   // row index per output variant
    std::vector<int64_t> pos_missing, pos_filtered;
    std::vector<uint64_t> err_line;
    std::vector<int32_t> err_code;
    std::vector<int64_t> err_aux;
    fm_vcf_info info{};
};

namespace {

// (start, end) pairs -> merged, sorted, disjoint unsigned [s, e); `any` over half-open intervals only
// depends on their union.  as_usize: the mask path casts both ends to usize (process.rs:4566-4577).
std::vector<uint64_t> vcf_normalise_intervals(const int64_t *iv, size_t n, bool as_usize) {
    std::vector<std::pair<uint64_t, uint64_t>> v;
    v.reserve(n);
    for (size_t i = 0; i < n; ++i) {
        const int64_t s = iv[2 * i], e = iv[2 * i + 1];
        uint64_t us, ue;
        if (as_usize) {
            us = (uint64_t)s;
            ue = (uint64_t)e;
        } else {  // pos >= s && pos < e with pos >= 0
            if (e <= 0) continue;
            us = s < 0 ? 0 : (uint64_t)s;
            ue = (uint64_t)e;
        }
        if (us < ue) v.emplace_back(us, ue);
    }
    std::sort(v.begin(), v.end());
    std::vector<uint64_t> out;
    for (auto &p : v) {
        if (!out.empty() && p.first <= out[out.size() - 1]) {
            if (p.second > out[out.size() - 1]) out[out.size() - 1] = p.second;
        } else {
            out.push_back(p.first);
            out.push_back(p.second);
        }
    }
    return out;
}

__global__ void __launch_bounds__(256)
fm_k_vcf_rowflag(const fm::VcfLine *__restrict__ recs, uint32_t n, uint32_t *__restrict__ flag) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flag[i] = (recs[i].status == fm::VCF_CAND && !(recs[i].indel & 1)) ? 1u : 0u;
    else if (i == n) flag[i] = 0u;
}

// Per-thread pinned host scratch: device -> host reads of counters and per-line records land here with truly
// asynchronous copies (a pageable destination makes every small cudaMemcpyAsync a blocking driver round trip).
struct PinnedScratch {
    uint8_t *p = nullptr;
    size_t cap = 0;
    uint8_t *ensure(size_t bytes) {
        if (bytes > cap) {
            if (p) cudaFreeHost(p);
            p = nullptr;
            cap = 0;
            const size_t want = std::max<size_t>(bytes + bytes / 2, (size_t)1 << 20);
            CK(cudaHostAlloc((void **)&p, want, cudaHostAllocDefault));
            cap = want;
        }
        return p;
    }
    ~PinnedScratch() {
        if (p) cudaFreeHost(p);
    }
};
thread_local PinnedScratch t_pinned;

__global__ void fm_k_vcf_index_ends(uint32_t *line_start, uint32_t *tabs_before, uint32_t n_lines, uint32_t n_bytes,
                                    uint32_t tab_total) {
    // line 0 starts at byte 0; an unterminated last line ends at the end of the text (a terminated one wrote the
    // same values itself)
    line_start[0] = 0;
    tabs_before[0] = 0;
    line_start[n_lines] = n_bytes;
    tabs_before[n_lines] = tab_total;
}

struct VcfShared {  // validated parameters + their device copies, shared by every chunk of a call
    fm::VcfParams P{};
    size_t n_kept = 0, max_ploidy = 0;
    DevBuf<int64_t> d_regions;
    DevBuf<uint64_t> d_allow, d_mask;
    DevBuf<int32_t> d_c2s;
};

void vcf_prepare(VcfShared &sh, const char *chr, const int64_t *regions, size_t n_regions, const uint32_t *kept,
                 size_t n_kept, uint16_t min_gq, int allow_mode, const int64_t *allow, size_t n_allow, int mask_mode,
                 const int64_t *mask, size_t n_mask, size_t max_ploidy) {
    if (!chr) fail(FM_ERR_INVALID_ARG, "chr is NULL");
    if (n_regions && !regions) fail(FM_ERR_INVALID_ARG, "regions is NULL");
    if (n_kept && !kept) fail(FM_ERR_INVALID_ARG, "kept_col_indices is NULL");
    if (max_ploidy < 1 || max_ploidy > (size_t)fm::VCF_MAX_PLOIDY) fail(FM_ERR_INVALID_ARG, "max_ploidy must be 1..8");
    if ((unsigned)allow_mode > 2u || (unsigned)mask_mode > 2u) fail(FM_ERR_INVALID_ARG, "unknown allow/mask mode");
    if ((allow_mode == FM_VCF_INTERVALS && n_allow && !allow) || (mask_mode == FM_VCF_INTERVALS && n_mask && !mask))
        fail(FM_ERR_INVALID_ARG, "interval list is NULL");
    for (size_t i = 0; i < n_kept; ++i) {
        if (kept[i] < 9) fail(FM_ERR_INVALID_ARG, "kept column index below 9 (the first sample column)");
        if (i && kept[i] <= kept[i - 1]) fail(FM_ERR_INVALID_ARG, "kept_col_indices must be strictly increasing");
    }
    if (n_kept && kept[n_kept - 1] >= (1u << 30)) fail(FM_ERR_UNSUPPORTED, "column index too large");
    for (size_t i = 1; i < n_regions; ++i)
        if (regions[2 * i] < regions[2 * i - 2] || regions[2 * i + 1] < regions[2 * i - 1])
            fail(FM_ERR_INVALID_ARG, "regions must be sorted (process_vcf passes merged, sorted regions)");
    fm::VcfParams &P = sh.P;
    {  // normalize_chr_prefix(chr.trim())
        std::string c(chr);
        auto ws = [](char x) { return x == ' ' || (x >= 9 && x <= 13); };
        size_t a = 0, b = c.size();
        while (a < b && ws(c[a])) ++a;
        while (b > a && ws(c[b - 1])) --b;
        c = c.substr(a, b - a);
        if (c.rfind("chr", 0) == 0 || c.rfind("Chr", 0) == 0 || c.rfind("CHR", 0) == 0) c = c.substr(3);
        if (c.size() > 63) fail(FM_ERR_INVALID_ARG, "chromosome name longer than 63 bytes");
        memcpy(P.chr, c.data(), c.size());
        P.chr_len = (uint32_t)c.size();
    }
    std::vector<uint64_t> allow_n, mask_n;
    if (allow_mode == FM_VCF_INTERVALS) allow_n = vcf_normalise_intervals(allow, n_allow, false);
    if (mask_mode == FM_VCF_INTERVALS) mask_n = vcf_normalise_intervals(mask, n_mask, true);
    sh.d_regions.alloc(std::max<size_t>(2 * n_regions, 2));
    sh.d_allow.alloc(std::max<size_t>(allow_n.size(), 2));
    sh.d_mask.alloc(std::max<size_t>(mask_n.size(), 2));
    sh.d_regions.upload(regions, 2 * n_regions);
    sh.d_allow.upload(allow_n.data(), allow_n.size());
    sh.d_mask.upload(mask_n.data(), mask_n.size());
    const int32_t max_idx = n_kept ? (int32_t)kept[n_kept - 1] : -1;
    std::vector<int32_t> col2slot((size_t)(max_idx + 1), -1);
    for (size_t i = 0; i < n_kept; ++i) col2slot[kept[i]] = (int32_t)i;
    sh.d_c2s.alloc(std::max<size_t>(col2slot.size(), 1));
    sh.d_c2s.upload(col2slot.data(), col2slot.size());
    CK(cudaStreamSynchronize(stream()));  // the host vectors above go out of scope
    P.regions = sh.d_regions.p;
    P.n_regions = (uint32_t)n_regions;
    P.allow_mode = allow_mode;
    P.mask_mode = mask_mode;
    P.allow = sh.d_allow.p;
    P.mask = sh.d_mask.p;
    P.n_allow = (uint32_t)(allow_n.size() / 2);
    P.n_mask = (uint32_t)(mask_n.size() / 2);
    P.max_idx = max_idx;
    P.min_gq = min_gq;
    P.n_samples = (uint32_t)n_kept;
    P.max_ploidy = (uint32_t)max_ploidy;
    P.col2slot = sh.d_c2s.p;
    sh.n_kept = n_kept;
    sh.max_ploidy = max_ploidy;
}

struct VcfChunkOut {
    std::vector<fm::VcfLine> recs;  // per line of the chunk
    std::vector<uint32_t> rows;     // chunk-local row of every line
    uint8_t *d_gt = nullptr;        // [n_rows][S][P]
    size_t n_rows = 0;
    float index_ms = 0.f, parse_ms = 0.f;
};

// One chunk of whole lines resident at d_text (16-byte aligned, zero-padded): line index, fixed fields, rows, samples.
void vcf_chunk(const VcfShared &sh, const uint8_t *d_text, size_t n_bytes, char last_byte, VcfChunkOut &out) {
    if (n_bytes == 0) return;
    const int sms = sm_count(t_device);
    Timer t_index, t_parse;
    const uint64_t n16 = (n_bytes + 15) / 16;
    const uint32_t n_tiles = (uint32_t)((n16 + 255) / 256);
    // tile counts with one zero element appended, so that the exclusive scans end in the totals
    const size_t nt1 = (size_t)n_tiles + 1;
    DevBuf<uint32_t> d_tile(4 * nt1);  // nl, tab, nl_before, tab_before
    uint32_t *t_nl = d_tile.p, *t_tab = d_tile.p + nt1, *t_nlb = d_tile.p + 2 * nt1, *t_tabb = d_tile.p + 3 * nt1;
    uint32_t *h_tot = reinterpret_cast<uint32_t *>(t_pinned.ensure(64));
    t_index.start();
    CK(cudaMemsetAsync(t_nl + n_tiles, 0, 4, stream()));
    CK(cudaMemsetAsync(t_tab + n_tiles, 0, 4, stream()));
    fm::fm_k_vcf_count<<<n_tiles, 256, 0, stream()>>>(reinterpret_cast<const uint4 *>(d_text), n16, t_nl, t_tab);
    CK(cudaGetLastError());
    size_t tmp_bytes = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, t_nl, t_nlb, (int)(2 * nt1), stream()));
    DevBuf<uint8_t> d_tmp(std::max<size_t>(tmp_bytes, 16));
    // one scan over [nl..., 0, tab..., 0]: nl_before[k] for the first half; the second half is offset by the
    // newline total, which fm_k_vcf_index subtracts through tab_before[0]
    CK(cub::DeviceScan::ExclusiveSum(d_tmp.p, tmp_bytes, t_nl, t_nlb, (int)(2 * nt1), stream()));
    CK(cudaMemcpyAsync(h_tot, t_nlb + n_tiles, 4, cudaMemcpyDeviceToHost, stream()));            // newline total
    CK(cudaMemcpyAsync(h_tot + 1, t_tabb + n_tiles, 4, cudaMemcpyDeviceToHost, stream()));        // + tab total
    CK(cudaStreamSynchronize(stream()));
    const uint32_t nl_total = h_tot[0], tab_total = h_tot[1] - h_tot[0];
    const size_t n_lines = (size_t)nl_total + (last_byte != '\n' ? 1 : 0);
    DevBuf<uint32_t> d_ls(n_lines + 1), d_tb(n_lines + 1);
    fm_k_vcf_index_ends<<<1, 1, 0, stream()>>>(d_ls.p, d_tb.p, (uint32_t)n_lines, (uint32_t)n_bytes, tab_total);
    CK(cudaGetLastError());
    fm::fm_k_vcf_index<<<n_tiles, 256, 0, stream()>>>(reinterpret_cast<const uint4 *>(d_text), n16, t_nlb, t_tabb,
                                                      nl_total, d_ls.p, d_tb.p);
    CK(cudaGetLastError());
    t_index.stop();
    g_launches += 3;
    fm::VcfParams P = sh.P;
    P.text = d_text;
    P.line_start = d_ls.p;
    P.tabs_before = d_tb.p;
    P.n_lines = (uint32_t)n_lines;
    DevBuf<fm::VcfLine> d_recs(n_lines);
    DevBuf<uint32_t> d_flag(n_lines + 1), d_row(n_lines + 1);  // one zero flag appended: the scan ends in the total
    t_parse.start();
    {
        const uint32_t blocks = (uint32_t)std::min<uint64_t>((n_lines + 7) / 8, 32ull * sms);
        fm::fm_k_vcf_fixed<<<blocks, 256, 0, stream()>>>(P, d_recs.p);
        CK(cudaGetLastError());
        fm_k_vcf_rowflag<<<(uint32_t)((n_lines + 256) / 256), 256, 0, stream()>>>(d_recs.p, (uint32_t)n_lines, d_flag.p);
        CK(cudaGetLastError());
    }
    CK(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_flag.p, d_row.p, (int)(n_lines + 1), stream()));
    DevBuf<uint8_t> d_tmp2(std::max<size_t>(tmp_bytes, 16));
    CK(cub::DeviceScan::ExclusiveSum(d_tmp2.p, tmp_bytes, d_flag.p, d_row.p, (int)(n_lines + 1), stream()));
    CK(cudaMemcpyAsync(h_tot + 2, d_row.p + n_lines, 4, cudaMemcpyDeviceToHost, stream()));
    CK(cudaStreamSynchronize(stream()));
    out.n_rows = h_tot[2];
    const size_t row_bytes = sh.n_kept * sh.max_ploidy;
    out.d_gt = static_cast<uint8_t *>(dev_alloc(std::max<size_t>(out.n_rows * row_bytes, 16)));
    {
        const uint32_t blocks = (uint32_t)std::min<uint64_t>(n_lines, 16ull * sms);
        fm::fm_k_vcf_samples<<<blocks, 256, 0, stream()>>>(P, d_recs.p, d_row.p, out.d_gt,
                                                           (uint32_t)(((n_bytes + 15) / 16) * 16 + 16));
        CK(cudaGetLastError());
    }
    t_parse.stop();
    g_launches += 3;
    {
        uint8_t *hp = t_pinned.ensure(64 + n_lines * (sizeof(fm::VcfLine) + 4));  // h_tot was consumed above
        CK(cudaMemcpyAsync(hp, d_recs.p, n_lines * sizeof(fm::VcfLine), cudaMemcpyDeviceToHost, stream()));
        CK(cudaMemcpyAsync(hp + n_lines * sizeof(fm::VcfLine), d_row.p, n_lines * 4, cudaMemcpyDeviceToHost, stream()));
        CK(cudaStreamSynchronize(stream()));
        const fm::VcfLine *hr = reinterpret_cast<const fm::VcfLine *>(hp);
        const uint32_t *hw = reinterpret_cast<const uint32_t *>(hp + n_lines * sizeof(fm::VcfLine));
        out.recs.assign(hr, hr + n_lines);
        out.rows.assign(hw, hw + n_lines);
    }
    out.index_ms = t_index.ms();
    out.parse_ms = t_parse.ms();
}

// Statistics, errors and the output order over the chunks of a call (in text order).
void vcf_finish(const VcfShared &sh, std::vector<VcfChunkOut> &chunks, float h2d_ms, fm_vcf_batch **out) {
    const size_t n_kept = sh.n_kept, max_ploidy = sh.max_ploidy, row_bytes = n_kept * max_ploidy;
    auto b = std::unique_ptr<fm_vcf_batch, void (*)(fm_vcf_batch *)>(new fm_vcf_batch(), [](fm_vcf_batch *x) {
        fm_vcf_batch_release(x);
    });
    b->device = t_device;
    b->S = n_kept;
    b->P = max_ploidy;
    fm_vcf_info &I = b->info;
    I.n_samples = n_kept;
    I.max_ploidy = max_ploidy;
    I.h2d_ms = h2d_ms;
    size_t n_lines = 0, n_rows = 0;
    for (auto &c : chunks) {
        n_lines += c.recs.size();
        n_rows += c.n_rows;
        I.index_ms += c.index_ms;
        I.parse_ms += c.parse_ms;
    }
    b->n_lines = n_lines;
    b->n_rows = n_rows;
    I.n_lines = n_lines;
    // genotype rows of all chunks in one buffer
    if (chunks.size() == 1) {
        b->d_gt = chunks[0].d_gt;
        chunks[0].d_gt = nullptr;
    } else if (!chunks.empty()) {
        b->d_gt = static_cast<uint8_t *>(dev_alloc(std::max<size_t>(n_rows * row_bytes, 16)));
        size_t r0 = 0;
        for (auto &c : chunks) {
            if (c.n_rows && row_bytes)
                CK(cudaMemcpyAsync(b->d_gt + r0 * row_bytes, c.d_gt, c.n_rows * row_bytes, cudaMemcpyDeviceToDevice,
                                   stream()));
            r0 += c.n_rows;
        }
        CK(cudaStreamSynchronize(stream()));
        for (auto &c : chunks) {
            dev_free(c.d_gt);
            c.d_gt = nullptr;
        }
    }
    struct Kept {
        const fm::VcfLine *r;
        uint32_t row;
    };
    std::vector<Kept> keep;
    keep.reserve(n_rows);
    size_t line0 = 0, row0 = 0;
    for (auto &c : chunks) {
        for (size_t li = 0; li < c.recs.size(); ++li) {
            const fm::VcfLine &r = c.recs[li];
            if (r.status == fm::VCF_SKIP) continue;
            if (r.status != fm::VCF_CAND) {
                b->err_line.push_back(line0 + li);
                b->err_code.push_back(r.status);
                // field count for the two format errors, the offending 1-based POS otherwise
                b->err_aux.push_back(r.status <= fm::VCF_E_MISSING_COLUMN ? r.pos0 : (int64_t)((uint64_t)r.pos0 + 1));
                continue;
            }
            const bool indel = r.indel & 1;
            I.total_variants++;
            if (r.flags & 2) I.filtered_due_to_allow++;
            if (r.flags & 1) I.filtered_due_to_mask++;
            if (r.indel & 2) I.mnp_variants++;
            if (r.flags & 4) I.low_gq_variants++;
            if (r.flags & 8) I.missing_data_variants++;
            I.total_data_points += n_kept;
            I.missing_data_points += r.missing_points;
            if (r.missing_points) b->pos_missing.push_back(r.pos0);
            if (r.flags != 0 || indel) {
                I.filtered_variants++;
                b->pos_filtered.push_back(r.pos0);
            }
            if (!indel) keep.push_back(Kept{&r, (uint32_t)(row0 + c.rows[li])});
        }
        line0 += c.recs.size();
        row0 += c.n_rows;
    }
    auto uniq = [](std::vector<int64_t> &v) {
        if (!std::is_sorted(v.begin(), v.end())) std::sort(v.begin(), v.end());
        v.erase(std::unique(v.begin(), v.end()), v.end());
    };
    uniq(b->pos_missing);
    uniq(b->pos_filtered);
    I.n_positions_with_missing = b->pos_missing.size();
    I.n_filtered_positions = b->pos_filtered.size();
    I.n_errors = b->err_line.size();
    // sort by position (stable), ties by the variant's compressed genotype bytes (process.rs:4377-4386);
    // a position-sorted VCF only needs the tie scan
    auto by_pos = [](const Kept &x, const Kept &y) { return x.r->pos0 < y.r->pos0; };
    if (!std::is_sorted(keep.begin(), keep.end(), by_pos)) std::stable_sort(keep.begin(), keep.end(), by_pos);
    for (size_t i = 0; i < keep.size();) {
        size_t j = i + 1;
        while (j < keep.size() && keep[j].r->pos0 == keep[i].r->pos0) ++j;
        if (j - i > 1 && row_bytes) {
            std::unordered_map<uint32_t, std::vector<uint8_t>> data;  // row -> compact CompressedGenotypes::data
            std::vector<uint8_t> raw(row_bytes);
            for (size_t k = i; k < j; ++k) {
                CK(cudaMemcpy(raw.data(), b->d_gt + (size_t)keep[k].row * row_bytes, row_bytes, cudaMemcpyDeviceToHost));
                const size_t st = std::max<size_t>(keep[k].r->stride, 1);
                std::vector<uint8_t> cdat(n_kept * st);
                for (size_t s = 0; s < n_kept; ++s)
                    for (size_t q = 0; q < st; ++q) cdat[s * st + q] = raw[s * max_ploidy + q];
                data.emplace(keep[k].row, std::move(cdat));
            }
            std::stable_sort(keep.begin() + i, keep.begin() + j,
                             [&](const Kept &x, const Kept &y) { return data[x.row] < data[y.row]; });
        }
        i = j;
    }
    b->var.resize(keep.size());
    b->order.resize(keep.size());
    for (size_t i = 0; i < keep.size(); ++i) {
        b->var[i] = *keep[i].r;
        if (b->var[i].stride == 0 && n_kept) b->var[i].stride = 1;  // CompressedGenotypes::new: max_ploidy.max(1)
        b->order[i] = keep[i].row;
    }
    I.n_variants = keep.size();
    b->d_order = static_cast<uint32_t *>(dev_alloc(std::max<size_t>(keep.size(), 4) * 4));
    if (!keep.empty())
        CK(cudaMemcpyAsync(b->d_order, b->order.data(), keep.size() * 4, cudaMemcpyHostToDevice, stream()));
    CK(cudaStreamSynchronize(stream()));
    *out = b.release();
}

struct VcfTrace {  // FM_VCF_TRACE=1: wall-clock phases of fm_vcf_parse on stderr
    bool on = env_u32_early("FM_VCF_TRACE", 0) != 0;
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    void mark(const char *what) {
        if (!on) return;
        const auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[fm_vcf] %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};

struct VcfChunkGuard {  // frees chunk buffers on every exit path
    std::vector<VcfChunkOut> v;
    ~VcfChunkGuard() {
        for (auto &c : v)
            if (c.d_gt) dev_free(c.d_gt);
    }
};

}  // namespace

fm_status fm_vcf_parse_device(const char *d_text, size_t n_bytes, char host_last_byte, const char *chr,
                              const int64_t *regions, size_t n_regions, const uint32_t *kept_col_indices,
                              size_t n_kept, uint16_t min_gq, int allow_mode, const int64_t *allow, size_t n_allow,
                              int mask_mode, const int64_t *mask, size_t n_mask, size_t max_ploidy,
                              fm_vcf_batch **out) {
    return guarded([&] {
        if (!out) fail(FM_ERR_INVALID_ARG, "out is NULL");
        *out = nullptr;
        if (n_bytes && !d_text) fail(FM_ERR_INVALID_ARG, "text is NULL");
        if (n_bytes >= (1ull << 31)) fail(FM_ERR_UNSUPPORTED, "more than 2^31 bytes of device text per call");
        if (reinterpret_cast<uintptr_t>(d_text) & 15u) fail(FM_ERR_INVALID_ARG, "device text must be 16-byte aligned");
        require_device();
        CK(cudaSetDevice(t_device));
        VcfShared sh;
        vcf_prepare(sh, chr, regions, n_regions, kept_col_indices, n_kept, min_gq, allow_mode, allow, n_allow, mask_mode,
                    mask, n_mask, max_ploidy);
        VcfChunkGuard g;
        if (n_bytes) {
            g.v.resize(1);
            vcf_chunk(sh, reinterpret_cast<const uint8_t *>(d_text), n_bytes, host_last_byte, g.v[0]);
        }
        vcf_finish(sh, g.v, 0.f, out);
    });
}

// Host text: cut into chunks of whole lines; an upload thread copies chunk after chunk on its own stream while
// this thread indexes and parses the chunks that have arrived (the stage is PCIe-bound: parse hides under the copy).
fm_status fm_vcf_parse(const char *text, size_t n_bytes, const char *chr, const int64_t *regions, size_t n_regions,
                       const uint32_t *kept_col_indices, size_t n_kept, uint16_t min_gq, int allow_mode,
                       const int64_t *allow, size_t n_allow, int mask_mode, const int64_t *mask, size_t n_mask,
                       size_t max_ploidy, fm_vcf_batch **out) {
    return guarded([&] {
        FM_NVTX("fm_vcf_parse");
        if (!out) fail(FM_ERR_INVALID_ARG, "out is NULL");
        *out = nullptr;
        if (n_bytes && !text) fail(FM_ERR_INVALID_ARG, "text is NULL");
        if (n_bytes >= (1ull << 40)) fail(FM_ERR_UNSUPPORTED, "more than 2^40 bytes per call");
        require_device();
        CK(cudaSetDevice(t_device));
        VcfTrace tr;
        VcfShared sh;
        vcf_prepare(sh, chr, regions, n_regions, kept_col_indices, n_kept, min_gq, allow_mode, allow, n_allow, mask_mode,
                    mask, n_mask, max_ploidy);
        tr.mark("prepare");
        // chunk boundaries on line ends
        size_t target = (size_t)env_u32_early("FM_VCF_CHUNK_MB", 64) << 20;
        if (const uint32_t tb = env_u32_early("FM_VCF_CHUNK_BYTES", 0)) target = tb;  // tests: many tiny chunks
        std::vector<size_t> cut{0};
        while (cut.back() < n_bytes) {
            size_t end = cut.back() + target;
            if (end >= n_bytes) {
                end = n_bytes;
            } else {
                const void *nl = memchr(text + end, '\n', std::min<size_t>(n_bytes - end, (size_t)1 << 30));
                end = nl ? (size_t)(static_cast<const char *>(nl) - text) + 1 : n_bytes;
            }
            if (end - cut.back() >= (1ull << 31)) fail(FM_ERR_UNSUPPORTED, "a single line run exceeds 2^31 bytes");
            cut.push_back(end);
        }
        const size_t nc = cut.size() - 1;
        // device layout: every chunk starts 16-byte aligned and is followed by >= 32 zero bytes
        std::vector<size_t> doff(nc + 1, 0);
        for (size_t c = 0; c < nc; ++c) doff[c + 1] = doff[c] + ((cut[c + 1] - cut[c] + 15) / 16) * 16 + 32;
        DevBuf<uint8_t> d_text(std::max<size_t>(doff[nc], 64));
        VcfChunkGuard g;
        g.v.resize(nc);
        const int dev = t_device;
        std::vector<cudaEvent_t> ev(nc, nullptr);
        std::atomic<size_t> recorded{0};
        std::atomic<int> copy_err{0};
        std::string copy_msg;
        float h2d_ms = 0.f;
        cudaStream_t cs = nullptr;
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        auto cleanup = [&] {
            for (auto &e : ev)
                if (e) cudaEventDestroy(e);
            if (e0) cudaEventDestroy(e0);
            if (e1) cudaEventDestroy(e1);
            if (cs) cudaStreamDestroy(cs);
        };
        try {
            CK(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
            CK(cudaEventCreate(&e0));
            CK(cudaEventCreate(&e1));
            for (auto &e : ev) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            CK(cudaStreamSynchronize(stream()));  // d_text may be a recycled block still in use on this stream
            tr.mark("alloc + streams");
            std::thread uploader([&] {
                try {
                    CK(cudaSetDevice(dev));
                    CK(cudaEventRecord(e0, cs));
                    for (size_t c = 0; c < nc; ++c) {
                        const size_t nb = cut[c + 1] - cut[c], body = ((nb + 15) / 16) * 16;
                        const size_t tail = body >= 16 ? body - 16 : 0;  // partial last word + padding read zero
                        CK(cudaMemsetAsync(d_text.p + doff[c] + tail, 0, body + 32 - tail, cs));
                        h2d(d_text.p + doff[c], text + cut[c], nb, cs);
                        CK(cudaEventRecord(ev[c], cs));
                        recorded.store(c + 1, std::memory_order_release);
                    }
                    CK(cudaEventRecord(e1, cs));
                    CK(cudaStreamSynchronize(cs));
                } catch (const FmError &e) {
                    copy_msg = e.msg;
                    copy_err.store(e.code ? e.code : FM_ERR_CUDA);
                    recorded.store(nc, std::memory_order_release);
                } catch (...) {  // nothing may escape a std::thread
                    copy_msg = "upload thread failed";
                    copy_err.store(FM_ERR_CUDA);
                    recorded.store(nc, std::memory_order_release);
                }
            });
            try {
                for (size_t c = 0; c < nc; ++c) {
                    while (recorded.load(std::memory_order_acquire) <= c && !copy_err.load()) std::this_thread::yield();
                    if (copy_err.load()) break;
                    CK(cudaStreamWaitEvent(stream(), ev[c], 0));
                    vcf_chunk(sh, d_text.p + doff[c], cut[c + 1] - cut[c], text[cut[c + 1] - 1], g.v[c]);
                }
            } catch (...) {
                uploader.join();
                throw;
            }
            tr.mark("chunks parsed");
            uploader.join();
            if (copy_err.load()) fail(copy_err.load(), copy_msg);
            if (nc) CK(cudaEventElapsedTime(&h2d_ms, e0, e1));
        } catch (...) {
            cleanup();
            throw;
        }
        cleanup();
        tr.mark("join + cleanup");
        t_tim.h2d_ms += h2d_ms;
        vcf_finish(sh, g.v, h2d_ms, out);
        tr.mark("finish");
    });
}

fm_status fm_vcf_batch_info(const fm_vcf_batch *b, fm_vcf_info *out) {
    if (!b || !out) return FM_ERR_INVALID_ARG;
    *out = b->info;
    return FM_OK;
}

fm_status fm_vcf_batch_variants(const fm_vcf_batch *b, int64_t *pos0, uint8_t *flags, uint8_t *stride, uint8_t *ref,
                                uint8_t *n_alt, uint8_t *alts) {
    if (!b) return FM_ERR_INVALID_ARG;
    for (size_t i = 0; i < b->var.size(); ++i) {
        const fm::VcfLine &r = b->var[i];
        if (pos0) pos0[i] = r.pos0;
        if (flags) flags[i] = r.flags;
        if (stride) stride[i] = r.stride;
        if (ref) ref[i] = r.ref;
        if (n_alt) n_alt[i] = r.n_alt;
        if (alts) memcpy(alts + i * fm::VCF_MAX_ALTS, r.alts, fm::VCF_MAX_ALTS);
    }
    return FM_OK;
}

fm_status fm_vcf_batch_genotypes(const fm_vcf_batch *b, uint8_t *gt) {
    return guarded([&] {
        if (!b || !gt) fail(FM_ERR_INVALID_ARG, "batch or output is NULL");
        const size_t n = b->var.size(), row_bytes = b->S * b->P;
        if (!n || !row_bytes) return;
        CK(cudaSetDevice(b->device));
        DevBuf<uint8_t> d_out(n * row_bytes);
        const uint32_t blocks = (uint32_t)std::min<uint64_t>((n * row_bytes + 255) / 256, 32ull * sm_count(b->device));
        fm::fm_k_vcf_gather_rows<<<blocks, 256, 0, stream()>>>(b->d_gt, b->d_order, n, (uint32_t)row_bytes, d_out.p);
        CK(cudaGetLastError());
        g_launches++;
        CK(cudaMemcpyAsync(gt, d_out.p, n * row_bytes, cudaMemcpyDeviceToHost, stream()));
        CK(cudaStreamSynchronize(stream()));
    });
}

fm_status fm_vcf_batch_positions(const fm_vcf_batch *b, int which, int64_t *out, size_t capacity) {
    if (!b || (which != 0 && which != 1)) return FM_ERR_INVALID_ARG;
    const std::vector<int64_t> &v = which ? b->pos_filtered : b->pos_missing;
    if (capacity < v.size() || (!out && !v.empty())) return FM_ERR_INVALID_ARG;
    if (!v.empty()) memcpy(out, v.data(), v.size() * 8);
    return FM_OK;
}

fm_status fm_vcf_batch_errors(const fm_vcf_batch *b, uint64_t *line_index, int32_t *code, int64_t *aux,
                              size_t capacity) {
    if (!b || capacity < b->err_line.size()) return FM_ERR_INVALID_ARG;
    for (size_t i = 0; i < b->err_line.size(); ++i) {
        if (line_index) line_index[i] = b->err_line[i];
        if (code) code[i] = b->err_code[i];
        if (aux) aux[i] = b->err_aux[i];
    }
    return FM_OK;
}

fm_status fm_vcf_batch_matrix(const fm_vcf_batch *b, int pass_only, fm_matrix **out) {
    return guarded([&] {
        if (!b || !out) fail(FM_ERR_INVALID_ARG, "batch or out is NULL");
        *out = nullptr;
        CK(cudaSetDevice(b->device));
        std::vector<uint32_t> order;
        std::vector<int64_t> pos;
        size_t ploidy = 0;  // from_variants: longest genotype over the selected variants (stats.rs:349-359)
        for (size_t i = 0; i < b->var.size(); ++i) {
            if (pass_only && b->var[i].flags != 0) continue;
            order.push_back(b->order[i]);
            pos.push_back(b->var[i].pos0);
            // a variant whose samples are all None has no genotype at all: its recorded stride of 1 is only the
            // CompressedGenotypes floor and does not count
            if (b->var[i].missing_points < b->S) ploidy = std::max<size_t>(ploidy, b->var[i].stride);
        }
        if (order.empty() || b->S == 0) return;  // from_variants: None
        if (ploidy == 0) return;  // effectively no data (stats.rs:362-365)
        const size_t V = order.size(), S = b->S;
        DevBuf<uint32_t> d_ord(V), d_max(1);
        d_ord.upload(order.data(), V);
        CK(cudaMemsetAsync(d_max.p, 0, 4, stream()));
        uint8_t *d_data = static_cast<uint8_t *>(dev_alloc(std::max<size_t>(V * S * ploidy, 16)));
        fm_matrix *m = nullptr;
        try {
            if (b->P == 2 && ploidy == 2 && (S * 2) % 16 == 0) {  // whole 16-byte words per row: eight samples per thread
                const uint32_t row_u4 = (uint32_t)(S * 2 / 16);
                const uint32_t blocks = (uint32_t)std::min<uint64_t>((V * row_u4 + 255) / 256, 32ull * sm_count(b->device));
                fm::fm_k_vcf_to_matrix_p2<<<blocks, 256, 0, stream()>>>(reinterpret_cast<const uint4 *>(b->d_gt), d_ord.p, V,
                                                                        row_u4, reinterpret_cast<uint4 *>(d_data), d_max.p);
            } else {
                const uint32_t blocks = (uint32_t)std::min<uint64_t>((V * S + 255) / 256, 32ull * sm_count(b->device));
                fm::fm_k_vcf_to_matrix<<<blocks, 256, 0, stream()>>>(b->d_gt, d_ord.p, V, (uint32_t)S, (uint32_t)b->P,
                                                                     (uint32_t)ploidy, d_data, d_max.p);
            }
            CK(cudaGetLastError());
            g_launches++;
            uint32_t mx = 0;
            CK(cudaMemcpyAsync(&mx, d_max.p, 4, cudaMemcpyDeviceToHost, stream()));
            CK(cudaStreamSynchronize(stream()));
            if (mx > 127) fail(FM_ERR_UNSUPPORTED, "allele index above 127 in a VCF batch matrix");
            m = matrix_common(V, S, ploidy, (uint8_t)mx, pos.data());
            m->d_data = d_data;
            d_data = nullptr;
            m->has_missing = true;  // from_variants always returns Some(missing)
            m->in_band = true;
            m->d_pos = static_cast<int64_t *>(dev_alloc(std::max<size_t>(V, 1) * 8));
            CK(cudaMemcpyAsync(m->d_pos, m->pos.data(), V * 8, cudaMemcpyHostToDevice, stream()));
            CK(cudaStreamSynchronize(stream()));
            build_allele_remap(m);
        } catch (...) {
            if (d_data) dev_free(d_data);
            if (m) fm_matrix_release(m);
            throw;
        }
        *out = m;
    });
}

// The same matrix as PACKED rows (2 bits per genotype, resident): the batch's genotypes go straight from the parser's
// output to full-row bit words -- the reference-layout u8 matrix is never materialised (SURVEY 8 f1).  Biallelic
// batches only: when an allele index above 1 turns up the call fails with FM_ERR_UNSUPPORTED and the caller uses
// fm_vcf_batch_matrix.
fm_status fm_vcf_batch_matrix_packed(const fm_vcf_batch *b, int pass_only, fm_matrix **out) {
    return guarded([&] {
        FM_NVTX("fm_vcf_batch_matrix_packed");
        if (!b || !out) fail(FM_ERR_INVALID_ARG, "batch or out is NULL");
        *out = nullptr;
        CK(cudaSetDevice(b->device));
        std::vector<uint32_t> order;
        std::vector<int64_t> pos;
        size_t ploidy = 0;  // from_variants: longest genotype over the selected variants (stats.rs:349-359)
        for (size_t i = 0; i < b->var.size(); ++i) {
            if (pass_only && b->var[i].flags != 0) continue;
            order.push_back(b->order[i]);
            pos.push_back(b->var[i].pos0);
            if (b->var[i].missing_points < b->S) ploidy = std::max<size_t>(ploidy, b->var[i].stride);
        }
        if (order.empty() || b->S == 0 || ploidy == 0) return;  // from_variants: None
        const size_t V = order.size(), S = b->S;
        fm_matrix *m = matrix_common(V, S, ploidy, 1, pos.data());
        try {
            m->has_missing = true;  // from_variants always returns Some(missing)
            m->streamed = true;
            ensure_packed_storage(m, true);
            DevBuf<uint32_t> d_ord(V), d_max(1);
            d_ord.upload(order.data(), V);
            CK(cudaMemsetAsync(d_max.p, 0, 4, stream()));
            const uint64_t words = (uint64_t)V * m->rw;
            const uint32_t blocks = (uint32_t)std::min<uint64_t>((words + 255) / 256, 32ull * sm_count(b->device));
            fm::fm_k_vcf_to_packed<<<std::max(blocks, 1u), 256, 0, stream()>>>(b->d_gt, d_ord.p, V, (uint32_t)S, (uint32_t)b->P,
                                                                                (uint32_t)ploidy, m->rw, m->d_abits, m->d_cbits,
                                                                                d_max.p);
            CK(cudaGetLastError());
            g_launches++;
            uint32_t mx = 0;
            CK(cudaMemcpyAsync(&mx, d_max.p, 4, cudaMemcpyDeviceToHost, stream()));
            m->d_pos = static_cast<int64_t *>(dev_alloc(std::max<size_t>(V, 1) * 8));
            CK(cudaMemcpyAsync(m->d_pos, m->pos.data(), V * 8, cudaMemcpyHostToDevice, stream()));
            CK(cudaStreamSynchronize(stream()));
            if (mx > 1)
                fail(FM_ERR_UNSUPPORTED, "packed rows carry one allele bit per cell: this batch has allele indices above 1 "
                                         "(use fm_vcf_batch_matrix)");
            m->max_allele = (uint8_t)mx;
        } catch (...) {
            fm_matrix_release(m);
            throw;
        }
        *out = m;
    });
}

fm_status fm_vcf_batch_release(fm_vcf_batch *b) {
    if (!b) return FM_OK;
    cudaSetDevice(b->device);
    if (b->d_gt) dev_free(b->d_gt);
    if (b->d_order) dev_free(b->d_order);
    delete b;
    return FM_OK;
}

// ------------------------------------------------------------------------------------ pairwise differences
fm_status fm_pairwise_differences(fm_matrix *m, size_t n_samples, uint32_t *differences, uint32_t *comparable,
                                  uint64_t *pair_start, int64_t *positions, size_t positions_capacity,
                                  size_t *n_positions_out) {
    return guarded([&] {
        FM_NVTX("fm_pairwise_differences (transpose + pair bit-GEMM)");
        require_device();
        if (!m) fail(FM_ERR_INVALID_ARG, "matrix is NULL");
        if (n_samples > m->S) fail(FM_ERR_INVALID_ARG, "n_samples exceeds the matrix's sample count");
        if (m->ploidy < 1 || m->ploidy > 2)
            fail(FM_ERR_UNSUPPORTED, "pairwise differences support ploidy 1 and 2 on the GPU path");
        if (m->streamed && !m->packed)
            fail(FM_ERR_UNSUPPORTED, "pairwise differences need resident rows: this matrix was streamed as u8 rows");
        uint32_t n_bits = 1;
        while ((1u << n_bits) <= m->plane_max_allele) ++n_bits;
        if (n_bits > 4)
            fail(FM_ERR_UNSUPPORTED, "more than 16 distinct allele values (or allele indices above 15 on a streamed / "
                                     "device-owned matrix) are not supported on the GPU path");
        if (n_samples >= (1u << 21)) fail(FM_ERR_UNSUPPORTED, "more than 2^21 samples per pairwise call");
        const uint64_t n_pairs = n_samples < 2 ? 0 : (uint64_t)n_samples * (n_samples - 1) / 2;
        if (n_pairs && !differences) fail(FM_ERR_INVALID_ARG, "differences is NULL");
        if (n_pairs == 0) {
            if (pair_start) pair_start[0] = 0;
            if (n_positions_out) *n_positions_out = 0;
            return;
        }
        set_dev(m);
        const uint32_t PL = (uint32_t)m->ploidy, S = (uint32_t)n_samples, V = (uint32_t)m->V;
        const bool hc = m->has_missing;
        const uint32_t n_words = (V + 31) / 32, n_chunks = (n_words + fm::kPwKT - 1) / fm::kPwKT;
        fm::PwLayout L{(S + fm::kPwBlk - 1) / fm::kPwBlk, (hc ? PL : 0u) + PL * (m->packed ? 1u : n_bits)};
        const size_t plane_words = (size_t)n_chunks * L.n_blk * L.tile_words();
        DevBuf<uint32_t> d_planes(std::max<size_t>(plane_words, 4));
        DevBuf<uint32_t> d_diff(n_pairs), d_comp(comparable ? n_pairs : 0);

        // 1. transpose into K-tiled sample-major planes
        Timer tm;
        tm.start();
        if (plane_words) {
            CK(cudaMemsetAsync(d_planes.p, 0, plane_words * 4, stream()));
            const uint64_t tasks = m->packed ? (uint64_t)n_words * ((S * PL + 31) / 32) : (uint64_t)n_words * ((S + 31) / 32);
            const uint32_t grid = (uint32_t)std::min<uint64_t>((tasks + 7) / 8, 64ull * sm_count(m->device));
            if (m->packed) {
                const uint32_t n_cell_words = (S * PL + 31) / 32;
                if (PL == 1)
                    fm::fm_k_sample_planes_packed<1><<<grid, 256, 0, stream()>>>(m->d_abits, m->d_cbits, m->rw, V, S, n_words,
                                                                                n_cell_words, L, d_planes.p);
                else
                    fm::fm_k_sample_planes_packed<2><<<grid, 256, 0, stream()>>>(m->d_abits, m->d_cbits, m->rw, V, S, n_words,
                                                                                n_cell_words, L, d_planes.p);
            } else {
                const uint32_t miss_mode = !hc ? 0u : (m->in_band ? 2u : 1u);
                auto run = [&](auto kern) {
                    kern<<<grid, 256, 0, stream()>>>(m->d_data, m->d_missing, miss_mode, m->d_lut, V, S, (uint64_t)m->stride,
                                                     n_words, L, d_planes.p);
                };
                const uint32_t form = (PL - 1) * 4 + (n_bits - 1);  // one instantiation per (ploidy, allele bits)
                switch (form) {
                    case 0: run(fm::fm_k_sample_planes<1, 1>); break;
                    case 1: run(fm::fm_k_sample_planes<1, 2>); break;
                    case 2: run(fm::fm_k_sample_planes<1, 3>); break;
                    case 3: run(fm::fm_k_sample_planes<1, 4>); break;
                    case 4: run(fm::fm_k_sample_planes<2, 1>); break;
                    case 5: run(fm::fm_k_sample_planes<2, 2>); break;
                    case 6: run(fm::fm_k_sample_planes<2, 3>); break;
                    default: run(fm::fm_k_sample_planes<2, 4>); break;
                }
            }
            CK(cudaGetLastError());
            g_launches++;
        }
        tm.stop();
        t_tim.repack_ms += tm.ms();

        // 2. upper-triangle bit-GEMM over sample pairs
        const uint64_t n_tiles = (uint64_t)L.n_blk * (L.n_blk + 1) / 2;
        const size_t smem = (size_t)fm::kPwStages * 2 * L.tile_words() * 4 + 2 * fm::kPwStages * 8;
        auto kern = hc ? fm::fm_k_pairwise_counts<true> : fm::fm_k_pairwise_counts<false>;
        CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        Timer tk;
        tk.start();
        kern<<<(uint32_t)n_tiles, (fm::kPwConsumerWarps + 1) * 32, smem, stream()>>>(d_planes.p, L, n_chunks, S, V, d_diff.p,
                                                                                    comparable ? d_comp.p : nullptr);
        CK(cudaGetLastError());
        g_launches++;
        tk.stop();
        t_tim.stats_ms += tk.ms();
        t_tim.stats_launches++;
        d_diff.download(differences, n_pairs);
        if (comparable) d_comp.download(comparable, n_pairs);

        // 3. positions: exclusive scan of the counts, then one warp per pair
        if (pair_start || positions) {
            DevBuf<uint64_t> d_start(n_pairs + 1);
            thrust::transform_iterator<fm::U32ToU64, const uint32_t *> diff64(d_diff.p, fm::U32ToU64());
            size_t tmp_bytes = 0;
            CK(cub::DeviceScan::InclusiveSum(nullptr, tmp_bytes, diff64, d_start.p + 1, (int64_t)n_pairs, stream()));
            DevBuf<uint8_t> d_tmp(std::max<size_t>(tmp_bytes, 16));
            CK(cudaMemsetAsync(d_start.p, 0, 8, stream()));
            CK(cub::DeviceScan::InclusiveSum(d_tmp.p, tmp_bytes, diff64, d_start.p + 1, (int64_t)n_pairs, stream()));
            uint64_t total = 0;
            CK(cudaMemcpyAsync(&total, d_start.p + n_pairs, 8, cudaMemcpyDeviceToHost, stream()));
            if (pair_start) d_start.download(pair_start, n_pairs + 1);
            CK(cudaStreamSynchronize(stream()));
            if (n_positions_out) *n_positions_out = (size_t)total;
            if (positions) {
                if (total > positions_capacity)
                    fail(FM_ERR_INVALID_ARG, "positions capacity too small: *n_positions_out holds the number needed");
                if (total) {
                    if ((n_pairs + 7) / 8 >= (1ull << 31)) fail(FM_ERR_UNSUPPORTED, "too many pairs for a positions call");
                    DevBuf<int64_t> d_out(total);
                    const uint32_t blocks = (uint32_t)((n_pairs + 7) / 8);
                    if (hc)
                        fm::fm_k_pairwise_positions<true><<<blocks, 256, 0, stream()>>>(d_planes.p, L, n_words, S, n_pairs,
                                                                                        d_start.p, m->d_pos, d_out.p);
                    else
                        fm::fm_k_pairwise_positions<false><<<blocks, 256, 0, stream()>>>(d_planes.p, L, n_words, S, n_pairs,
                                                                                         d_start.p, m->d_pos, d_out.p);
                    CK(cudaGetLastError());
                    g_launches++;
                    d_out.download(positions, total);
                }
            }
        } else if (n_positions_out) {
            CK(cudaStreamSynchronize(stream()));
            uint64_t total = 0;
            for (uint64_t i = 0; i < n_pairs; ++i) total += differences[i];
            *n_positions_out = (size_t)total;
        }
        CK(cudaStreamSynchronize(stream()));
    });
}

// ------------------------------------------------------------------------------------ synthetic cohorts
fm_status fm_synth_fill(uint8_t *d_data, uint64_t *d_missing, size_t V, size_t S, size_t ploidy,
                        uint64_t first_variant, uint64_t seed, const uint16_t *pop_of_sample, double sigma,
                        double missing_rate) {
    return guarded([&] {
        require_device();
        CK(cudaSetDevice(t_device));
        const uint64_t stride = (uint64_t)S * ploidy;
        const uint64_t total = (uint64_t)V * stride;
        if (total == 0) return;
        if (!d_data) fail(FM_ERR_INVALID_ARG, "d_data is NULL");
        if (stride >= (1ull << 32)) fail(FM_ERR_UNSUPPORTED, "row stride exceeds 2^32 entries");
        if ((reinterpret_cast<uintptr_t>(d_data) & 15u) != 0) fail(FM_ERR_INVALID_ARG, "d_data must be 16-byte aligned");
        DevBuf<uint16_t> d_pop;
        if (pop_of_sample) {
            d_pop.alloc(S);
            d_pop.upload(pop_of_sample, S);
        }
        const uint32_t sigma_q = (uint32_t)std::min(65536.0, std::max(0.0, sigma * 65536.0));
        const uint32_t miss_q = (uint32_t)std::min(65536.0, std::max(0.0, missing_rate * 65536.0 + 0.5));
        const uint64_t n_words = (total + 63) / 64;
        const uint32_t blocks = (uint32_t)std::min<uint64_t>((n_words + 255) / 256, 64ull * sm_count(t_device));
        fm::fm_k_synth<<<blocks, 256, 0, stream()>>>(d_data, d_missing, total, (uint32_t)stride, (uint32_t)ploidy,
                                                     first_variant, seed, pop_of_sample ? d_pop.p : nullptr,
                                                     sigma_q, miss_q);
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(stream()));
    });
}

// ------------------------------------------------------------------------------------ bench hooks
fm_status fm_bench_diversity(fm_group *const *groups, size_t n_groups, int mode, const int64_t *mask_iv,
                             size_t n_mask, int iterations, fm_comm *comm, fm_bench_result *out, double *last_pi,
                             double *last_theta) {
    return guarded([&] {
        if (!groups || !n_groups || !out || iterations < 1) fail(FM_ERR_INVALID_ARG, "bad argument");
        if ((last_pi || last_theta) && mode != 1) fail(FM_ERR_INVALID_ARG, "per-site tracks need mode 1");
        require_device();
        std::memset(out, 0, sizeof(*out));
        fm_matrix *m = groups[0]->m;
        set_dev(m);
        const uint32_t V = (uint32_t)m->V;
        struct PerGroup {
            DevBuf<double> part_pi[2], pi, theta, sd[2];  // batch / super-batch partials double-buffered by step
            DevBuf<uint32_t> part_u[2];                    // parity: reductions and exchange of step i overlap step i+1
            DevBuf<uint64_t> su[2];
        };
        std::vector<PerGroup> pg(n_groups);
        DevBuf<int64_t> d_mask;
        DevBuf<uint32_t> d_flags, d_flags2;  // double-buffered by step parity
        std::vector<int64_t> merged;
        const fm::PassGeom G = batch_range(0, V);  // every group's batches
        const uint32_t nb_all = G.n_batches;
        if (mode == 1 && mask_iv) {
            merge_intervals(mask_iv, n_mask, merged);
            d_mask.alloc(std::max<size_t>(merged.size(), 2));
            d_mask.upload(merged.data(), merged.size());
            d_flags.alloc(std::max<uint32_t>(nb_all, 1));
            d_flags2.alloc(std::max<uint32_t>(nb_all, 1));
        }
        const bool use_flags = mode == 1 && mask_iv && nb_all;
        uint32_t *flagbuf[2] = {d_flags.p, d_flags2.p};
        // The plane launches of one step, one set per step parity: the groups whose rows fit the row pass in ONE
        // launch of it (fm_k_plane_pass_seq), then one column-chunked launch per group with wider rows.
        // launch_groups[l]: the groups whose partials launch l writes.
        std::vector<std::vector<size_t>> launch_groups(1);
        for (size_t i = 0; i < n_groups; ++i) {
            if (row_lanes_log2(groups[i]->wq) < 5)
                launch_groups[0].push_back(i);
            else
                launch_groups.push_back({i});
        }
        const bool rows = !launch_groups[0].empty();
        if (!rows) launch_groups.erase(launch_groups.begin());
        std::vector<fm::RowSeg> segs[2];
        std::vector<fm::ChunkParams> chunked[2];
        uint64_t bytes = 0;
        for (size_t i = 0; i < n_groups; ++i) {
            fm_group *g = groups[i];
            if (g->m != m) fail(FM_ERR_INVALID_ARG, "groups must share one matrix");
            const size_t nb = std::max<uint32_t>(nb_all, 1);
            for (int k = 0; k < 2; ++k) {
                pg[i].part_pi[k].alloc(nb);
                pg[i].part_u[k].alloc(nb * 2);
                pg[i].sd[k].alloc(nb / fm::kSuperBatches + 2);
                pg[i].su[k].alloc(2 * (nb / fm::kSuperBatches + 2));
            }
            bytes += (uint64_t)V * plane_site_bytes(planes_of(g));
            if (i < 8) out->group_bytes[i] = (uint64_t)V * plane_site_bytes(planes_of(g)) + (mode == 1 ? (uint64_t)V * 16u : 0);
            if (mode == 1) {
                pg[i].pi.alloc(std::max<uint32_t>(V, 1));
                pg[i].theta.alloc(std::max<uint32_t>(V, 1));
                bytes += (uint64_t)V * 16u;
            }
            for (int k = 0; k < 2; ++k) {
                fm::DivEpilogue e{};
                set_tables(e, g);
                e.pi_form = FM_PIFORM_COUNTS;
                e.part_pi = pg[i].part_pi[k].p;
                e.part_u = pg[i].part_u[k].p;
                if (mode == 1) {
                    e.pi_out = pg[i].pi.p;
                    e.theta_out = pg[i].theta.p;
                    e.pi_form = FM_PIFORM_COMPONENTS;
                    if (use_flags) e.site_flags = flagbuf[k];
                }
                if (row_lanes_log2(g->wq) < 5)
                    segs[k].push_back(div_seg(g, e, 0, V));
                else
                    chunked[k].push_back(fm::ChunkParams{planes_of(g), make_geom(g, 0, V), e});
            }
        }
        RowPlan plan[2];
        for (int k = 0; k < 2 && rows; ++k)
            if (!plan_rows(segs[k], nullptr, plan[k])) fail(FM_ERR_INVALID_ARG, "internal: the groups do not fit one row pass");
        const size_t n_launch = launch_groups.size();
        EventPairs evs;
        std::vector<std::pair<cudaEvent_t, cudaEvent_t>> spans, comm_spans;
        cudaEvent_t t0 = evs.next(), t1 = evs.next();
        // Two streams: the plane passes run back to back on the main stream; everything small --
        // the mask lookup of the NEXT step, the partial reductions and the peer exchange of THIS
        // step -- runs on a side stream underneath them (partials / flags are double-buffered by
        // step parity).  The step's kernels never wait for a peer.
        struct SideStream {
            cudaStream_t s = nullptr;
            ~SideStream() {
                if (s) cudaStreamDestroy(s);
            }
        } side, xchg;  // side: mask lookup + reductions; xchg: the peer exchange (may wait for other ranks)
        CK(cudaStreamCreateWithFlags(&side.s, cudaStreamNonBlocking));
        if (comm) CK(cudaStreamCreateWithFlags(&xchg.s, cudaStreamNonBlocking));
        std::vector<cudaEvent_t> flags_ready(iterations, nullptr), side_done(iterations, nullptr);
        auto ev = [&]() {
            cudaEvent_t e;
            CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            evs.ev.push_back(e);
            return e;
        };
        auto launch_flags = [&](int it) {  // on the side stream, into buffer it & 1
            launch_site_flags(m, 0, V, 0, nb_all, d_mask.p, (uint32_t)(merged.size() / 2), nullptr, 0, flagbuf[it & 1],
                              side.s);
            flags_ready[it] = ev();
            CK(cudaEventRecord(flags_ready[it], side.s));
            out->other_launches++;
        };
        CK(cudaStreamSynchronize(stream()));
        // start line on the device: an exchange without payload is a barrier over the mailboxes, so every rank's t0
        // fires within microseconds of the others (the host-side barrier before this call leaves the ranks hundreds
        // of microseconds apart after their own setup above, which the first timed exchange would then absorb)
        if (comm) comm_launch(comm, nullptr, 0, 0, nullptr, 0, stream());
        CK(cudaEventRecord(t0, stream()));
        if (use_flags) {
            CK(cudaStreamWaitEvent(side.s, t0, 0));
            launch_flags(0);
        }
        uint32_t s_lo = 0, n_super = 0;
        super_range(G, s_lo, n_super);
        for (int it = 0; it < iterations; ++it) {
            const int pb = it & 1;
            // buffers of parity pb were last read by the side work of step it - 2
            if (it >= 2) CK(cudaStreamWaitEvent(stream(), side_done[it - 2], 0));
            if (use_flags) CK(cudaStreamWaitEvent(stream(), flags_ready[it], 0));
            if (use_flags && it + 1 < iterations) launch_flags(it + 1);  // next step's mask bits, under this step's passes
            for (size_t l = 0; l < n_launch; ++l) {
                cudaEvent_t a = evs.next(), b = evs.next();
                CK(cudaEventRecord(a, stream()));
                if (rows && l == 0)
                    launch_rows(plan[pb], m->device);
                else
                    launch_chunked(chunked[pb][l - (rows ? 1 : 0)], m->device);
                CK(cudaEventRecord(b, stream()));
                spans.emplace_back(a, b);
                out->plane_launches++;
                // side stream: reduce the partials of this launch's groups while the next pass streams
                CK(cudaStreamWaitEvent(side.s, b, 0));
                for (size_t i : launch_groups[l]) {
                    if (!nb_all) break;
                    launch_reduce(pg[i].part_pi[pb].p, 1, pg[i].part_u[pb].p, 2, G, pg[i].sd[pb].p, pg[i].su[pb].p,
                                  side.s);
                    out->other_launches++;
                }
            }
            if (comm) {  // fold the region totals of every group and exchange them with all ranks
                fm::CommFold folds[4];
                uint32_t nf = 0, words = 0;
                for (size_t i = 0; i < n_groups && nf < 4 && nb_all; ++i) {
                    folds[nf++] = fm::CommFold{pg[i].sd[pb].p,
                                               reinterpret_cast<const unsigned long long *>(pg[i].su[pb].p), n_super, 1u,
                                               2u};
                    words += 3;
                }
                cudaEvent_t red = ev(), a = evs.next(), b = evs.next();
                CK(cudaEventRecord(red, side.s));  // this step's reductions
                CK(cudaStreamWaitEvent(xchg.s, red, 0));
                CK(cudaEventRecord(a, xchg.s));
                comm_launch(comm, nullptr, words, 0, folds, nf, xchg.s);
                CK(cudaEventRecord(b, xchg.s));
                comm_spans.emplace_back(a, b);
                out->other_launches++;
                side_done[it] = b;  // buffers of this parity are free once the exchange has read them
            } else {
                side_done[it] = ev();
                CK(cudaEventRecord(side_done[it], side.s));
            }
        }
        CK(cudaStreamWaitEvent(stream(), side_done[iterations - 1], 0));  // all side work is inside the timed region
        CK(cudaEventRecord(t1, stream()));
        CK(cudaEventSynchronize(t1));
        float total = 0.f, plane = 0.f;
        CK(cudaEventElapsedTime(&total, t0, t1));
        for (size_t si = 0; si < spans.size(); ++si) {
            float t = 0.f;
            CK(cudaEventElapsedTime(&t, spans[si].first, spans[si].second));
            plane += t;
            const size_t gi = si % n_launch;
            if (gi < 8) out->group_ms_avg[gi] += t / (float)iterations;
        }
        if (comm) comm_check_status(comm);
        for (auto &sp : comm_spans) {
            float t = 0.f;
            CK(cudaEventElapsedTime(&t, sp.first, sp.second));
            out->comm_ms_avg += t / (float)comm_spans.size();
        }
        out->step_ms_avg = total / (float)iterations;
        out->plane_ms_avg = spans.empty() ? 0.f : plane / (float)spans.size();
        out->plane_bytes_per_step = bytes;
        // the tracks are written by every step into the same buffers: after the last one they hold its results
        for (size_t i = 0; i < n_groups && V; ++i) {
            if (last_pi)
                CK(cudaMemcpyAsync(last_pi + i * V, pg[i].pi.p, (size_t)V * sizeof(double), cudaMemcpyDefault, stream()));
            if (last_theta)
                CK(cudaMemcpyAsync(last_theta + i * V, pg[i].theta.p, (size_t)V * sizeof(double), cudaMemcpyDefault,
                                   stream()));
        }
        if (last_pi || last_theta) CK(cudaStreamSynchronize(stream()));
        // region totals of the LAST timed step (parity check of the run: bench.py compares them with the public
        // call and, for N > 1, the exchanged totals with a rank-ordered sum of every rank's local ones)
        const int pl = (iterations - 1) & 1;
        for (size_t i = 0; i < n_groups && i < 8 && nb_all; ++i) {
            std::vector<double> hd(n_super);
            std::vector<uint64_t> hu((size_t)n_super * 2);
            pg[i].sd[pl].download(hd.data(), n_super);
            pg[i].su[pl].download(hu.data(), (size_t)n_super * 2);
            CK(cudaStreamSynchronize(stream()));
            out->last_pi_sum[i] = fm::fm_comm_fold_host(hd.data(), n_super, 1, 0);  // association of the exchange fold
            for (uint32_t sb = 0; sb < n_super; ++sb) {
                out->last_seg[i] += hu[2 * (size_t)sb];
                out->last_unc[i] += hu[2 * (size_t)sb + 1];
            }
        }
        if (comm) {
            unsigned long long w[24] = {};
            const size_t nw = std::min<size_t>(n_groups, 8) * 3;
            CK(cudaMemcpyAsync(w, comm->d_merged, nw * 8, cudaMemcpyDeviceToHost, stream()));
            CK(cudaStreamSynchronize(stream()));
            for (size_t i = 0; i < n_groups && i < 8; ++i) {
                std::memcpy(&out->merged_pi_sum[i], &w[3 * i], 8);
                out->merged_seg[i] = w[3 * i + 1];
                out->merged_unc[i] = w[3 * i + 2];
            }
        }
    });
}

}  // extern "C"
