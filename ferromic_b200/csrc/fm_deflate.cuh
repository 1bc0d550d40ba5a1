// fm_deflate.cuh -- BGZF deflate on the device (DESIGN §0 row f7).  The input is cut into blocks of 0xff00 bytes, as
// bgzip cuts them, and every block becomes one BGZF member (gzip header with the `BC` subfield, one DEFLATE block,
// CRC32 + ISIZE trailer).  fm_k_deflate_members runs one CTA per block with the block staged in shared memory:
//
//   load      the block into shared memory (zero padded), clear the tables
//   match     LZ77 candidates, one position per thread, in chunks of DEFL_THREADS positions.  A position has two
//             candidates: the nearest earlier position of its 32-position group with the same 3 bytes (a warp vote,
//             __match_any_sync) and the hash table's entry, which holds the largest position + 1 of the EARLIER
//             chunks with the same hash (atomicMax after every chunk: the table is a pure function of the input).
//             The longer match wins (ties: the nearer one); lengths 3..258 at distances up to 32768.
//   parse     one thread walks the per-position match lengths in shared memory (greedy with a one-step lazy
//             check) and marks the token starts in a bitmap
//   huffman   literal/length and distance histograms (shared atomics on counts: order-free), length-limited codes
//             (15 bits; 7 for the code-length code) that are always complete: a tree with fewer than two used
//             symbols gets partners, as zlib does.  Then the smallest of dynamic, fixed and stored is chosen.
//   emit      every thread sums the bits of the tokens that start in its DEFL_SEG positions, a block-wide
//             exclusive scan places them, and the threads OR their bits into the member's slot in parallel
//   crc       one slice per thread (crc32_raw / crc32_slice_term / crc32_finish of fm_bgzf.cuh)
//
// fm_k_deflate_compact then copies the members, placed by an exclusive scan of their sizes, contiguously.
//
// Every phase is a __host__ __device__ function of (shared state, block, thread, thread count).  deflate_block_serial
// runs the same phases thread after thread on the CPU, so a CPU build (tests/bgzf_deflate_host.cpp) produces
// byte-identical members: no phase depends on the order in which its threads run, and the only warp-level step (the
// vote of the match phase) has a serial equivalent.
#pragma once
#include <stdint.h>

#include "fm_bgzf.cuh"

namespace fm {

constexpr uint32_t DEFL_BLOCK = 0xff00;                     // input bytes per member
constexpr uint32_t DEFL_THREADS = 512;                      // threads per CTA
constexpr uint32_t DEFL_SEG = 128;                          // positions per thread in the token phases
constexpr uint32_t DEFL_HBITS = 13;                         // hash table: 8192 entries
constexpr uint32_t DEFL_SLOT = 65536;                       // bytes of a member's slot (BSIZE <= 65536)
constexpr uint32_t DEFL_DATA_WORDS = (DEFL_BLOCK + 16) / 4;  // the block + zero padding for 4-byte compares
constexpr uint32_t DEFL_BITMAP_WORDS = DEFL_BLOCK / 32;
constexpr uint32_t DEFL_HEADER = 18, DEFL_TRAILER = 8;
static_assert(DEFL_THREADS * DEFL_SEG >= DEFL_BLOCK && DEFL_SEG % 32 == 0, "segments cover the block");
static_assert(DEFL_THREADS % 32 == 0, "chunks are whole warps");

enum : uint32_t { DEFL_STORED = 0, DEFL_FIXED = 1, DEFL_DYNAMIC = 2 };

struct DeflateShared {
    uint32_t data[DEFL_DATA_WORDS];  // the block, little-endian words, zero beyond n
    uint8_t len[DEFL_BLOCK];         // 0: literal; L - 2 for a match of L in 3..256; 255 for 258
    uint32_t head[1u << DEFL_HBITS];  // hash -> largest position + 1 of the earlier chunks (0: none)
    uint32_t start[DEFL_BITMAP_WORDS];  // token starts
    uint32_t crc_tab[256];
    uint32_t freq_lit[288], freq_dist[32], freq_cl[20];  // token counts (freq_lit[256]: end of block)
    uint32_t eff[288 + 32 + 20];     // the counts with partners added: what the trees are built from
    uint16_t order[288 + 32 + 20];   // used symbols by (count, symbol)
    uint32_t used[3];                // used symbols per tree
    uint32_t hw[2 * 288];            // tree build scratch: node weights
    uint16_t hparent[2 * 288], hdepth[2 * 288];
    uint16_t bl[16], next[16];
    uint16_t code_lit[288], code_dist[32], code_cl[20];  // bit-reversed canonical codes
    uint8_t len_lit[288], len_dist[32], len_cl[20];
    uint8_t rle_sym[288 + 32], rle_extra[288 + 32];
    uint32_t seg_bits[DEFL_THREADS];  // token bits per thread, then their exclusive scan
    uint32_t wsum[DEFL_THREADS / 32];
    uint32_t n, kind, hlit, hdist, hclen, n_rle, hdr_bits, payload, crc_xor, tok_bits;
};

struct DeflateBlock {
    const uint8_t *in;  // the block's input bytes
    uint32_t n;         // 1..DEFL_BLOCK
    uint32_t *slot;     // DEFL_SLOT / 4 words: the member
    uint16_t *dist;     // DEFL_BLOCK entries: match distance per position (written by the match phase)
};

// ------------------------------------------------------------------------------------------------- helpers
FM_BGZF_HD uint32_t defl_ctz(uint32_t x) {
#ifdef __CUDA_ARCH__
    return (uint32_t)__ffs((int)x) - 1;
#else
    return (uint32_t)__builtin_ctz(x);
#endif
}
FM_BGZF_HD void defl_or(uint32_t *p, uint32_t v) {
#ifdef __CUDA_ARCH__
    atomicOr(p, v);
#else
    *p |= v;
#endif
}
FM_BGZF_HD void defl_add(uint32_t *p, uint32_t v) {
#ifdef __CUDA_ARCH__
    atomicAdd(p, v);
#else
    *p += v;
#endif
}
FM_BGZF_HD void defl_max(uint32_t *p, uint32_t v) {
#ifdef __CUDA_ARCH__
    atomicMax(p, v);
#else
    if (*p < v) *p = v;
#endif
}
FM_BGZF_HD void defl_xor(uint32_t *p, uint32_t v) {
#ifdef __CUDA_ARCH__
    atomicXor(p, v);
#else
    *p ^= v;
#endif
}
FM_BGZF_HD uint32_t defl_clz(uint32_t x) {  // x != 0
#ifdef __CUDA_ARCH__
    return (uint32_t)__clz((int)x);
#else
    return (uint32_t)__builtin_clz(x);
#endif
}
// `nbits` (<= 32, value < 2^nbits) bits at bit `pos` of the zeroed word array `o`, LSB first
FM_BGZF_HD void defl_put(uint32_t *o, uint32_t pos, uint32_t value, uint32_t nbits) {
    if (!nbits) return;
    const uint32_t w = pos >> 5, sh = pos & 31;
    defl_or(o + w, value << sh);
    if (sh + nbits > 32) defl_or(o + w + 1, value >> (32 - sh));
}
FM_BGZF_HD uint32_t defl_load4(const uint32_t *d, uint32_t p) {
    const uint32_t w = p >> 2, s = (p & 3) * 8, lo = d[w];
#ifdef __CUDA_ARCH__
    return __funnelshift_r(lo, d[w + 1], s);
#else
    return s ? (lo >> s) | (d[w + 1] << (32 - s)) : lo;
#endif
}
FM_BGZF_HD uint32_t defl_byte(const DeflateShared &S, uint32_t p) { return (S.data[p >> 2] >> ((p & 3) * 8)) & 0xffu; }
// common prefix of positions i and j (< i), at most maxlen
FM_BGZF_HD uint32_t defl_match_len(const uint32_t *d, uint32_t i, uint32_t j, uint32_t maxlen) {
    uint32_t L = 0;
    while (L < maxlen) {
        const uint32_t x = defl_load4(d, i + L) ^ defl_load4(d, j + L);
        if (x) {
            L += defl_ctz(x) >> 3;
            break;
        }
        L += 4;
    }
    return L < maxlen ? L : maxlen;
}
// the 3 bytes at p (valid when p + 3 <= n); invalid positions get a key no valid position and no other lane has
FM_BGZF_HD uint32_t defl_key(const DeflateShared &S, uint32_t p) {
    return p + 3 <= S.n ? defl_load4(S.data, p) & 0xffffffu : 0x1000000u | (p & 31);
}
FM_BGZF_HD uint32_t defl_hash(uint32_t key) { return (key * 2654435761u) >> (32 - DEFL_HBITS); }
FM_BGZF_HD uint32_t defl_match_of(uint32_t v) { return v == 255 ? 258u : v + 2; }  // v != 0
// length L (3..258) -> symbol 257..285, extra bits, extra value
FM_BGZF_HD void defl_len_code(uint32_t L, uint32_t &sym, uint32_t &xb, uint32_t &xv) {
    if (L == 258) {
        sym = 285, xb = 0, xv = 0;
        return;
    }
    const uint32_t l = L - 3;
    if (l < 8) {
        sym = 257 + l, xb = 0, xv = 0;
        return;
    }
    const uint32_t x = 29 - defl_clz(l);  // floor(log2 l) - 2
    sym = 257 + 4 * x + 4 + ((l >> x) - 4), xb = x, xv = l & ((1u << x) - 1);
}
// distance 1..32768 -> symbol 0..29, extra bits, extra value
FM_BGZF_HD void defl_dist_code(uint32_t d, uint32_t &sym, uint32_t &xb, uint32_t &xv) {
    const uint32_t dd = d - 1;
    if (dd < 4) {
        sym = dd, xb = 0, xv = 0;
        return;
    }
    const uint32_t x = 30 - defl_clz(dd);  // floor(log2 dd) - 1
    sym = 2 * x + 2 + ((dd >> x) & 1), xb = x, xv = dd & ((1u << x) - 1);
}
FM_BGZF_HD uint32_t defl_len_extra(uint32_t sym) { return sym < 265 || sym == 285 ? 0u : (sym - 261) / 4; }
FM_BGZF_HD uint32_t defl_dist_extra(uint32_t sym) { return sym < 4 ? 0u : (sym - 2) / 2; }

// ------------------------------------------------------------------------------------------------- phases
FM_BGZF_HD void defl_load(DeflateShared &S, const DeflateBlock &B, uint32_t t, uint32_t nt) {
    if (t == 0) {
        S.n = B.n;
        S.crc_xor = 0;
    }
    for (uint32_t w = t; w < DEFL_DATA_WORDS; w += nt) {
        uint32_t v = 0;
        for (uint32_t k = 0; k < 4; ++k)
            if (4 * w + k < B.n) v |= (uint32_t)B.in[4 * w + k] << (8 * k);
        S.data[w] = v;
    }
    for (uint32_t i = t; i < (1u << DEFL_HBITS); i += nt) S.head[i] = 0;
    for (uint32_t i = t; i < DEFL_BITMAP_WORDS; i += nt) S.start[i] = 0;
    for (uint32_t i = t; i < 256; i += nt) S.crc_tab[i] = crc32_table_entry(i);
    for (uint32_t i = t; i < 288 + 32 + 20; i += nt) {
        if (i < 288) S.freq_lit[i] = 0;
        else if (i < 320) S.freq_dist[i - 288] = 0;
        else S.freq_cl[i - 320] = 0;
    }
}

// Candidates and match length of position c * nt + t; chunk c's positions are inserted by defl_insert afterwards.
FM_BGZF_HD void defl_match(DeflateShared &S, const DeflateBlock &B, uint32_t c, uint32_t t, uint32_t nt) {
    const uint32_t i = c * nt + t, n = B.n, key = defl_key(S, i);
    uint32_t jb = ~0u;  // nearest earlier position of the 32-group with the same 3 bytes
#ifdef __CUDA_ARCH__
    const uint32_t lane = i & 31, lower = __match_any_sync(0xffffffffu, key) & ((1u << lane) - 1);
    if (lower) jb = (i & ~31u) + 31 - __clz(lower);
#else
    if (i + 3 <= n)
        for (uint32_t k = i; k-- > (i & ~31u);)
            if (defl_key(S, k) == key) {
                jb = k;
                break;
            }
#endif
    if (i >= n) return;
    uint32_t best = 0, dist = 0;
    if (i + 3 <= n) {
        const uint32_t maxlen = n - i < 258 ? n - i : 258;
        if (jb != ~0u) {
            best = defl_match_len(S.data, i, jb, maxlen);
            dist = i - jb;
        }
        const uint32_t ja = S.head[defl_hash(key)];
        if (best < maxlen && ja && i - (ja - 1) <= 32768) {
            const uint32_t L = defl_match_len(S.data, i, ja - 1, maxlen);
            if (L > best) best = L, dist = i - (ja - 1);
        }
    }
    if (best == 257) best = 256;  // 257 costs what 256 does; 258 has its own symbol
    S.len[i] = best < 3 ? 0 : best == 258 ? 255 : (uint8_t)(best - 2);
    if (best >= 3) B.dist[i] = (uint16_t)dist;
}
FM_BGZF_HD void defl_insert(DeflateShared &S, const DeflateBlock &B, uint32_t c, uint32_t t, uint32_t nt) {
    const uint32_t i = c * nt + t;
    if (i + 3 <= B.n) defl_max(&S.head[defl_hash(defl_key(S, i))], i + 1);
}

// Serial: greedy with a one-step lazy check (a longer match at the next position turns this one into a literal).
FM_BGZF_HD void defl_parse(DeflateShared &S) {
    const uint32_t n = S.n;
    uint32_t p = 0, cw = 0, acc = 0;
    while (p < n) {
        const uint32_t v = S.len[p];
        uint32_t L = 1;
        if (v) {
            L = defl_match_of(v);
            const uint32_t v1 = p + 1 < n ? S.len[p + 1] : 0;
            if (v1 && defl_match_of(v1) > L) {
                S.len[p] = 0;
                L = 1;
            }
        }
        if ((p >> 5) != cw) {
            S.start[cw] = acc;
            cw = p >> 5;
            acc = 0;
        }
        acc |= 1u << (p & 31);
        p += L;
    }
    S.start[cw] = acc;
}

// Visits the tokens that start in thread t's positions: f(position, literal byte or ~0, match length, distance).
template <class F>
FM_BGZF_HD void defl_tokens(const DeflateShared &S, const DeflateBlock &B, uint32_t t, F &&f) {
    const uint32_t p0 = t * DEFL_SEG;
    if (p0 >= S.n) return;
    for (uint32_t w = p0 / 32; w < (p0 + DEFL_SEG) / 32 && w < DEFL_BITMAP_WORDS; ++w) {
        uint32_t bits = S.start[w];
        while (bits) {
            const uint32_t i = w * 32 + defl_ctz(bits);
            bits &= bits - 1;
            const uint32_t v = S.len[i];
            if (v) f(i, ~0u, defl_match_of(v), (uint32_t)B.dist[i]);
            else f(i, defl_byte(S, i), 1u, 0u);
        }
    }
}

FM_BGZF_HD void defl_histogram(DeflateShared &S, const DeflateBlock &B, uint32_t t, uint32_t) {
    if (t == 0) defl_add(&S.freq_lit[256], 1);
    defl_tokens(S, B, t, [&](uint32_t, uint32_t lit, uint32_t L, uint32_t d) {
        if (lit != ~0u) {
            defl_add(&S.freq_lit[lit], 1);
            return;
        }
        uint32_t s, xb, xv;
        defl_len_code(L, s, xb, xv);
        defl_add(&S.freq_lit[s], 1);
        defl_dist_code(d, s, xb, xv);
        defl_add(&S.freq_dist[s], 1);
    });
}

// Tree k (0: literal/length, 1: distance, 2: code length): nsym symbols from offset `base` of eff / order.
struct DeflTree {
    uint32_t base, nsym, maxbits;
};
FM_BGZF_HD DeflTree defl_tree(uint32_t k) {
    return k == 0 ? DeflTree{0, 286, 15} : k == 1 ? DeflTree{288, 30, 15} : DeflTree{320, 19, 7};
}

// Serial: the counts tree k is built from; fewer than two used symbols get partners of count 1 (smallest unused
// symbols first), so that every code is complete.
FM_BGZF_HD void defl_partners(DeflateShared &S, uint32_t k) {
    const DeflTree T = defl_tree(k);
    const uint32_t *f = k == 0 ? S.freq_lit : k == 1 ? S.freq_dist : S.freq_cl;
    uint32_t used = 0;
    for (uint32_t s = 0; s < T.nsym; ++s) {
        S.eff[T.base + s] = f[s];
        used += f[s] != 0;
    }
    for (uint32_t s = 0; s < T.nsym && used < 2; ++s)
        if (!S.eff[T.base + s]) {
            S.eff[T.base + s] = 1;
            ++used;
        }
    S.used[k] = used;
}
// Parallel: symbol s of tree k takes its rank among the used symbols by (count, symbol).
FM_BGZF_HD void defl_rank(DeflateShared &S, uint32_t k, uint32_t s) {
    const DeflTree T = defl_tree(k);
    if (s >= T.nsym) return;
    const uint32_t *e = S.eff + T.base, es = e[s];
    if (!es) return;
    uint32_t r = 0;
    for (uint32_t u = 0; u < T.nsym; ++u) r += e[u] && (e[u] < es || (e[u] == es && u < s));
    S.order[T.base + r] = (uint16_t)s;
}
// Serial: Huffman code lengths of tree k from the ranked counts (two-queue construction), limited to maxbits so that
// the code stays complete (the Kraft sum is brought back to exactly 1, as miniz does), then the canonical codes.
FM_BGZF_HD void defl_build(DeflateShared &S, uint32_t k, uint8_t *lens, uint16_t *codes) {
    const DeflTree T = defl_tree(k);
    const uint32_t m = S.used[k], *e = S.eff + T.base;
    const uint16_t *ord = S.order + T.base;
    for (uint32_t s = 0; s < T.nsym + (k == 0 ? 2u : k == 1 ? 2u : 1u); ++s) lens[s] = 0;
    // leaves 0..m-1 (ascending count), internal nodes m..2m-2 (created in ascending weight)
    for (uint32_t i = 0; i < m; ++i) S.hw[i] = e[ord[i]];
    uint32_t li = 0, ii = m, nn = m;
    for (uint32_t r = 0; r + 1 < m; ++r) {
        uint32_t pick[2];
        for (int q = 0; q < 2; ++q) {
            if (li < m && (ii >= nn || S.hw[li] <= S.hw[ii])) pick[q] = li++;
            else pick[q] = ii++;
        }
        S.hw[nn] = S.hw[pick[0]] + S.hw[pick[1]];
        S.hparent[pick[0]] = S.hparent[pick[1]] = (uint16_t)nn;
        ++nn;
    }
    for (uint32_t L = 0; L < 16; ++L) S.bl[L] = 0;
    S.hdepth[nn - 1] = 0;
    for (uint32_t v = nn - 1; v-- > 0;) S.hdepth[v] = (uint16_t)(S.hdepth[S.hparent[v]] + 1);
    for (uint32_t i = 0; i < m; ++i) S.bl[S.hdepth[i] < T.maxbits ? S.hdepth[i] : T.maxbits]++;
    uint32_t total = 0;
    for (uint32_t L = 1; L <= T.maxbits; ++L) total += (uint32_t)S.bl[L] << (T.maxbits - L);
    while (total > (1u << T.maxbits)) {
        S.bl[T.maxbits]--;
        for (uint32_t L = T.maxbits - 1; L > 0; --L)
            if (S.bl[L]) {
                S.bl[L]--;
                S.bl[L + 1] += 2;
                break;
            }
        --total;
    }
    uint32_t r = 0;  // the rarest symbols take the longest codes
    for (uint32_t L = T.maxbits; L > 0; --L)
        for (uint32_t c = S.bl[L]; c; --c) lens[ord[r++]] = (uint8_t)L;
    // canonical codes, bit-reversed for LSB-first emission
    uint32_t code = 0;
    for (uint32_t L = 1; L < 16; ++L) {
        code = (code + S.bl[L - 1]) << 1;
        S.next[L] = (uint16_t)code;
    }
    S.next[0] = 0;
    for (uint32_t s = 0; s < T.nsym; ++s) {
        const uint32_t L = lens[s];
        if (!L) continue;
        const uint32_t c = S.next[L]++;
        uint32_t rev = 0;
        for (uint32_t b = 0; b < L; ++b) rev |= ((c >> b) & 1u) << (L - 1 - b);
        codes[s] = (uint16_t)rev;
    }
}
FM_BGZF_HD void defl_fixed_codes(DeflateShared &S) {
    for (uint32_t s = 0; s < 288; ++s) S.len_lit[s] = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
    for (uint32_t s = 0; s < 32; ++s) S.len_dist[s] = 5;
    for (uint32_t L = 0; L < 16; ++L) S.bl[L] = 0;
    for (uint32_t s = 0; s < 288; ++s) S.bl[S.len_lit[s]]++;
    S.bl[0] = 0;
    uint32_t code = 0;
    for (uint32_t L = 1; L < 16; ++L) {
        code = (code + S.bl[L - 1]) << 1;
        S.next[L] = (uint16_t)code;
    }
    for (uint32_t s = 0; s < 288 + 32; ++s) {
        const uint32_t L = s < 288 ? S.len_lit[s] : 5, c = s < 288 ? S.next[L]++ : s - 288;
        uint32_t rev = 0;
        for (uint32_t b = 0; b < L; ++b) rev |= ((c >> b) & 1u) << (L - 1 - b);
        if (s < 288) S.code_lit[s] = (uint16_t)rev;
        else S.code_dist[s - 288] = (uint16_t)rev;
    }
}

// Serial: run-length symbols (16/17/18) of lens[0, n) appended to the RLE list, as zlib's scan_tree cuts them.
FM_BGZF_HD void defl_rle(DeflateShared &S, const uint8_t *lens, uint32_t n) {
    auto emit = [&](uint32_t sym, uint32_t extra) {
        S.rle_sym[S.n_rle] = (uint8_t)sym;
        S.rle_extra[S.n_rle] = (uint8_t)extra;
        S.n_rle++;
        S.freq_cl[sym]++;
    };
    int prev = -1;
    uint32_t next = lens[0], count = 0, max_count = next ? 7 : 138, min_count = next ? 4 : 3;
    for (uint32_t s = 0; s < n; ++s) {
        const uint32_t cur = next;
        next = s + 1 < n ? lens[s + 1] : 0xffffu;
        if (++count < max_count && cur == next) continue;
        if (count < min_count) {
            while (count--) emit(cur, 0);
        } else if (cur != 0) {
            if ((int)cur != prev) {
                emit(cur, 0);
                --count;
            }
            emit(16, count - 3);
        } else if (count <= 10) {
            emit(17, count - 3);
        } else {
            emit(18, count - 11);
        }
        count = 0;
        prev = (int)cur;
        if (next == 0) max_count = 138, min_count = 3;
        else if (cur == next) max_count = 6, min_count = 3;
        else max_count = 7, min_count = 4;
    }
}

// the order of the code-length code lengths in the block header: 16 17 18 0 8 7 9 6 10 5 11 4 12 3 13 2 14 1 15
FM_BGZF_HD uint32_t defl_cl_order(uint32_t i) {
    return i < 3 ? 16 + i : i == 3 ? 0u : (i & 1) ? 7 - (i - 5) / 2 : 8 + (i - 4) / 2;
}

// Serial, after the literal/length and distance trees: HLIT / HDIST, the run-length list and its counts.
FM_BGZF_HD void defl_tables(DeflateShared &S) {
    uint32_t hlit = 286, hdist = 30;
    while (hlit > 257 && !S.len_lit[hlit - 1]) --hlit;
    while (hdist > 1 && !S.len_dist[hdist - 1]) --hdist;
    S.hlit = hlit;
    S.hdist = hdist;
    S.n_rle = 0;
    defl_rle(S, S.len_lit, hlit);
    defl_rle(S, S.len_dist, hdist);
}

// Serial, after the code-length tree: the sizes of the three encodings; keeps the smallest (ties: stored, then
// fixed) and leaves that encoding's codes in code_lit / code_dist.
FM_BGZF_HD void defl_choose(DeflateShared &S) {
    uint32_t hclen = 19;
    while (hclen > 4 && !S.len_cl[defl_cl_order(hclen - 1)]) --hclen;
    S.hclen = hclen;
    uint32_t hdr = 3 + 14 + 3 * hclen;
    for (uint32_t r = 0; r < S.n_rle; ++r) {
        const uint32_t s = S.rle_sym[r];
        hdr += S.len_cl[s] + (s == 16 ? 2u : s == 17 ? 3u : s == 18 ? 7u : 0u);
    }
    uint32_t dyn = hdr, fix = 3;
    for (uint32_t s = 0; s < 286; ++s) {
        const uint32_t f = S.freq_lit[s], x = s > 256 ? defl_len_extra(s) : 0u;
        dyn += f * (S.len_lit[s] + x);
        fix += f * ((s < 144 ? 8u : s < 256 ? 9u : s < 280 ? 7u : 8u) + x);
    }
    for (uint32_t s = 0; s < 30; ++s) {
        const uint32_t f = S.freq_dist[s], x = defl_dist_extra(s);
        dyn += f * (S.len_dist[s] + x);
        fix += f * (5 + x);
    }
    const uint32_t stored = S.n + 5, dyn_b = (dyn + 7) / 8, fix_b = (fix + 7) / 8;
    S.kind = DEFL_STORED;
    S.payload = stored;
    if (fix_b < S.payload) S.kind = DEFL_FIXED, S.payload = fix_b;
    if (dyn_b < S.payload) S.kind = DEFL_DYNAMIC, S.payload = dyn_b;
    S.hdr_bits = S.kind == DEFL_DYNAMIC ? hdr : 3;
    if (S.kind == DEFL_FIXED) defl_fixed_codes(S);
}

// Bits of the tokens that start in thread t's positions.
FM_BGZF_HD void defl_token_bits(DeflateShared &S, const DeflateBlock &B, uint32_t t, uint32_t) {
    uint32_t bits = 0;
    if (S.kind != DEFL_STORED)
        defl_tokens(S, B, t, [&](uint32_t, uint32_t lit, uint32_t L, uint32_t d) {
            if (lit != ~0u) {
                bits += S.len_lit[lit];
                return;
            }
            uint32_t s, xb, xv;
            defl_len_code(L, s, xb, xv);
            bits += S.len_lit[s] + xb;
            defl_dist_code(d, s, xb, xv);
            bits += S.len_dist[s] + xb;
        });
    S.seg_bits[t] = bits;
}

// Thread t's CRC slice term (the block's bytes [t * DEFL_SEG, ...) of crc32_slice_term).
FM_BGZF_HD void defl_crc(DeflateShared &S, uint32_t t, uint32_t) {
    const uint32_t n = S.n, b0 = t * DEFL_SEG < n ? t * DEFL_SEG : n, b1 = b0 + DEFL_SEG < n ? b0 + DEFL_SEG : n;
    if (b1 > b0)
        defl_xor(&S.crc_xor, crc32_slice_term(crc32_raw(S.crc_tab, reinterpret_cast<const uint8_t *>(S.data) + b0,
                                                        b1 - b0), b1, n));
}

FM_BGZF_HD uint32_t defl_member_bytes(const DeflateShared &S) { return DEFL_HEADER + S.payload + DEFL_TRAILER; }

FM_BGZF_HD void defl_zero_slot(const DeflateShared &S, const DeflateBlock &B, uint32_t t, uint32_t nt) {
    for (uint32_t w = t; w < (defl_member_bytes(S) + 7) / 4; w += nt) B.slot[w] = 0;
}

// Serial: the gzip header, the deflate block header (and the dynamic tables), the end of block, the trailer.
FM_BGZF_HD void defl_frame(DeflateShared &S, const DeflateBlock &B, uint32_t token_bits) {
    uint32_t *o = B.slot;
    const uint32_t size = defl_member_bytes(S);
    defl_put(o, 0, 0x04088b1fu, 32);          // ID1 ID2 CM=8 FLG=FEXTRA
    defl_put(o, 32, 0, 32);                   // MTIME 0
    defl_put(o, 64, 0xff00u, 16);             // XFL 0, OS 255
    defl_put(o, 80, 0x43420006u, 32);         // XLEN 6, 'B' 'C'
    defl_put(o, 112, 2 | (size - 1) << 16, 32);  // SLEN 2, BSIZE - 1
    const uint32_t at = DEFL_HEADER * 8;
    uint32_t p = at;
    if (S.kind == DEFL_STORED) {
        defl_put(o, p, 1, 8);  // BFINAL, BTYPE 00, padding
        defl_put(o, p + 8, S.n | (~S.n & 0xffffu) << 16, 32);
    } else {
        defl_put(o, p, S.kind == DEFL_FIXED ? 3u : 5u, 3);
        p += 3;
        if (S.kind == DEFL_DYNAMIC) {
            defl_put(o, p, S.hlit - 257, 5);
            defl_put(o, p + 5, S.hdist - 1, 5);
            defl_put(o, p + 10, S.hclen - 4, 4);
            p += 14;
            for (uint32_t i = 0; i < S.hclen; ++i, p += 3) defl_put(o, p, S.len_cl[defl_cl_order(i)], 3);
            for (uint32_t r = 0; r < S.n_rle; ++r) {
                const uint32_t s = S.rle_sym[r], xb = s == 16 ? 2u : s == 17 ? 3u : s == 18 ? 7u : 0u;
                defl_put(o, p, S.code_cl[s], S.len_cl[s]);
                p += S.len_cl[s];
                defl_put(o, p, S.rle_extra[r], xb);
                p += xb;
            }
        }
        defl_put(o, at + S.hdr_bits + token_bits, S.code_lit[256], S.len_lit[256]);
    }
    const uint32_t tr = (DEFL_HEADER + S.payload) * 8;
    defl_put(o, tr, crc32_finish(S.crc_xor, S.n), 32);
    defl_put(o, tr + 32, S.n, 32);
}

// Thread t's share of the deflate data: its tokens at the scanned offset, or its bytes of the stored block.
FM_BGZF_HD void defl_emit(const DeflateShared &S, const DeflateBlock &B, uint32_t t, uint32_t nt) {
    uint32_t *o = B.slot;
    if (S.kind == DEFL_STORED) {
        for (uint32_t w = t; w * 4 < S.n; w += nt) {
            const uint32_t nb = S.n - w * 4 < 4 ? S.n - w * 4 : 4;
            defl_put(o, (DEFL_HEADER + 5 + w * 4) * 8, nb == 4 ? S.data[w] : S.data[w] & ((1u << (8 * nb)) - 1), 8 * nb);
        }
        return;
    }
    uint32_t p = DEFL_HEADER * 8 + S.hdr_bits + S.seg_bits[t];
    defl_tokens(S, B, t, [&](uint32_t, uint32_t lit, uint32_t L, uint32_t d) {
        if (lit != ~0u) {
            defl_put(o, p, S.code_lit[lit], S.len_lit[lit]);
            p += S.len_lit[lit];
            return;
        }
        uint32_t s, xb, xv;
        defl_len_code(L, s, xb, xv);
        defl_put(o, p, S.code_lit[s], S.len_lit[s]);
        p += S.len_lit[s];
        defl_put(o, p, xv, xb);
        p += xb;
        defl_dist_code(d, s, xb, xv);
        defl_put(o, p, S.code_dist[s], S.len_dist[s]);
        p += S.len_dist[s];
        defl_put(o, p, xv, xb);
        p += xb;
    });
}

// The serial CPU build of fm_k_deflate_members' block: the same phases, thread after thread.  Returns the member's
// size; B.slot receives it.
inline uint32_t deflate_block_serial(DeflateShared &S, const DeflateBlock &B) {
    const uint32_t nt = DEFL_THREADS;
    for (uint32_t t = 0; t < nt; ++t) defl_load(S, B, t, nt);
    for (uint32_t c = 0; c * nt < B.n; ++c) {
        for (uint32_t t = 0; t < nt; ++t) defl_match(S, B, c, t, nt);
        for (uint32_t t = 0; t < nt; ++t) defl_insert(S, B, c, t, nt);
    }
    defl_parse(S);
    for (uint32_t t = 0; t < nt; ++t) defl_histogram(S, B, t, nt);
    defl_partners(S, 0);
    defl_partners(S, 1);
    for (uint32_t s = 0; s < 288; ++s) defl_rank(S, 0, s);
    for (uint32_t s = 0; s < 32; ++s) defl_rank(S, 1, s);
    defl_build(S, 0, S.len_lit, S.code_lit);
    defl_build(S, 1, S.len_dist, S.code_dist);
    defl_tables(S);
    defl_partners(S, 2);
    for (uint32_t s = 0; s < 19; ++s) defl_rank(S, 2, s);
    defl_build(S, 2, S.len_cl, S.code_cl);
    defl_choose(S);
    for (uint32_t t = 0; t < nt; ++t) defl_token_bits(S, B, t, nt);
    uint32_t run = 0;  // exclusive scan of the token bits
    for (uint32_t t = 0; t < nt; ++t) {
        const uint32_t b = S.seg_bits[t];
        S.seg_bits[t] = run;
        run += b;
    }
    for (uint32_t t = 0; t < nt; ++t) defl_crc(S, t, nt);
    for (uint32_t t = 0; t < nt; ++t) defl_zero_slot(S, B, t, nt);
    defl_frame(S, B, run);
    for (uint32_t t = 0; t < nt; ++t) defl_emit(S, B, t, nt);
    return defl_member_bytes(S);
}

#ifdef __CUDACC__
// One CTA per block of DEFL_BLOCK input bytes: member b goes to slots + b * DEFL_SLOT / 4, its size to sizes[b].
// dist: DEFL_BLOCK u16 per member (match distances; too large for shared memory next to the block and the lengths,
// and read only at token starts after the parse).
__global__ void __launch_bounds__(DEFL_THREADS, 1)
fm_k_deflate_members(const uint8_t *__restrict__ in, uint64_t n, uint32_t *__restrict__ slots,
                     uint16_t *__restrict__ dist, uint32_t *__restrict__ sizes) {
    extern __shared__ uint4 defl_smem[];
    DeflateShared &S = *reinterpret_cast<DeflateShared *>(defl_smem);
    const uint32_t t = threadIdx.x, nt = DEFL_THREADS;
    const uint64_t b = blockIdx.x, off = b * DEFL_BLOCK;
    const DeflateBlock B{in + off, (uint32_t)(n - off < DEFL_BLOCK ? n - off : DEFL_BLOCK), slots + b * (DEFL_SLOT / 4),
                         dist + b * DEFL_BLOCK};
    defl_load(S, B, t, nt);
    __syncthreads();
    for (uint32_t c = 0; c * nt < B.n; ++c) {
        defl_match(S, B, c, t, nt);
        __syncthreads();
        defl_insert(S, B, c, t, nt);
        __syncthreads();
    }
    if (t == 0) defl_parse(S);
    __syncthreads();
    defl_histogram(S, B, t, nt);
    __syncthreads();
    if (t == 0) defl_partners(S, 0);
    if (t == 32) defl_partners(S, 1);
    __syncthreads();
    if (t < 288) defl_rank(S, 0, t);
    else if (t < 320) defl_rank(S, 1, t - 288);
    __syncthreads();
    if (t == 0) {  // the trees share defl_build's scratch
        defl_build(S, 0, S.len_lit, S.code_lit);
        defl_build(S, 1, S.len_dist, S.code_dist);
        defl_tables(S);
        defl_partners(S, 2);
    }
    __syncthreads();
    if (t < 19) defl_rank(S, 2, t);
    __syncthreads();
    if (t == 0) {
        defl_build(S, 2, S.len_cl, S.code_cl);
        defl_choose(S);
    }
    __syncthreads();
    defl_token_bits(S, B, t, nt);
    defl_crc(S, t, nt);
    __syncthreads();
    {  // exclusive scan of seg_bits
        const uint32_t v = S.seg_bits[t], lane = t & 31, w = t >> 5;
        uint32_t x = v;
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= (uint32_t)o) x += y;
        }
        if (lane == 31) S.wsum[w] = x;
        __syncthreads();
        if (t == 0) {
            uint32_t run = 0;
            for (uint32_t k = 0; k < nt / 32; ++k) {
                const uint32_t s = S.wsum[k];
                S.wsum[k] = run;
                run += s;
            }
        }
        __syncthreads();
        S.seg_bits[t] = S.wsum[w] + x - v;
        if (t == nt - 1) S.tok_bits = S.wsum[w] + x;
    }
    defl_zero_slot(S, B, t, nt);
    __syncthreads();
    if (t == 0) {
        defl_frame(S, B, S.tok_bits);
        sizes[b] = defl_member_bytes(S);
    }
    defl_emit(S, B, t, nt);
}

// Member b's bytes from its slot to out + offs[b] (offs: exclusive scan of sizes).
__global__ void __launch_bounds__(256)
fm_k_deflate_compact(const uint32_t *__restrict__ slots, const uint32_t *__restrict__ sizes,
                     const uint64_t *__restrict__ offs, uint8_t *__restrict__ out) {
    const uint64_t b = blockIdx.x;
    const uint8_t *src = reinterpret_cast<const uint8_t *>(slots + b * (DEFL_SLOT / 4));
    uint8_t *dst = out + offs[b];
    for (uint32_t i = threadIdx.x, n = sizes[b]; i < n; i += blockDim.x) dst[i] = src[i];
}
#endif

}  // namespace fm
