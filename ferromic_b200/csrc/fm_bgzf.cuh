// fm_bgzf.cuh -- BGZF inflate on the device (DESIGN §0 row f6).  A BGZF stream (what bgzip / tabix write) is a chain of
// independent gzip members of at most 64 KiB each; every member header carries its compressed size (the `BC` extra
// subfield) and its trailer the inflated size (ISIZE) and CRC32.  A host walk over the headers (bgzf_walk) therefore
// gives every member's input range and exact output offset before any decoding, and the members decode
// independently: fm_k_inflate_members runs one warp per member and writes straight to the member's offset.
//
// Decoding is full DEFLATE (RFC 1951): stored, fixed- and dynamic-Huffman blocks, several per member, codes up to 15
// bits, distances up to 32768 inside the member (BGZF members share no window).  All 32 lanes of the warp run the
// same bit reader and symbol decoder in lockstep (uniform loads from shared / global memory, no divergence), and lane
// j keeps the j-th token of a batch of 32.  The warp then writes the batch's literals at once and retires its
// back-references and stored runs in order, 32 bytes wide, because a match may read what an earlier token of the
// same batch wrote.  The CRC32 of the member is computed by the same warp from its output: a table CRC per lane
// slice, combined with the GF(2) shift operator (the math of zlib's crc32_combine).
//
// Malformed input comes from outside the program and must be rejected, never fault: every read of compressed bits
// is bounded by the member's end (reads past it yield zeros, and consuming them is an error), every table index is
// bounded, every write is bounded by ISIZE and every distance by the bytes already produced.  The bit reader, the
// table builder, the symbol decoder and the token checks are __host__ __device__ so a CPU build of the same code
// (tests/bgzf_host.cpp) runs under the sanitizers.
#pragma once
#include <stdint.h>

#include <vector>

#ifdef __CUDACC__
#include <cuda_runtime.h>
#define FM_BGZF_HD __host__ __device__ __forceinline__
#else
#define FM_BGZF_HD inline
#endif
#ifdef __CUDA_ARCH__
#define FM_BGZF_SYNCWARP() __syncwarp()
#else
#define FM_BGZF_SYNCWARP() ((void)0)
#endif

namespace fm {

// per-member error codes (device array, reported once with the first bad member)
enum : int32_t {
    BGZF_OK = 0,
    BGZF_E_TRUNCATED = 1,     // the deflate data ends before the final block does
    BGZF_E_BLOCK_TYPE = 2,    // block type 3
    BGZF_E_STORED_LEN = 3,    // stored block LEN != ~NLEN
    BGZF_E_CODE_LENGTHS = 4,  // over-subscribed / incomplete code, bad repeat, too many symbols, no end-of-block code
    BGZF_E_SYMBOL = 5,        // a bit pattern that is no code, or litlen 286/287, distance 30/31
    BGZF_E_DISTANCE = 6,      // a distance beyond the bytes produced
    BGZF_E_OVERFLOW = 7,      // more output than ISIZE
    BGZF_E_SIZE = 8,          // less output than ISIZE
    BGZF_E_CRC = 9,           // CRC32 differs from the trailer
    BGZF_E_TRAILING = 10,     // bytes left between the final block and the trailer
};

inline const char *bgzf_error_text(int32_t e) {
    switch (e) {
        case BGZF_E_TRUNCATED: return "deflate data truncated";
        case BGZF_E_BLOCK_TYPE: return "invalid deflate block type 3";
        case BGZF_E_STORED_LEN: return "stored block length does not match its complement";
        case BGZF_E_CODE_LENGTHS: return "invalid Huffman code lengths";
        case BGZF_E_SYMBOL: return "invalid Huffman code";
        case BGZF_E_DISTANCE: return "back-reference distance beyond the bytes produced";
        case BGZF_E_OVERFLOW: return "inflated data longer than ISIZE";
        case BGZF_E_SIZE: return "inflated data shorter than ISIZE";
        case BGZF_E_CRC: return "CRC32 mismatch";
        case BGZF_E_TRAILING: return "bytes between the final deflate block and the trailer";
        default: return "unknown error";
    }
}

struct BgzfMember {
    uint64_t off;      // first byte of the member in the stream
    uint64_t in_off;   // first byte of the member's deflate data in the stream
    uint64_t out_off;  // first inflated byte (exclusive scan of ISIZE)
    uint32_t in_len;   // deflate data bytes (BSIZE + 1 - header - 8-byte trailer)
    uint32_t isize;
    uint32_t crc;
    uint32_t pad;
};

// ------------------------------------------------------------------------------------------- host member walk
enum : int { BGZF_WALK_OK = 0, BGZF_WALK_PARSE = 1, BGZF_WALK_NOT_BGZF = 2 };
struct BgzfWalkError {
    int kind = BGZF_WALK_OK;
    uint64_t member = 0, offset = 0;
    const char *what = "";
};

// Checks every member header of gz[0, n) and appends the members to `mem` in stream order; returns the error of the
// first bad member (kind BGZF_WALK_OK when the stream is well formed).  The empty EOF member (ISIZE 0) is legal
// anywhere.
inline BgzfWalkError bgzf_walk(const uint8_t *gz, uint64_t n, std::vector<BgzfMember> &mem) {
    auto le16 = [&](uint64_t o) { return (uint32_t)gz[o] | (uint32_t)gz[o + 1] << 8; };
    auto le32 = [&](uint64_t o) { return le16(o) | le16(o + 2) << 16; };
    BgzfWalkError e;
    uint64_t off = 0, out = 0, idx = 0;
    auto bad = [&](int kind, const char *what) {
        e.kind = kind;
        e.member = idx;
        e.offset = off;
        e.what = what;
        return e;
    };
    while (off < n) {
        const uint64_t rem = n - off;
        if (rem < 2 || gz[off] != 0x1f || gz[off + 1] != 0x8b) return bad(BGZF_WALK_PARSE, "not a gzip member");
        if (rem < 18) return bad(BGZF_WALK_PARSE, "truncated member header");
        if (gz[off + 2] != 8) return bad(BGZF_WALK_PARSE, "compression method is not deflate");
        const uint32_t flg = gz[off + 3];
        if (flg & 0xe0) return bad(BGZF_WALK_PARSE, "reserved header flag set");
        if (!(flg & 4) || (flg & 0x1a)) return bad(BGZF_WALK_NOT_BGZF, "gzip member without the BGZF header");
        const uint64_t xlen = le16(off + 10);
        if (12 + xlen > rem) return bad(BGZF_WALK_PARSE, "truncated member header");
        int64_t bsize = -1;
        for (uint64_t p = off + 12, end = off + 12 + xlen; p < end;) {
            if (end - p < 4) return bad(BGZF_WALK_PARSE, "malformed extra field");
            const uint64_t slen = le16(p + 2);
            if (end - p - 4 < slen) return bad(BGZF_WALK_PARSE, "malformed extra field");
            if (gz[p] == 66 && gz[p + 1] == 67 && slen == 2) bsize = le16(p + 4);
            p += 4 + slen;
        }
        if (bsize < 0) return bad(BGZF_WALK_NOT_BGZF, "gzip member without the BGZF header");
        const uint64_t bs = (uint64_t)bsize + 1;
        if (bs < 12 + xlen + 8) return bad(BGZF_WALK_PARSE, "BSIZE smaller than the member's header and trailer");
        if (bs > rem) return bad(BGZF_WALK_PARSE, "member extends past the end of the stream (truncated)");
        const uint32_t isize = le32(off + bs - 4);
        if (isize > 65536) return bad(BGZF_WALK_PARSE, "ISIZE above 65536");
        mem.push_back(BgzfMember{off, off + 12 + xlen, out, (uint32_t)(bs - 12 - xlen - 8), isize, le32(off + bs - 8), 0});
        out += isize;
        off += bs;
        ++idx;
    }
    return e;
}

// --------------------------------------------------------------------------------------------------- CRC32
FM_BGZF_HD uint32_t crc32_table_entry(uint32_t i) {
    uint32_t c = i;
    for (int k = 0; k < 8; ++k) c = (c & 1) ? (c >> 1) ^ 0xedb88320u : c >> 1;
    return c;
}
// a * b modulo the CRC polynomial, reflected (zlib's multmodp); x^0 is 1 << 31
FM_BGZF_HD uint32_t crc32_mulmodp(uint32_t a, uint32_t b) {
    uint32_t p = 0;
    for (int i = 0; i < 32; ++i) {
        if (a & (0x80000000u >> i)) p ^= b;
        b = (b & 1) ? (b >> 1) ^ 0xedb88320u : b >> 1;
    }
    return p;
}
// x^(8 n) modulo the polynomial: the operator that moves a CRC register over n zero bytes
FM_BGZF_HD uint32_t crc32_x8n(uint64_t n) {
    uint32_t r = 1u << 31, sq = 1u << 23;  // x^0, x^8
    for (; n; n >>= 1) {
        if (n & 1) r = crc32_mulmodp(sq, r);
        sq = crc32_mulmodp(sq, sq);
    }
    return r;
}
// raw register over data from a zero register (no pre/post inversion)
FM_BGZF_HD uint32_t crc32_raw(const uint32_t *tab, const uint8_t *p, uint32_t n) {
    uint32_t r = 0;
    for (uint32_t i = 0; i < n; ++i) r = tab[(r ^ p[i]) & 0xffu] ^ (r >> 8);
    return r;
}
// The CRC32 of n bytes from the raw registers of its slices: slice k of `lanes` covers [k*len, min((k+1)*len, n)).
// crc = ~(init shifted over n bytes  ^  XOR_k raw_k shifted over the bytes after slice k)
FM_BGZF_HD uint32_t crc32_slice_term(uint32_t raw, uint32_t slice_end, uint32_t n) {
    return crc32_mulmodp(crc32_x8n(n - slice_end), raw);
}
FM_BGZF_HD uint32_t crc32_finish(uint32_t xor_of_terms, uint32_t n) {
    return ~(crc32_mulmodp(crc32_x8n(n), 0xffffffffu) ^ xor_of_terms);
}

// --------------------------------------------------------------------------------------------------- DEFLATE
struct InflateBits {
    const uint8_t *p;
    uint32_t n;    // bytes of deflate data
    uint32_t pos;  // next byte to load (may pass n: those loads read zero)
    uint64_t buf;  // pending bits, LSB first
    uint32_t cnt;  // bits in buf
};
// After a refill buf holds >= 57 bits: enough for the longest token (15 + 5 + 15 + 13 bits).
FM_BGZF_HD void bits_refill(InflateBits &b) {
    while (b.cnt <= 56) {
        const uint64_t v = b.pos < b.n ? b.p[b.pos] : 0u;
        ++b.pos;
        b.buf |= v << b.cnt;
        b.cnt += 8;
    }
}
FM_BGZF_HD uint32_t bits_take(InflateBits &b, uint32_t k) {  // k <= cnt
    const uint32_t v = (uint32_t)(b.buf & ((1ull << k) - 1));
    b.buf >>= k;
    b.cnt -= k;
    return v;
}
FM_BGZF_HD uint64_t bits_consumed(const InflateBits &b) { return (uint64_t)b.pos * 8 - b.cnt; }
FM_BGZF_HD bool bits_overrun(const InflateBits &b) { return bits_consumed(b) > (uint64_t)b.n * 8; }

// Canonical Huffman table: a FAST-bit first-level table (entry = symbol | length << 9, 0 = not in the table) and the
// per-length counts with the symbols sorted by (length, symbol) for the codes longer than FAST bits.
template <int FAST, int NSYM>
struct HuffTable {
    uint16_t fast[1 << FAST];
    uint16_t count[16];
    uint16_t sym[NSYM];
};
constexpr int LIT_FAST = 10, DIST_FAST = 8, CL_FAST = 7;
struct InflateTables {
    HuffTable<LIT_FAST, 288> lit;
    HuffTable<DIST_FAST, 32> dist;
    HuffTable<CL_FAST, 19> cl;
    uint8_t lens[288 + 32];
};

// Builds t from len[0, n) (each <= 15).  Lanes `lane` of `nlanes` share the fills; every lane returns the same
// status.  Over-subscribed sets are rejected, incomplete ones too unless the longest code has 1 bit (a single
// distance code) or `complete_only`; an all-zero set builds an empty table whose every lookup fails.
template <int FAST, int NSYM>
FM_BGZF_HD int huff_build(HuffTable<FAST, NSYM> &t, const uint8_t *len, int n, bool complete_only, int lane,
                                 int nlanes) {
    int cnt[16] = {0};
    for (int s = 0; s < n; ++s) cnt[len[s] & 15]++;
    cnt[0] = 0;
    int left = 1, maxlen = 0;
    for (int L = 1; L <= 15; ++L) {
        left = (left << 1) - cnt[L];
        if (left < 0) return BGZF_E_CODE_LENGTHS;
        if (cnt[L]) maxlen = L;
    }
    if (left > 0 && maxlen > 0 && (complete_only || maxlen > 1)) return BGZF_E_CODE_LENGTHS;
    FM_BGZF_SYNCWARP();  // every lane is done with the previous table
    int offs[16], first[16], code = 0, total = 0;
    for (int L = 1; L <= 15; ++L) {
        offs[L] = total;
        total += cnt[L];
        code = (code + cnt[L - 1]) << 1;
        first[L] = code;
        if (lane == 0) t.count[L] = (uint16_t)cnt[L];
    }
    if (lane == 0) {
        t.count[0] = 0;
        int o[16];
        for (int L = 0; L < 16; ++L) o[L] = offs[L];
        for (int s = 0; s < n; ++s)
            if (len[s]) t.sym[o[len[s]]++] = (uint16_t)s;
    }
    for (int i = lane; i < (1 << FAST); i += nlanes) t.fast[i] = 0;
    FM_BGZF_SYNCWARP();
    for (int i = lane; i < total; i += nlanes) {
        int L = 1;
        while (L < 15 && i >= offs[L] + cnt[L]) ++L;
        if (L > FAST) break;  // sorted by length: the rest are longer too
        uint32_t c = (uint32_t)(first[L] + (i - offs[L])), r = 0;
        for (int k = 0; k < L; ++k) r |= ((c >> k) & 1u) << (L - 1 - k);
        const uint16_t e = (uint16_t)(t.sym[i] | L << 9);
        for (uint32_t k = r; k < (1u << FAST); k += 1u << L) t.fast[k] = e;
    }
    FM_BGZF_SYNCWARP();
    return BGZF_OK;
}

// Next symbol (buf holds >= 15 bits), or -1 for a bit pattern that is no code.
template <int FAST, int NSYM>
FM_BGZF_HD int huff_decode(const HuffTable<FAST, NSYM> &t, InflateBits &b) {
    const uint32_t e = t.fast[b.buf & ((1u << FAST) - 1)];
    if (e) {
        bits_take(b, e >> 9);
        return (int)(e & 511u);
    }
    int code = 0, first = 0, index = 0;
    uint64_t bb = b.buf;
    for (int L = 1; L <= 15; ++L) {
        code |= (int)(bb & 1);
        bb >>= 1;
        const int c = t.count[L];
        if (code - c < first) {
            bits_take(b, L);
            return t.sym[index + (code - first)];  // < sum of counts <= NSYM
        }
        index += c;
        first = (first + c) << 1;
        code <<= 1;
    }
    return -1;
}

enum : uint32_t { TK_LIT = 0, TK_MATCH = 1, TK_STORED = 2, TK_END = 3, TK_ERR = 4 };
struct InflateToken {
    uint32_t kind;
    uint32_t pos;  // output offset in the member
    uint32_t len;  // match / stored length
    uint32_t a;    // literal byte, match distance, or stored run's input offset
};
enum : uint32_t { INF_HEADER = 0, INF_HUFF = 1, INF_DONE = 2 };
struct InflateState {
    InflateBits b;
    uint32_t out;    // bytes produced
    uint32_t isize;  // bytes the member must produce
    uint32_t mode;
    uint32_t last;   // the current block is the final one
    int32_t err;
};
FM_BGZF_HD void inflate_init(InflateState &s, const uint8_t *p, uint32_t n, uint32_t isize) {
    s.b = InflateBits{p, n, 0, 0, 0};
    s.out = 0;
    s.isize = isize;
    s.mode = INF_HEADER;
    s.last = 0;
    s.err = BGZF_OK;
}

// The next token of the member.  Every write it implies lies in [0, isize) and every match reads only bytes already
// produced; TK_END means the member decoded to exactly isize bytes and the final block ends at the data's last byte.
FM_BGZF_HD InflateToken inflate_next(InflateState &s, InflateTables &T, int lane, int nlanes) {
    auto fail = [&](int32_t e) {
        s.err = e;
        s.mode = INF_DONE;
        return InflateToken{TK_ERR, s.out, 0, 0};
    };
    InflateBits &b = s.b;
    for (;;) {
        if (s.mode == INF_DONE) return InflateToken{s.err ? TK_ERR : TK_END, s.out, 0, 0};
        bits_refill(b);
        if (bits_overrun(b)) return fail(BGZF_E_TRUNCATED);
        if (s.mode == INF_HEADER) {
            if (s.last) {
                if ((bits_consumed(b) + 7) / 8 != b.n) return fail(BGZF_E_TRAILING);
                if (s.out != s.isize) return fail(BGZF_E_SIZE);
                s.mode = INF_DONE;
                continue;
            }
            s.last = bits_take(b, 1);
            const uint32_t type = bits_take(b, 2);
            if (type == 0) {
                bits_take(b, b.cnt & 7u);  // to the byte boundary
                const uint32_t len = bits_take(b, 16), nlen = bits_take(b, 16);
                if (len != (~nlen & 0xffffu)) return fail(BGZF_E_STORED_LEN);
                const uint32_t at = b.pos - b.cnt / 8;  // first stored byte
                if (bits_overrun(b) || (uint64_t)at + len > b.n) return fail(BGZF_E_TRUNCATED);
                if ((uint64_t)s.out + len > s.isize) return fail(BGZF_E_OVERFLOW);
                b.pos = at + len;
                b.buf = 0;
                b.cnt = 0;
                if (!len) continue;
                const InflateToken t{TK_STORED, s.out, len, at};
                s.out += len;
                return t;
            }
            if (type == 3) return fail(BGZF_E_BLOCK_TYPE);
            int e;
            if (type == 1) {
                for (int i = 0; i < 288; ++i) T.lens[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : 8;
                for (int i = 0; i < 32; ++i) T.lens[288 + i] = 5;
                e = huff_build(T.lit, T.lens, 288, false, lane, nlanes);
                if (!e) e = huff_build(T.dist, T.lens + 288, 32, false, lane, nlanes);
            } else {
                const uint32_t nlen = bits_take(b, 5) + 257, ndist = bits_take(b, 5) + 1, ncl = bits_take(b, 4) + 4;
                if (nlen > 286 || ndist > 30) return fail(BGZF_E_CODE_LENGTHS);
                uint8_t cl[19] = {0};
                const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
                for (uint32_t i = 0; i < ncl; ++i) {
                    bits_refill(b);
                    cl[order[i]] = (uint8_t)bits_take(b, 3);
                }
                e = huff_build(T.cl, cl, 19, true, lane, nlanes);
                uint32_t i = 0;
                while (!e && i < nlen + ndist) {
                    bits_refill(b);
                    const int sym = huff_decode(T.cl, b);
                    if (sym < 0) {
                        e = BGZF_E_SYMBOL;
                    } else if (sym < 16) {
                        T.lens[i++] = (uint8_t)sym;
                    } else {
                        uint32_t rep;
                        uint8_t v = 0;
                        if (sym == 16) {
                            if (i == 0) {
                                e = BGZF_E_CODE_LENGTHS;
                                break;
                            }
                            v = T.lens[i - 1];
                            rep = 3 + bits_take(b, 2);
                        } else {
                            rep = sym == 17 ? 3 + bits_take(b, 3) : 11 + bits_take(b, 7);
                        }
                        if (i + rep > nlen + ndist) {
                            e = BGZF_E_CODE_LENGTHS;
                            break;
                        }
                        while (rep--) T.lens[i++] = v;
                    }
                }
                if (!e && bits_overrun(b)) e = BGZF_E_TRUNCATED;
                if (!e && T.lens[256] == 0) e = BGZF_E_CODE_LENGTHS;  // no end-of-block code
                if (!e) e = huff_build(T.lit, T.lens, (int)nlen, false, lane, nlanes);
                if (!e) e = huff_build(T.dist, T.lens + nlen, (int)ndist, false, lane, nlanes);
            }
            if (e) return fail(e);
            s.mode = INF_HUFF;
            continue;
        }
        // INF_HUFF: one literal, the end of the block, or one match
        const int sym = huff_decode(T.lit, b);
        if (sym < 0 || sym > 285) return fail(BGZF_E_SYMBOL);
        if (sym < 256) {
            if (s.out >= s.isize) return fail(BGZF_E_OVERFLOW);
            return InflateToken{TK_LIT, s.out++, 1, (uint32_t)sym};
        }
        if (sym == 256) {
            s.mode = INF_HEADER;
            continue;
        }
        const uint32_t i = (uint32_t)sym - 257;
        uint32_t len;
        if (i < 8) len = 3 + i;
        else if (i == 28) len = 258;
        else {
            const uint32_t x = (i - 4) >> 2;
            len = ((4 + (i & 3)) << x) + 3 + bits_take(b, x);
        }
        const int d = huff_decode(T.dist, b);
        if (d < 0 || d > 29) return fail(BGZF_E_SYMBOL);
        uint32_t dist;
        if (d < 4) dist = 1 + (uint32_t)d;
        else {
            const uint32_t x = ((uint32_t)d - 2) >> 1;
            dist = ((2 + ((uint32_t)d & 1)) << x) + 1 + bits_take(b, x);
        }
        if (bits_overrun(b)) return fail(BGZF_E_TRUNCATED);
        if (dist > s.out) return fail(BGZF_E_DISTANCE);
        if ((uint64_t)s.out + len > s.isize) return fail(BGZF_E_OVERFLOW);
        const InflateToken t{TK_MATCH, s.out, len, dist};
        s.out += len;
        return t;
    }
}

#ifdef __CUDACC__
constexpr int INFLATE_WARPS = 4;  // members per block

// One warp per member of mem[0, n_mem): inflate member m to out + (mem[m].out_off - out_base) and check its length
// and CRC32.  A bad member stores its code in err[m] and lowers *first_bad to m.  80 registers: ptxas's own choice
// (56) spills the decoder state.
__global__ void __maxnreg__(80)
fm_k_inflate_members(const uint8_t *__restrict__ in, const BgzfMember *__restrict__ mem, uint32_t n_mem,
                     uint8_t *__restrict__ out, uint64_t out_base, int32_t *__restrict__ err,
                     uint32_t *__restrict__ first_bad) {
    __shared__ uint32_t crc_tab[256];
    __shared__ InflateTables tabs[INFLATE_WARPS];
    for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) crc_tab[i] = crc32_table_entry(i);
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31, w = threadIdx.x >> 5, m = blockIdx.x * INFLATE_WARPS + w;
    if (m >= n_mem) return;
    const BgzfMember M = mem[m];
    InflateTables &T = tabs[w];
    uint8_t *dst = out + (M.out_off - out_base);
    InflateState s;
    inflate_init(s, in + M.in_off, M.in_len, M.isize);
    for (;;) {
        InflateToken mine{TK_END, 0, 0, 0};
        uint32_t nt = 0;
        bool end = false;
        while (nt < 32) {
            const InflateToken t = inflate_next(s, T, (int)lane, 32);
            if (t.kind >= TK_END) {
                end = true;
                break;
            }
            if (lane == nt) mine = t;
            ++nt;
        }
        if (mine.kind == TK_LIT) dst[mine.pos] = (uint8_t)mine.a;
        __syncwarp();
        for (uint32_t j = 0; j < nt; ++j) {
            const uint32_t kind = __shfl_sync(0xffffffffu, mine.kind, j);
            if (kind == TK_LIT) continue;
            const uint32_t pos = __shfl_sync(0xffffffffu, mine.pos, j), len = __shfl_sync(0xffffffffu, mine.len, j),
                           a = __shfl_sync(0xffffffffu, mine.a, j);
            if (kind == TK_STORED) {
                for (uint32_t k = lane; k < len; k += 32) dst[pos + k] = s.b.p[a + k];
            } else {  // out[p+k] = out[p-dist + k % dist]: every source byte precedes the match
                for (uint32_t k = lane; k < len; k += 32) dst[pos + k] = dst[pos - a + (k < a ? k : k % a)];
            }
            __syncwarp();
        }
        if (end) break;
    }
    int32_t code = s.err;
    if (code == BGZF_OK) {
        const uint32_t n = M.isize, per = (n + 31) / 32, b0 = min(lane * per, n), b1 = min(b0 + per, n);
        uint32_t term = crc32_slice_term(crc32_raw(crc_tab, dst + b0, b1 - b0), b1, n);
        for (int o = 16; o; o >>= 1) term ^= __shfl_xor_sync(0xffffffffu, term, o);
        if (crc32_finish(term, n) != M.crc) code = BGZF_E_CRC;
    }
    if (code != BGZF_OK && lane == 0) {
        err[m] = code;
        atomicMin(first_bad, m);
    }
}

// Last '\n' of text[0, n) as index + 1 (0: none) into res[0] (zeroed by the caller); res[1] = text[n - 1].
__global__ void __launch_bounds__(256)
fm_k_text_tail(const uint8_t *__restrict__ text, uint32_t n, uint32_t *__restrict__ res) {
    uint32_t best = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        if (text[i] == '\n') best = i + 1;
    for (int o = 16; o; o >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, o));
    if ((threadIdx.x & 31) == 0 && best) atomicMax(res, best);
    if (blockIdx.x == 0 && threadIdx.x == 0) res[1] = n ? text[n - 1] : 0u;
}
#endif

}  // namespace fm
