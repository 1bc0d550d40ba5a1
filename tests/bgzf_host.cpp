// CPU harness of the BGZF decoder (ferromic_b200/csrc/fm_bgzf.cuh): the member walk, the bit reader, the table
// builder, the symbol decoder and the token checks that fm_k_inflate_members runs, driven serially on the host so
// AddressSanitizer and UBSan watch every access.  Test infrastructure, built by tests/bgzf_host.py.
#include "../ferromic_b200/csrc/fm_bgzf.cuh"

#include <algorithm>
#include <cstring>
#include <memory>
#include <vector>

extern "C" {

// Inflates the whole stream into out[0, min(capacity, total)).  Returns 0, 100 + walk error kind, or the first bad
// member's BGZF_E_* code; *bad_member is that member's index (-1 when none).
int bh_inflate(const uint8_t *gz, size_t n, uint8_t *out, size_t capacity, uint64_t *total, int64_t *bad_member) {
    std::vector<fm::BgzfMember> mem;
    *bad_member = -1;
    *total = 0;
    const fm::BgzfWalkError we = fm::bgzf_walk(gz, n, mem);
    if (we.kind != fm::BGZF_WALK_OK) {
        *bad_member = (int64_t)we.member;
        return 100 + we.kind;
    }
    for (auto &m : mem) *total += m.isize;
    uint32_t tab[256];
    for (uint32_t i = 0; i < 256; ++i) tab[i] = fm::crc32_table_entry(i);
    auto T = std::make_unique<fm::InflateTables>();
    for (size_t k = 0; k < mem.size(); ++k) {
        const fm::BgzfMember &M = mem[k];
        std::vector<uint8_t> in(gz + M.in_off, gz + M.in_off + M.in_len);  // exact extent: reads past it are caught
        std::unique_ptr<uint8_t[]> dst(new uint8_t[M.isize ? M.isize : 1]);
        fm::InflateState s;
        fm::inflate_init(s, in.data(), M.in_len, M.isize);
        for (;;) {
            const fm::InflateToken t = fm::inflate_next(s, *T, 0, 1);
            if (t.kind >= fm::TK_END) break;
            if (t.kind == fm::TK_LIT) dst[t.pos] = (uint8_t)t.a;
            else if (t.kind == fm::TK_STORED) std::memcpy(&dst[t.pos], &in[t.a], t.len);
            else
                for (uint32_t i = 0; i < t.len; ++i) dst[t.pos + i] = dst[t.pos - t.a + (i < t.a ? i : i % t.a)];
        }
        int code = s.err;
        if (code == fm::BGZF_OK) {  // the device's 32 lane slices, combined the same way
            const uint32_t per = (M.isize + 31) / 32;
            uint32_t term = 0;
            for (uint32_t lane = 0; lane < 32; ++lane) {
                const uint32_t b0 = std::min(lane * per, M.isize), b1 = std::min(b0 + per, M.isize);
                term ^= fm::crc32_slice_term(fm::crc32_raw(tab, dst.get() + b0, b1 - b0), b1, M.isize);
            }
            if (fm::crc32_finish(term, M.isize) != M.crc) code = fm::BGZF_E_CRC;
        }
        if (code != fm::BGZF_OK) {
            *bad_member = (int64_t)k;
            return code;
        }
        if (M.out_off < capacity)
            std::memcpy(out + M.out_off, dst.get(), std::min<uint64_t>(M.isize, capacity - M.out_off));
    }
    return 0;
}
}
