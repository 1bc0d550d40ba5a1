// CPU harness of the BGZF encoder (ferromic_b200/csrc/fm_deflate.cuh): deflate_block_serial runs the phases of
// fm_k_deflate_members thread after thread, so its members are the device's bytes, here under AddressSanitizer and
// UBSan.  The decoder harness (bgzf_host.cpp) is built into the same object, so a test can compress with the
// project's encoder and inflate with the project's decoder.  Test infrastructure, built by tests/bgzf_deflate_host.py.
#include "bgzf_host.cpp"
#include "../ferromic_b200/csrc/fm_deflate.cuh"

extern "C" {

// BGZF members of in[0, n) (+ the 28-byte EOF member when eof) into out[0, min(capacity, total)); *total = the
// stream's size.  Returns 0.
int bh_deflate(const uint8_t *in, size_t n, int eof, uint8_t *out, size_t capacity, uint64_t *total) {
    static const uint8_t kEof[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 0x42, 0x43, 2, 0,
                                     0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    auto S = std::make_unique<fm::DeflateShared>();
    std::vector<uint32_t> slot(fm::DEFL_SLOT / 4);
    std::vector<uint16_t> dist(fm::DEFL_BLOCK);
    uint64_t o = 0;
    auto put = [&](const uint8_t *p, size_t k) {
        if (o < capacity) std::memcpy(out + o, p, std::min<uint64_t>(k, capacity - o));
        o += k;
    };
    for (size_t off = 0; off < n; off += fm::DEFL_BLOCK) {
        const uint32_t m = (uint32_t)std::min<size_t>(fm::DEFL_BLOCK, n - off);
        std::vector<uint8_t> blk(in + off, in + off + m);  // exact extent: reads past it are caught
        const fm::DeflateBlock B{blk.data(), m, slot.data(), dist.data()};
        const uint32_t size = fm::deflate_block_serial(*S, B);
        put(reinterpret_cast<const uint8_t *>(slot.data()), size);
    }
    if (eof) put(kEof, sizeof(kEof));
    *total = o;
    return 0;
}

// The member walk of fm_bgzf.cuh over gz[0, n): 0, or 100 + the walk's error kind.  *n_members = members found.
int bh_walk(const uint8_t *gz, size_t n, uint64_t *n_members) {
    std::vector<fm::BgzfMember> mem;
    const fm::BgzfWalkError e = fm::bgzf_walk(gz, n, mem);
    *n_members = mem.size();
    return e.kind == fm::BGZF_WALK_OK ? 0 : 100 + e.kind;
}
}
