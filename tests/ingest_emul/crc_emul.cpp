// TEST SIDE: the BGZF CRC-32 of the device ingest (metamlst_b200/csrc/bgzf_crc.cuh) compiled for the host and driven the way
// csrc/ingest.cu's crc_kernel drives it: kCrcThreads segments of one frame, combined level by level in the order of the warp
// shuffles and the cross-warp step, then compared against the trailer value.  Checked against zlib by tests/test_ingest_crc.py.
#include <cstdint>
#include <cstring>
#include <vector>

#include "bgzf_crc.cuh"

using namespace bgzf_crc;

namespace {

struct Tables {
    uint32_t T[8][256];
    uint32_t O[kCrcLevels][4][256];
    std::vector<uint32_t> zeros;
    Tables() : zeros(65536 + 16) {
        for (uint32_t v = 0; v < 256; ++v) T[0][v] = t0_entry(v);
        for (int k = 1; k < 8; ++k)
            for (uint32_t v = 0; v < 256; ++v) T[k][v] = zero_byte(T[k - 1][v], T[0]);
        uint32_t ops[kCrcLevels][32];
        make_ops(ops);
        for (uint32_t k = 0; k < kCrcLevels; ++k)
            for (uint32_t j = 0; j < 4; ++j)
                for (uint32_t v = 0; v < 256; ++v) O[k][j][v] = op_entry(ops[k], j, v);
        make_zeros(zeros.data(), 65536 + 15);   // + 15: emul_frame_crc32 converts block || 0^z
    }
};
const Tables& tables() { static const Tables t; return t; }

uint32_t frame_raw(const uint8_t* blk, uint32_t n) {
    const Tables& tb = tables();
    uint32_t r[kCrcThreads];
    for (uint32_t t = 0; t < kCrcThreads; ++t) r[t] = segment(blk, n, t, tb.T);
    for (uint32_t k = 0; k < kCrcLevels; ++k) {
        const uint32_t d = 1u << k;
        for (uint32_t t = 0; t + d < kCrcThreads; t += 2 * d) r[t] = shift(r[t], tb.O[k]) ^ r[t + d];
    }
    return r[0];
}

}  // namespace

extern "C" {

// zlib.crc32(block || 0^z) as the kernel's frame gives it, with z = zero bytes between the block's end and the frame's; the block is
// copied to `mis` bytes past a 16-byte boundary first (mis = 0 .. 15).
uint32_t emul_frame_crc32(const uint8_t* p, uint32_t n, uint32_t mis, uint32_t* z) {
    std::vector<uint8_t> buf(static_cast<size_t>(n) + 64 + 16);
    uint8_t* base = buf.data() + ((16 - reinterpret_cast<uintptr_t>(buf.data()) % 16) % 16);
    memset(base, 0xa5, static_cast<size_t>(n) + 48);   // bytes around the block are not zero: they must be masked
    memcpy(base + mis, p, n);
    const uint64_t a = reinterpret_cast<uintptr_t>(base + mis);
    *z = static_cast<uint32_t>(frame_end(a, n) - (a + n));
    return frame_raw(base + mis, n) ^ tables().zeros[n + *z];
}

// 1 when the kernel's comparison accepts `trailer` (zlib convention) as the CRC of the block placed `mis` bytes past a 16-byte boundary.
int emul_check(const uint8_t* p, uint32_t n, uint32_t mis, uint32_t trailer) {
    std::vector<uint8_t> buf(static_cast<size_t>(n) + 64 + 16);
    uint8_t* base = buf.data() + ((16 - reinterpret_cast<uintptr_t>(buf.data()) % 16) % 16);
    memset(base, 0x5a, static_cast<size_t>(n) + 48);
    memcpy(base + mis, p, n);
    return matches(frame_raw(base + mis, n), trailer ^ tables().zeros[n], base + mis, n, tables().T[0]) ? 1 : 0;
}

// Raw CRC (initial value 0, no final xor) one byte at a time, and crc32(0^n): the two identities the kernel rests on.
uint32_t emul_raw(const uint8_t* p, uint32_t n) {
    uint32_t c = 0;
    for (uint32_t i = 0; i < n; ++i) c = step1(c, p[i], tables().T[0]);
    return c;
}
uint32_t emul_zeros(uint32_t n) { return tables().zeros[n]; }

}
