// CRC-32 (zlib's: reflected polynomial 0xEDB88320) of the inflated BGZF blocks of the DEVICE ingest (csrc/ingest.cu, crc_kernel),
// written as host/device inline functions so that the same text runs in the kernel and -- compiled by g++ in tests/ingest_emul --
// on the host against zlib before a GPU ever sees it.
//
// Everything works on RAW CRCs (initial value 0, no final xor), which are linear over GF(2):
//   raw(A || B) = shift_|B|(raw(A)) ^ raw(B),   shift_L = L zero-byte steps, a constant 32x32 matrix for a fixed L;
//   raw(0^k || M) = raw(M)                     (leading zero bytes leave a zero register at zero);
//   raw(M) = crc32(M) ^ crc32(0^|M|)           (zlib's trailer value -> the raw value to compare against: make_zeros).
// A block of n <= 65536 bytes at an arbitrary address A is checked as one FRAME of kCrcThreads segments of kCrcSeg bytes each, whose
// end FE is A + n rounded up to 16 bytes: every segment starts 16-byte aligned, bytes before A read as zero (neutral), and the z = FE -
// (A + n) < 16 bytes after the block read as zero too, so the frame's raw CRC is shift_z(raw(M)).  Segment t's raw CRC comes from
// slice-by-8 tables; the frame's is the tree  r_t = shift_{kCrcSeg * 2^k}(r_t) ^ r_{t + 2^k},  k = 0 .. 7, one constant operator per
// level, each applied as four byte-table lookups.
#pragma once
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define CRC_HD __host__ __device__ __forceinline__
#define CRC_UNROLL _Pragma("unroll")
#else
#define CRC_HD inline
#define CRC_UNROLL
#endif

namespace bgzf_crc {

constexpr uint32_t kPoly = 0xEDB88320u;
constexpr uint32_t kCrcThreads = 256;                     // segments per frame (= threads of the kernel's CTA)
constexpr uint32_t kCrcLevels = 8;                        // log2(kCrcThreads): combine operators
constexpr uint32_t kCrcSeg = 272;                         // bytes per segment: 17 x 16, so that 65536 + 15 bytes fit in one frame
constexpr uint64_t kCrcFrame = static_cast<uint64_t>(kCrcThreads) * kCrcSeg;
static_assert(kCrcFrame >= 65536 + 15, "a frame holds the largest BGZF block at any alignment");

// ---- tables ---------------------------------------------------------------------------------------------------------------
// T[0] is the classic byte table; T[k][v] = raw CRC of byte v followed by k zero bytes (slice-by-8).
CRC_HD uint32_t t0_entry(uint32_t v) {
    uint32_t c = v;
    for (int i = 0; i < 8; ++i) c = (c & 1u) ? (c >> 1) ^ kPoly : (c >> 1);
    return c;
}
CRC_HD uint32_t zero_byte(uint32_t c, const uint32_t* t0) { return (c >> 8) ^ t0[c & 0xffu]; }

// One byte / eight bytes (little-endian words a = bytes 0..3, b = bytes 4..7) into a raw register.
CRC_HD uint32_t step1(uint32_t c, uint8_t byte, const uint32_t* t0) { return (c >> 8) ^ t0[(c ^ byte) & 0xffu]; }
CRC_HD uint32_t step8(uint32_t c, uint32_t a, uint32_t b, const uint32_t (*T)[256]) {
    c ^= a;
    return T[7][c & 0xffu] ^ T[6][(c >> 8) & 0xffu] ^ T[5][(c >> 16) & 0xffu] ^ T[4][c >> 24] ^
           T[3][b & 0xffu] ^ T[2][(b >> 8) & 0xffu] ^ T[1][(b >> 16) & 0xffu] ^ T[0][b >> 24];
}

// ---- GF(2) operators ------------------------------------------------------------------------------------------------------
// A 32x32 matrix is 32 columns: m[i] = image of bit i.  As byte tables: O[j][v] = image of (v << 8j).
CRC_HD uint32_t gf2_apply(const uint32_t* m, uint32_t x) {
    uint32_t r = 0;
    for (int i = 0; i < 32; ++i) if ((x >> i) & 1u) r ^= m[i];
    return r;
}
CRC_HD uint32_t op_entry(const uint32_t* m, uint32_t j, uint32_t v) {   // O[j][v] of the matrix m
    uint32_t r = 0;
    for (uint32_t i = 0; i < 8; ++i) if ((v >> i) & 1u) r ^= m[8 * j + i];
    return r;
}
CRC_HD uint32_t shift(uint32_t x, const uint32_t (*O)[256]) {
    return O[0][x & 0xffu] ^ O[1][(x >> 8) & 0xffu] ^ O[2][(x >> 16) & 0xffu] ^ O[3][x >> 24];
}

// ops[k] = shift by kCrcSeg * 2^k bytes, k = 0 .. kCrcLevels-1 (host: once per process; the kernel gets them as an argument).
inline void make_ops(uint32_t (*ops)[32]) {
    uint32_t t0[256];
    for (uint32_t v = 0; v < 256; ++v) t0[v] = t0_entry(v);
    uint32_t z1[32], acc[32], tmp[32];
    for (int i = 0; i < 32; ++i) { z1[i] = zero_byte(1u << i, t0); acc[i] = 1u << i; }
    for (uint32_t s = 0; s < kCrcSeg; ++s) {            // shift_kCrcSeg = z1^kCrcSeg
        for (int i = 0; i < 32; ++i) tmp[i] = gf2_apply(z1, acc[i]);
        memcpy(acc, tmp, sizeof(acc));
    }
    memcpy(ops[0], acc, sizeof(acc));
    for (uint32_t k = 1; k < kCrcLevels; ++k)
        for (int i = 0; i < 32; ++i) ops[k][i] = gf2_apply(ops[k - 1], ops[k - 1][i]);
}

// crc32(0^n) for n = 0 .. n_max (zlib convention): the trailer value of block n XOR this entry is the block's raw CRC.
inline void make_zeros(uint32_t* out, uint32_t n_max) {
    uint32_t t0[256];
    for (uint32_t v = 0; v < 256; ++v) t0[v] = t0_entry(v);
    uint32_t s = 0xffffffffu;
    out[0] = 0;
    for (uint32_t n = 1; n <= n_max; ++n) { s = zero_byte(s, t0); out[n] = s ^ 0xffffffffu; }
}

// ---- one block --------------------------------------------------------------------------------------------------------------
// End of the frame of the block at address a, n bytes: the frame is [frame_end - kCrcFrame, frame_end), both ends 16-byte aligned.
CRC_HD uint64_t frame_end(uint64_t a, uint32_t n) { return (a + n + 15u) & ~15ull; }

CRC_HD void load16(const uint8_t* p, uint32_t* w) {    // p is 16-byte aligned
#if defined(__CUDA_ARCH__)
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(p));   // the inflated stream is read-only while the kernel runs
    w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
#else
    memcpy(w, p, 16);   // little-endian host
#endif
}

// The bytes of the little-endian word at byte q of a chunk that fall inside [lo, hi) (chunk-relative, may be out of [0, 16]).
CRC_HD uint32_t keep(uint32_t w, int64_t q, int64_t lo, int64_t hi) {
    int64_t l = lo - q, h = hi - q;
    l = l < 0 ? 0 : (l > 4 ? 4 : l);
    h = h < 0 ? 0 : (h > 4 ? 4 : h);
    if (h <= l) return 0u;
    const uint32_t upto = h >= 4 ? 0xffffffffu : ((1u << (8 * h)) - 1u);
    const uint32_t from = ~((1u << (8 * l)) - 1u);   // l <= 3 here
    return w & upto & from;
}

// Raw CRC of segment t of the frame of the block at `blk` (n bytes).  Reads only 16-byte chunks that hold a byte of the block.
CRC_HD uint32_t segment(const uint8_t* blk, uint32_t n, uint32_t t, const uint32_t (*T)[256]) {
    const uint64_t a = reinterpret_cast<uintptr_t>(blk), e = a + n;
    const uint64_t s0 = frame_end(a, n) - kCrcFrame + static_cast<uint64_t>(t) * kCrcSeg, s1 = s0 + kCrcSeg;
    const uint64_t a16 = a & ~15ull;
    uint32_t c = 0;
    for (uint64_t p = s0 > a16 ? s0 : a16; p < s1; p += 64) {   // four chunks loaded before any is hashed: four loads in flight
        uint32_t w[4][4];
        CRC_UNROLL
        for (int i = 0; i < 4; ++i)
            if (p + 16 * i < s1) load16(reinterpret_cast<const uint8_t*>(static_cast<uintptr_t>(p + 16 * i)), w[i]);
        CRC_UNROLL
        for (int i = 0; i < 4; ++i) {
            const uint64_t q = p + 16 * i;
            if (q >= s1) break;
            if (q < a || q + 16 > e) {
                const int64_t lo = static_cast<int64_t>(a) - static_cast<int64_t>(q), hi = static_cast<int64_t>(e) - static_cast<int64_t>(q);
                for (int j = 0; j < 4; ++j) w[i][j] = keep(w[i][j], 4 * j, lo, hi);
            }
            c = step8(c, w[i][0], w[i][1], T);
            c = step8(c, w[i][2], w[i][3], T);
        }
    }
    return c;
}

// Does the frame's raw CRC match the block's expected raw CRC (trailer ^ crc32(0^n))?  The frame carries z zero bytes after the block.
CRC_HD bool matches(uint32_t frame_raw, uint32_t want_raw, const uint8_t* blk, uint32_t n, const uint32_t* t0) {
    const uint64_t a = reinterpret_cast<uintptr_t>(blk);
    const uint32_t z = static_cast<uint32_t>(frame_end(a, n) - (a + n));
    for (uint32_t i = 0; i < z; ++i) want_raw = zero_byte(want_raw, t0);
    return want_raw == frame_raw;
}

}  // namespace bgzf_crc
