// Per-record logic of the DEVICE-side BAM ingest (csrc/ingest.cu), written as host/device inline functions so that the same
// text runs in the CUDA kernels and -- compiled by g++ in tests/ingest_emul -- on the host against the C++ unpacker
// (csrc/bam_unpack.cpp) before a GPU ever sees it.  Semantics are those of bam_unpack.cpp phase 3-6, i.e. what the reference
// gets from `samtools view` text (metamlst.py:96-110: RNAME, 1st / 4th aux field by POSITION, len(SEQ)) and from pysam
// (cmseq/cmseq.py:527-545: CIGAR walk, base / quality at query_position, AS / XM by NAME).
//
// BAM record layout (little endian, unaligned): block_size i32 | refID i32 | pos i32 | l_read_name u8 | mapq u8 | bin u16 |
// n_cigar_op u16 | flag u16 | l_seq u32 | next_refID i32 | next_pos i32 | tlen i32 | read_name | cigar u32[] | seq 4-bit | qual | aux
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define ING_HD __host__ __device__ __forceinline__
#else
#define ING_HD inline
#endif

namespace ingest {

enum Err : uint32_t {
    E_NONE = 0,
    E_TRUNC = 1,        // truncated / malformed record (block_size < 32 or beyond the stream)
    E_OVERRUN = 2,      // fixed part + name + cigar + seq + qual overrun block_size, or l_read_name == 0
    E_NOREF = 3,        // RNAME '*': the reference crashes at metamlst.py:107
    E_PAIRED = 4,       // proper-pair mate: htslib overlap handling (H2) refused
    E_NEGPOS = 5,       // POS 0 on a reference
    E_REFSPAN = 6,      // reference span > 65535
    E_CIGQ = 7,         // CIGAR query length != l_seq
    E_AUX = 8,          // malformed aux field
    E_AUXPOS = 9,       // 1st / 4th aux field missing or not an integer (metamlst.py:109-110)
    E_AS0 = 10,         // 1st aux field outside int16
    E_XM3 = 11,         // negative 4th aux field
    E_NAMED = 12,       // record enters the pileup without integer AS:i / XM:i (cmseq/cmseq.py:545)
    E_NOQUAL = 13,      // record enters the pileup without base qualities (cmseq/cmseq.py:538)
    E_CHAIN = 14,       // record chain could not be established (internal)
    E_QLEN = 15,        // read longer than 65535 bases (len(SEQ) is carried as 16 bits)
    E_CRC = 16          // inflated BGZF block does not match its trailer's CRC-32 (index = block, opts.check_crc)
};

ING_HD uint32_t rd16(const uint8_t* p) { return static_cast<uint32_t>(p[0]) | (static_cast<uint32_t>(p[1]) << 8); }
ING_HD uint32_t rd32(const uint8_t* p) {
    return static_cast<uint32_t>(p[0]) | (static_cast<uint32_t>(p[1]) << 8) | (static_cast<uint32_t>(p[2]) << 16) | (static_cast<uint32_t>(p[3]) << 24);
}
ING_HD int32_t rdi32(const uint8_t* p) { return static_cast<int32_t>(rd32(p)); }

// ---- record chain ----------------------------------------------------------------------------------------------------------
// Offset of the record after the one at `off`, or 0 when the record at `off` is malformed (block_size < 32 or past the end).
ING_HD uint64_t next_record(const uint8_t* u, uint64_t off, uint64_t usize) {
    if (off + 4 > usize) return 0;
    const int32_t bs = rdi32(u + off);
    if (bs < 32 || off + 4 + static_cast<uint64_t>(bs) > usize) return 0;
    return off + 4 + static_cast<uint64_t>(bs);
}

// Could a BAM record START at `off`?  Used only to GUESS the first record boundary inside a BGZF block whose predecessor has
// not been walked yet; every guess is verified afterwards (the chain from block k must land exactly on the guess of block k+1),
// so a false positive costs a repair pass, never a wrong result.  The test is strict enough that a false positive needs ~12
// independent coincidences.
ING_HD bool plausible_record(const uint8_t* u, uint64_t off, uint64_t usize, int32_t n_ref, const uint32_t* ref_len) {
    if (off + 36 > usize) return false;
    const int32_t bs = rdi32(u + off);
    if (bs < 32 || bs > (1 << 28) || off + 4 + static_cast<uint64_t>(bs) > usize) return false;
    const int32_t tid = rdi32(u + off + 4), pos = rdi32(u + off + 8);
    if (tid < -1 || tid >= n_ref || pos < -1) return false;
    if (tid >= 0 && static_cast<int64_t>(pos) > static_cast<int64_t>(ref_len[tid])) return false;
    const uint32_t l_name = u[off + 12], n_cig = rd16(u + off + 16), l_seq = rd32(u + off + 20);
    if (l_name == 0) return false;
    const int32_t ntid = rdi32(u + off + 24), npos = rdi32(u + off + 28);
    if (ntid < -1 || ntid >= n_ref || npos < -1) return false;
    const uint64_t fixed = 32ull + l_name + 4ull * n_cig + (static_cast<uint64_t>(l_seq) + 1) / 2 + l_seq;
    if (fixed > static_cast<uint64_t>(bs)) return false;
    const uint8_t* name = u + off + 36;
    if (name[l_name - 1] != 0) return false;
    for (uint32_t i = 0; i + 1 < l_name; ++i) if (name[i] < 33 || name[i] > 126) return false;   // SAM: [!-?A-~]{1,254}
    const uint8_t* cig = name + l_name;
    for (uint32_t k = 0; k < n_cig; ++k) if ((cig[4 * k] & 15u) > 8u) return false;
    return true;
}

// ---- per-record fields -----------------------------------------------------------------------------------------------------
struct Core {
    uint64_t key;       // samtools sort key: tid << 33 | (pos + 1) << 1 | reverse strand
    uint32_t reflen;    // reference span (<= 65535)
    int16_t as0;        // 1st aux field by POSITION
    int16_t asn;        // AS:i by NAME (0 unless named_ok)
    uint16_t qlen;      // len(SEQ) as SAM prints it ('*' -> 1), saturated at 65535
    uint8_t xm3;        // 4th aux field by POSITION, saturated at 255
    uint8_t xmn;        // XM:i by NAME, saturated at 255
    uint8_t bits;       // bit 0: takes part in the pileup (flag & 4 clear); bit 1: named_ok
};

ING_HD uint32_t aux_size(uint8_t t, const uint8_t* p, const uint8_t* end) {
    switch (t) {
        case 'A': case 'c': case 'C': return 1;
        case 's': case 'S': return 2;
        case 'i': case 'I': case 'f': return 4;
        case 'Z': case 'H': {
            for (const uint8_t* z = p; z < end; ++z) if (*z == 0) return static_cast<uint32_t>(z - p) + 1;
            return 0;
        }
        case 'B': {
            if (end - p < 5) return 0;
            uint32_t es;
            switch (p[0]) { case 'c': case 'C': es = 1; break; case 's': case 'S': es = 2; break; case 'i': case 'I': case 'f': es = 4; break; default: return 0; }
            const uint64_t sz = 5ull + static_cast<uint64_t>(es) * rd32(p + 1);
            return sz > 0x7fffffffull ? 0u : static_cast<uint32_t>(sz);
        }
        default: return 0;
    }
}
ING_HD bool aux_int(uint8_t t, const uint8_t* p, int64_t* v) {
    switch (t) {
        case 'c': *v = static_cast<int8_t>(p[0]); return true;
        case 'C': *v = p[0]; return true;
        case 's': *v = static_cast<int16_t>(rd16(p)); return true;
        case 'S': *v = rd16(p); return true;
        case 'i': *v = rdi32(p); return true;
        case 'I': *v = rd32(p); return true;
        default: return false;
    }
}

ING_HD uint64_t hash64(const uint8_t* s, uint32_t n) {  // same two hashes as bam_unpack.cpp (128-bit QNAME key, H7)
    uint64_t h = 0xcbf29ce484222325ull;
    for (uint32_t i = 0; i < n; ++i) { h ^= s[i]; h *= 0x100000001b3ull; }
    h ^= h >> 30; h *= 0xbf58476d1ce4e5b9ull; h ^= h >> 27; h *= 0x94d049bb133111ebull; h ^= h >> 31;
    return h;
}
ING_HD uint64_t hash64b(const uint8_t* s, uint32_t n) {
    uint64_t h = 0x9e3779b97f4a7c15ull ^ (static_cast<uint64_t>(n) * 0xff51afd7ed558ccdull);
    for (uint32_t i = 0; i < n; ++i) { h = (h ^ s[i]) * 0xc6a4a7935bd1e995ull; h ^= h >> 47; }
    h ^= h >> 33; h *= 0xff51afd7ed558ccdull; h ^= h >> 33; h *= 0xc4ceb9fe1a85ec53ull; h ^= h >> 33;
    return h;
}

// One record at u + off (off from the record chain, so block_size is sane).  Returns E_NONE or the first refusal, in the order
// bam_unpack.cpp tests them.  qh: 2 x u64 or nullptr.
ING_HD uint32_t parse_record(const uint8_t* u, uint64_t off, int32_t n_ref, Core* out, uint64_t* qh) {
    const uint8_t* r = u + off;
    const uint32_t bs = rd32(r);
    const uint8_t* end = r + 4 + bs;
    const int32_t tid = rdi32(r + 4), pos = rdi32(r + 8);
    const uint32_t l_name = r[12], n_cig = rd16(r + 16), flag = rd16(r + 18), l_seq = rd32(r + 20);
    const uint8_t* q = r + 36;
    const uint8_t* cig = q + l_name;
    const uint8_t* seq = cig + 4ull * n_cig;
    const uint8_t* aux = seq + (static_cast<uint64_t>(l_seq) + 1) / 2 + l_seq;
    if (aux > end || l_name == 0) return E_OVERRUN;
    if (tid < 0 || tid >= n_ref) return E_NOREF;
    if (flag & 0x2u) return E_PAIRED;
    if (pos < 0) return E_NEGPOS;
    if (qh) { qh[0] = hash64(q, l_name - 1); qh[1] = hash64b(q, l_name - 1); }
    uint64_t rl = 0, qlsum = 0;
    for (uint32_t k = 0; k < n_cig; ++k) {
        const uint32_t cw = rd32(cig + 4 * k), op = cw & 15u, ln = cw >> 4;
        if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) rl += ln;
        if (op == 0 || op == 1 || op == 4 || op == 7 || op == 8) qlsum += ln;
    }
    if (rl > 65535) return E_REFSPAN;
    if (n_cig && l_seq && qlsum != l_seq) return E_CIGQ;
    Core c;
    c.key = (static_cast<uint64_t>(static_cast<uint32_t>(tid)) << 33) | ((static_cast<uint64_t>(static_cast<uint32_t>(pos)) + 1ull) << 1) | ((flag >> 4) & 1u);
    c.reflen = static_cast<uint32_t>(rl);
    if (l_seq > 65535u) return E_QLEN;
    const uint32_t ql = l_seq ? l_seq : 1u;  // SAM prints SEQ '*' when l_seq == 0: len() == 1 (metamlst.py:111,115)
    c.qlen = static_cast<uint16_t>(ql < 65535u ? ql : 65535u);
    int field = 0;
    int64_t v0 = 0, v3 = 0, vas = 0, vxm = 0;
    bool ok0 = false, ok3 = false, okas = false, okxm = false;
    for (const uint8_t* a2 = aux; a2 + 3 <= end; ++field) {
        const uint8_t t = a2[2];
        const uint8_t* val = a2 + 3;
        const uint32_t sz = aux_size(t, val, end);
        if (sz == 0 || val + sz > end) return E_AUX;
        int64_t v = 0;
        const bool isint = aux_int(t, val, &v);
        if (field == 0) { ok0 = isint; v0 = v; }
        if (field == 3) { ok3 = isint; v3 = v; }
        if (isint && a2[0] == 'A' && a2[1] == 'S' && !okas) { okas = true; vas = v; }
        if (isint && a2[0] == 'X' && a2[1] == 'M' && !okxm) { okxm = true; vxm = v; }
        a2 = val + sz;
    }
    if (field < 4 || !ok0 || !ok3) return E_AUXPOS;
    if (v0 < -32768 || v0 > 32767) return E_AS0;
    if (v3 < 0) return E_XM3;
    c.as0 = static_cast<int16_t>(v0);
    c.xm3 = static_cast<uint8_t>(v3 < 255 ? v3 : 255);
    const bool named_ok = okas && okxm && vas >= -32768 && vas <= 32767 && vxm >= 0;
    c.asn = named_ok ? static_cast<int16_t>(vas) : static_cast<int16_t>(0);
    c.xmn = named_ok ? static_cast<uint8_t>(vxm < 255 ? vxm : 255) : static_cast<uint8_t>(0);
    c.bits = static_cast<uint8_t>(((flag & 0x4u) ? 0u : 1u) | (named_ok ? 2u : 0u));
    *out = c;
    return E_NONE;
}

// ---- plane rows ------------------------------------------------------------------------------------------------------------
ING_HD uint32_t touched_words(uint32_t pos, uint32_t reflen) { return reflen ? (((pos & 31u) + reflen + 31u) >> 5) : 0u; }
ING_HD uint32_t row_words(uint32_t nw) {  // 3 planes, padded to an odd word count
    const uint32_t rw = 3u * nw;
    return rw + ((rw != 0u && (rw & 1u) == 0u) ? 1u : 0u);
}

// The record's plane row (include/mmlst.h: word-interleaved [V, B1, B0] per 32 contig columns, aligned to the contig's words).
// `row` (rw words) is written completely.  Returns E_NONE, E_NAMED or E_NOQUAL (the record is in the pileup: what pysam would
// raise on, cmseq/cmseq.py:538,545).
ING_HD uint32_t pack_record(const uint8_t* u, uint64_t off, uint32_t pos, uint32_t reflen, bool named_ok, int minqual, uint32_t* row, uint32_t rw) {
    for (uint32_t w = 0; w < rw; ++w) row[w] = 0;
    if (reflen == 0) return E_NONE;
    if (!named_ok) return E_NAMED;
    const uint8_t* r = u + off;
    const uint32_t l_name = r[12], n_cig = rd16(r + 16), l_seq = rd32(r + 20);
    const uint8_t* cig = r + 36 + l_name;
    const uint8_t* seq = cig + 4ull * n_cig;
    const uint8_t* qual = seq + (static_cast<uint64_t>(l_seq) + 1) / 2;
    if (l_seq && qual[0] == 0xff) return E_NOQUAL;
    uint32_t x = pos & 31u, y = 0;       // column inside the row, query index
    uint32_t wi = 0, pv = 0, p1 = 0, p0 = 0;
    for (uint32_t k = 0; k < n_cig; ++k) {
        const uint32_t cw = rd32(cig + 4 * k), op = cw & 15u, ln = cw >> 4;
        if (op == 0 || op == 7 || op == 8) {
            for (uint32_t t = 0; t < ln; ++t, ++x, ++y) {
                if ((x >> 5) != wi) {
                    uint32_t* w3 = row + 3 * wi;
                    w3[0] |= pv; w3[1] |= p1; w3[2] |= p0;
                    wi = x >> 5; pv = p1 = p0 = 0;
                }
                if (y >= l_seq) continue;                                   // qpos beyond l_qseq: quality 0
                if (static_cast<int>(qual[y]) < minqual) continue;         // H3: not in column.pileups at all
                const uint32_t nib = (seq[y >> 1] >> ((~y & 1u) << 2)) & 15u;
                // BAM 4-bit codes "=ACMGRSVTWYHKDBN": A=1 C=2 G=4 T=8 -> 2-bit code; anything else is a counted non-ACGT base
                const int cd = nib == 1u ? 0 : nib == 2u ? 1 : nib == 4u ? 2 : nib == 8u ? 3 : -1;
                const uint32_t bit = 1u << (x & 31u);
                if (cd >= 0) { pv |= bit; if (cd & 2) p1 |= bit; if (cd & 1) p0 |= bit; }
                else p0 |= bit;                                             // V=0, B0=1: bin N
            }
        } else if (op == 1 || op == 4) y += ln;
        else if (op == 2 || op == 3) x += ln;
    }
    if (pv | p1 | p0) {
        uint32_t* w3 = row + 3 * wi;
        w3[0] |= pv; w3[1] |= p1; w3[2] |= p0;
    }
    return E_NONE;
}

// The same row, one COLUMN at a time (the warp form of the packer: lane = column): class of contig column `col` for this record,
// 0 = not in the column (outside the span, deletion / ref-skip, quality under minqual, beyond l_seq); 1..4 = A,C,G,T with quality
// >= minqual; 5 = counted non-ACGT base (bin N).
ING_HD uint32_t column_class(const uint8_t* cig, uint32_t n_cig, const uint8_t* seq, const uint8_t* qual, uint32_t l_seq, uint32_t pos, uint32_t reflen,
                             uint32_t col, int minqual) {
    if (col < pos || col - pos >= reflen) return 0;
    const uint32_t rel = col - pos;
    uint32_t rx = 0, qy = 0;
    for (uint32_t k = 0; k < n_cig; ++k) {
        const uint32_t cw = rd32(cig + 4 * k), op = cw & 15u, ln = cw >> 4;
        if (op == 0 || op == 7 || op == 8) {
            if (rel - rx < ln) {
                const uint32_t y = qy + (rel - rx);
                if (y >= l_seq) return 0;
                if (static_cast<int>(qual[y]) < minqual) return 0;
                const uint32_t nib = (seq[y >> 1] >> ((~y & 1u) << 2)) & 15u;
                return nib == 1u ? 1u : nib == 2u ? 2u : nib == 4u ? 3u : nib == 8u ? 4u : 5u;
            }
            rx += ln; qy += ln;
        } else if (op == 1 || op == 4) qy += ln;
        else if (op == 2 || op == 3) {
            if (rel - rx < ln) return 0;
            rx += ln;
        }
    }
    return 0;
}

}  // namespace ingest
