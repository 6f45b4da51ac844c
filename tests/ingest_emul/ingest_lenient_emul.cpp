// TEST SIDE: the device ingest's per-record text (metamlst_b200/csrc/ingest_core.cuh) with opts.lenient_tags, compiled for the host and
// driven the way csrc/ingest.cu drives it: the record chain and the warp form of the packer come from ingest_emul.cpp, parse and pack
// run with the lenient flag, and the pack step counts the pileup records without integer AS:i / XM:i as pack_kernel does.
#include "ingest_emul.cpp"

extern "C" {

static uint64_t g_untagged = 0;

// parse_kernel with lenient_tags: returns 0 or (index << 8 | code) of the first refusal
uint64_t emul_parse_lenient(const uint8_t* u, const uint64_t* roff, uint64_t n, int32_t n_ref, uint64_t* key, uint16_t* reflen, int16_t* as0,
                            int16_t* asn, uint16_t* qlen, uint8_t* xm3, uint8_t* xmn, uint8_t* bits, uint64_t* qh) {
    for (uint64_t i = 0; i < n; ++i) {
        Core c;
        const uint32_t e = parse_record(u, roff[i], n_ref, &c, qh ? qh + 2 * i : nullptr, true);
        if (e != E_NONE) return (i << 8) | e;
        key[i] = c.key; reflen[i] = static_cast<uint16_t>(c.reflen); as0[i] = c.as0; asn[i] = c.asn; qlen[i] = c.qlen; xm3[i] = c.xm3; xmn[i] = c.xmn; bits[i] = c.bits;
    }
    return 0;
}

// pack_kernel with lenient_tags for records list[0..P); emul_untagged() then gives the count pack_kernel keeps in d_flags[5]
uint64_t emul_pack_lenient(const uint8_t* u, const uint64_t* roff, const uint32_t* list, uint64_t P, const int32_t* pos, const uint16_t* reflen,
                           const uint8_t* bits, int minqual, const uint64_t* rowoff, uint32_t* planes) {
    g_untagged = 0;
    for (uint64_t j = 0; j < P; ++j) {
        const uint32_t k = list[j];
        const uint32_t rw = row_words(touched_words(static_cast<uint32_t>(pos[k]), reflen[k]));
        const bool named_ok = (bits[k] & 2u) != 0;
        const uint32_t e = pack_record(u, roff[k], static_cast<uint32_t>(pos[k]), reflen[k], named_ok, minqual, planes + rowoff[j], rw, true);
        if (e != E_NONE) return (static_cast<uint64_t>(k) << 8) | e;
        if (reflen[k] && !named_ok) ++g_untagged;
    }
    return 0;
}

uint64_t emul_untagged() { return g_untagged; }

}  // extern "C"
