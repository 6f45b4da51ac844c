// Coverage column of stage 1 (hazard H7): per locus the sum over UNIQUE read names of len(SEQ) of the LAST passing
// record carrying that name (metamlst.py:127 `sequenceBank[species_gene][readCode] = len(sequence)` -- a dict, so later
// records overwrite earlier ones -- summed at metamlst.py:228).
//
// Read names reach the device as a 128-bit hash per record (two independent 64-bit hashes computed once at unpack);
// names are "equal" when both halves are: for n distinct names per locus the probability of ANY false merge is
// < n^2 / 2^129 (10^7 names: 3e-25).  The set is an open-addressing table in HBM claimed with one 128-bit
// compare-and-swap per new name (ATOMG.E.CAS.128); the value word is (file index + 1) << 16 | len(SEQ) under a 64-bit
// atomicMax, so "last record wins" is order-independent, hence identical for any launch shape or GPU count.
//   pass 1  insert_kernel : every passing record -> claim/find its (locus, name) slot, atomicMax the value
//   pass 2  sum_kernel    : every passing record looks its slot up again; the one record whose index IS the maximum
//                           adds its len(SEQ) to cov[locus] (warp-aggregated when the warp is on one locus)
// Record shards that cut through loci (a contiguous range of the sorted stream per rank) run the passes apart: between
// them every rank raises its own slots to the maximum any rank holds for the key (merge_kernel over the other ranks'
// occupied slots), so that only the rank holding the globally last record of a name adds it.
// Random 32-byte sector traffic, not a streaming kernel: it is off the headline pass and run only when the coverage
// column is wanted.
#include "common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr uint32_t FULL = 0xffffffffu;
constexpr uint64_t kMaxIdx = (1ull << 48) - 1;  // value word: (file index + 1) << 16 | len(SEQ)

struct __align__(16) Key128 { unsigned long long lo, hi; };

struct CovArgs {
    const uint32_t* tid; const int16_t* as0; const uint8_t* xm3; const uint16_t* qlen; const uint32_t* orig_idx;
    const unsigned long long* qhash;  // [n_rec][2]
    uint64_t n_rec, idx_base;
    const uint8_t* allow; const uint32_t* locus_of; uint32_t n_ref;
    int minscore, max_xm, min_read_len;
    Key128* keys; unsigned long long* vals; uint64_t mask;
    unsigned long long* cov;
};

__device__ __forceinline__ Key128 cas128(Key128* addr, Key128 cmp, Key128 val) {
    Key128 old;
    asm volatile("{\n\t.reg .b128 c, v, o;\n\tmov.b128 c, {%3, %4};\n\tmov.b128 v, {%5, %6};\n\t"
                 "atom.global.relaxed.gpu.cas.b128 o, [%2], c, v;\n\tmov.b128 {%0, %1}, o;\n\t}"
                 : "=l"(old.lo), "=l"(old.hi) : "l"(addr), "l"(cmp.lo), "l"(cmp.hi), "l"(val.lo), "l"(val.hi) : "memory");
    return old;
}
__device__ __forceinline__ Key128 ld128(const Key128* p) {
    Key128 k;
    asm volatile("ld.global.v2.u64 {%0, %1}, [%2];" : "=l"(k.lo), "=l"(k.hi) : "l"(p) : "memory");
    return k;
}
__device__ __forceinline__ uint64_t mix64(uint64_t h) {
    h ^= h >> 30; h *= 0xbf58476d1ce4e5b9ull; h ^= h >> 27; h *= 0x94d049bb133111ebull; h ^= h >> 31;
    return h;
}

// one record: passing? -> (locus, key, value, slot0)
struct Rec { bool pass; uint32_t locus; Key128 key; unsigned long long val; uint64_t slot; uint32_t ql; };

__device__ __forceinline__ Rec load_rec(const CovArgs& a, uint64_t i) {
    Rec r;
    r.pass = false; r.locus = 0; r.key = Key128{0, 0}; r.val = 0; r.slot = 0; r.ql = 0;
    if (i >= a.n_rec) return r;
    const uint32_t t = a.tid[i];
    if (t >= a.n_ref || !a.allow[t]) return r;
    const int as = a.as0[i];
    const int ql = a.qlen[i];
    const int xm = a.xm3[i];
    if (!((as >= a.minscore) && (ql >= a.min_read_len) && (xm <= a.max_xm))) return r;  // metamlst.py:115
    r.pass = true;
    r.locus = a.locus_of[t];
    r.ql = static_cast<uint32_t>(ql);
    r.key.lo = a.qhash[2 * i];
    const unsigned long long fold = static_cast<unsigned long long>(r.locus + 1u) * 0x9E3779B97F4A7C15ull;  // one set per locus
    r.key.hi = a.qhash[2 * i + 1] ^ fold;
    // {0,0} is the empty slot: remap it to {1, fold}, the key of the hash {1, 0} on the SAME locus (a collision of the 128-bit
    // hash, like any other), never to a key shared by every locus.  fold != 0: locus + 1 < 2^32 times an odd constant.
    if ((r.key.lo | r.key.hi) == 0ull) { r.key.lo = 1ull; r.key.hi = fold; }
    const unsigned long long idx = a.orig_idx ? static_cast<unsigned long long>(a.orig_idx[i]) : (a.idx_base + i);
    r.val = ((idx + 1ull) << 16) | static_cast<unsigned long long>(r.ql);
    r.slot = mix64(r.key.lo ^ mix64(r.key.hi)) & a.mask;
    return r;
}

__global__ void __launch_bounds__(kThreads) cov_insert_kernel(const CovArgs a) {
    const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
    for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < a.n_rec; i += stride) {
        const Rec r = load_rec(a, i);
        if (!r.pass) continue;
        uint64_t s = r.slot;
        for (uint64_t probe = 0; probe <= a.mask; ++probe, s = (s + 1) & a.mask) {
            // plain read first: 3 of 4 records of a read (K alignments on one locus) find their name already present.
            // A torn 128-bit read can only show a half-written key, which never EQUALS r.key; anything else is
            // settled by the CAS, whose returned value is authoritative.
            Key128 cur = ld128(a.keys + s);
            if (!(cur.lo == r.key.lo && cur.hi == r.key.hi)) {
                cur = cas128(a.keys + s, Key128{0, 0}, r.key);
                if (!(((cur.lo | cur.hi) == 0ull) || (cur.lo == r.key.lo && cur.hi == r.key.hi))) continue;  // other name: next slot
            }
            atomicMax(a.vals + s, r.val);
            break;
        }
    }
}

__global__ void __launch_bounds__(kThreads) cov_sum_kernel(const CovArgs a) {
    const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
    const uint64_t n_round = (a.n_rec + stride - 1) / stride;  // whole warps stay in the loop (warp-wide votes below)
    uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    for (uint64_t it = 0; it < n_round; ++it, i += stride) {
        const Rec r = load_rec(a, i);
        uint32_t add = 0;
        if (r.pass) {
            uint64_t s = r.slot;
            for (uint64_t probe = 0; probe <= a.mask; ++probe, s = (s + 1) & a.mask) {
                const Key128 cur = ld128(a.keys + s);
                if (cur.lo == r.key.lo && cur.hi == r.key.hi) {
                    if (a.vals[s] == r.val) add = r.ql;  // this record is the last one with the name
                    break;
                }
                if ((cur.lo | cur.hi) == 0ull) break;  // cannot happen after pass 1
            }
        }
        const uint32_t contributing = __ballot_sync(FULL, add != 0);
        if (contributing == 0) continue;
        const uint32_t leader = __ffs(contributing) - 1;
        const uint32_t l0 = __shfl_sync(FULL, r.locus, leader);
        if (__all_sync(FULL, add == 0 || r.locus == l0)) {
            const uint32_t tot = __reduce_add_sync(FULL, add);
            if ((threadIdx.x & 31u) == leader) atomicAdd(a.cov + l0, static_cast<unsigned long long>(tot));
        } else if (add) {
            atomicAdd(a.cov + r.locus, static_cast<unsigned long long>(add));
        }
    }
}

__global__ void __launch_bounds__(kThreads) cov_merge_kernel(const Key128* __restrict__ in_keys, const unsigned long long* __restrict__ in_vals,
                                                             uint64_t m, Key128* keys, unsigned long long* vals, uint64_t mask) {
    const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
    for (uint64_t j = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; j < m; j += stride) {
        const Key128 k = in_keys[j];
        if ((k.lo | k.hi) == 0ull) continue;  // padding / empty slot of the sender
        uint64_t s = mix64(k.lo ^ mix64(k.hi)) & mask;
        for (uint64_t probe = 0; probe <= mask; ++probe, s = (s + 1) & mask) {
            const Key128 cur = ld128(keys + s);
            if (cur.lo == k.lo && cur.hi == k.hi) {
                atomicMax(vals + s, in_vals[j]);
                break;
            }
            if ((cur.lo | cur.hi) == 0ull) break;  // no local record has the name: nothing to decide here
        }
    }
}

uint32_t grid_for(uint64_t n) {
    const uint64_t want = (n + kThreads - 1) / kThreads;
    const uint64_t cap = static_cast<uint64_t>(mmlst_num_sms()) * 16u;
    return static_cast<uint32_t>(want < cap ? want : cap);
}

int check_table(const char* who, const void* table, uint64_t table_slots) {
    if (!table) {
        mmlst_set_error("%s: null pointer", who);
        return MMLST_E_ARG;
    }
    if (table_slots < 2 || (table_slots & (table_slots - 1)) || (reinterpret_cast<uintptr_t>(table) & 15)) {
        mmlst_set_error("%s: table_slots must be a power of two and the table 16-byte aligned", who);
        return MMLST_E_ARG;
    }
    return MMLST_OK;
}

// pass: 1 = insert, 2 = sum, 3 = both
int coverage_passes(const char* who, int pass, const uint32_t* tid, const int16_t* as0, const uint8_t* xm3, const uint16_t* qlen,
                    const uint32_t* orig_idx, const uint64_t* qhash, uint64_t n_rec, uint64_t idx_base, const uint8_t* allow,
                    const uint32_t* locus_of, uint32_t n_ref, int minscore, int max_xm, int min_read_len, void* table,
                    uint64_t table_slots, uint64_t* cov, void* stream) {
    if (n_rec == 0) return MMLST_OK;
    if (!tid || !as0 || !xm3 || !qlen || !qhash || !allow || !locus_of || ((pass & 2) && !cov)) {
        mmlst_set_error("%s: null pointer", who);
        return MMLST_E_ARG;
    }
    if (int rc = check_table(who, table, table_slots)) return rc;
    if (!orig_idx && (idx_base >= kMaxIdx || n_rec > kMaxIdx - idx_base)) {  // (idx + 1) << 16 must not lose bits
        mmlst_set_error("%s: idx_base + n_rec = %llu exceeds the 48-bit file index of the value word", who,
                        static_cast<unsigned long long>(idx_base + n_rec));
        return MMLST_E_RANGE;
    }
    CovArgs a{tid, as0, xm3, qlen, orig_idx, reinterpret_cast<const unsigned long long*>(qhash), n_rec, idx_base, allow, locus_of, n_ref,
              minscore, max_xm, min_read_len, static_cast<Key128*>(table),
              reinterpret_cast<unsigned long long*>(static_cast<uint8_t*>(table) + 16 * table_slots), table_slots - 1,
              reinterpret_cast<unsigned long long*>(cov)};
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const uint32_t grid = grid_for(n_rec);
    if (pass & 1) {
        cov_insert_kernel<<<grid, kThreads, 0, s>>>(a);
        if (int rc = mmlst_cuda_fail(cudaGetLastError(), "cov_insert_kernel")) return rc;
    }
    if (pass & 2) {
        cov_sum_kernel<<<grid, kThreads, 0, s>>>(a);
        if (int rc = mmlst_cuda_fail(cudaGetLastError(), "cov_sum_kernel")) return rc;
    }
    return MMLST_OK;
}

}  // namespace

extern "C" uint64_t mmlst_coverage_table_slots(uint64_t n_names_upper_bound) {
    uint64_t s = 1024;
    while (s < 2 * n_names_upper_bound) s <<= 1;
    return s;
}

extern "C" int mmlst_coverage_dev(const uint32_t* tid, const int16_t* as0, const uint8_t* xm3, const uint16_t* qlen,
                                  const uint32_t* orig_idx, const uint64_t* qhash, uint64_t n_rec, uint64_t idx_base,
                                  const uint8_t* allow, const uint32_t* locus_of, uint32_t n_ref, int minscore, int max_xm,
                                  int min_read_len, void* table, uint64_t table_slots, uint64_t* cov, void* stream) {
    return coverage_passes("mmlst_coverage_dev", 3, tid, as0, xm3, qlen, orig_idx, qhash, n_rec, idx_base, allow, locus_of, n_ref,
                           minscore, max_xm, min_read_len, table, table_slots, cov, stream);
}

extern "C" int mmlst_coverage_insert_dev(const uint32_t* tid, const int16_t* as0, const uint8_t* xm3, const uint16_t* qlen,
                                         const uint32_t* orig_idx, const uint64_t* qhash, uint64_t n_rec, uint64_t idx_base,
                                         const uint8_t* allow, const uint32_t* locus_of, uint32_t n_ref, int minscore, int max_xm,
                                         int min_read_len, void* table, uint64_t table_slots, uint64_t* cov, void* stream) {
    return coverage_passes("mmlst_coverage_insert_dev", 1, tid, as0, xm3, qlen, orig_idx, qhash, n_rec, idx_base, allow, locus_of, n_ref,
                           minscore, max_xm, min_read_len, table, table_slots, cov, stream);
}

extern "C" int mmlst_coverage_sum_dev(const uint32_t* tid, const int16_t* as0, const uint8_t* xm3, const uint16_t* qlen,
                                      const uint32_t* orig_idx, const uint64_t* qhash, uint64_t n_rec, uint64_t idx_base,
                                      const uint8_t* allow, const uint32_t* locus_of, uint32_t n_ref, int minscore, int max_xm,
                                      int min_read_len, void* table, uint64_t table_slots, uint64_t* cov, void* stream) {
    return coverage_passes("mmlst_coverage_sum_dev", 2, tid, as0, xm3, qlen, orig_idx, qhash, n_rec, idx_base, allow, locus_of, n_ref,
                           minscore, max_xm, min_read_len, table, table_slots, cov, stream);
}

extern "C" int mmlst_coverage_merge_dev(const uint64_t* keys, const uint64_t* vals, uint64_t m, void* table, uint64_t table_slots,
                                        void* stream) {
    if (m == 0) return MMLST_OK;
    if (!keys || !vals || (reinterpret_cast<uintptr_t>(keys) & 15)) {
        mmlst_set_error("mmlst_coverage_merge_dev: keys must be non-null and 16-byte aligned, vals non-null");
        return MMLST_E_ARG;
    }
    if (int rc = check_table("mmlst_coverage_merge_dev", table, table_slots)) return rc;
    cov_merge_kernel<<<grid_for(m), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
        reinterpret_cast<const Key128*>(keys), reinterpret_cast<const unsigned long long*>(vals), m, static_cast<Key128*>(table),
        reinterpret_cast<unsigned long long*>(static_cast<uint8_t*>(table) + 16 * table_slots), table_slots - 1);
    return mmlst_cuda_fail(cudaGetLastError(), "cov_merge_kernel");
}
