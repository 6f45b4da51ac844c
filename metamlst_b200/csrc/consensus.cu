// Stage 2b: majority consensus + comparison with the chosen DB allele, one CTA per locus.
// Replaces cmseq/cmseq.py:202-209,234-237,551-554 and metaMLST_functions.py:260-276.  20 B/column in, 1 B out.
#include "common.cuh"

namespace {

constexpr int CONS_THREADS = 512;  // one column per thread for MLST-sized loci: all loads of a locus in flight at once

template <bool CONSUME>
__global__ void __launch_bounds__(CONS_THREADS) consensus_kernel(uint32_t* __restrict__ counts, const uint8_t* __restrict__ dbseq,
                                                        const unsigned long long* __restrict__ db_start,
                                                        const uint32_t* __restrict__ col_off, const uint32_t* __restrict__ n_loci_dev,
                                                        uint32_t mincov, uint8_t* __restrict__ cons,
                                                        uint32_t* __restrict__ holes, uint32_t* __restrict__ snps, unsigned long long* tl) {
    const uint32_t locus = blockIdx.x;
    tl_mark(tl, MMLST_TL_CONSENSUS, 0);
    pdl_wait();                  // counts (pileup) and the selection header are complete and visible
    // the launch covers max_loci CTAs and all four words exist for every one of them: fetched together, ONE round trip instead of three
    const uint32_t nl = n_loci_dev ? *n_loci_dev : 0xffffffffu;
    const uint32_t c0 = col_off[locus], c1 = col_off[locus + 1];
    const unsigned long long dbs = db_start ? db_start[locus] : 0ull;
    tl_mark(tl, MMLST_TL_CONSENSUS, 1, c1 + nl);   // header words have arrived
    if (locus >= nl) return;
    // DB sequence of the chosen allele: either pre-concatenated (column-aligned) or addressed through db_start[locus]
    const uint8_t* db_base = db_start ? dbseq + dbs - c0 : dbseq;
    uint32_t h = 0, s = 0;
    for (uint32_t col = c0 + threadIdx.x; col < c1; col += blockDim.x) {
        uint32_t* c = counts + static_cast<size_t>(col) * 5;
        const uint32_t A = c[0], C = c[1], G = c[2], T = c[3], N = c[4];
        if (CONSUME) { c[0] = 0; c[1] = 0; c[2] = 0; c[3] = 0; c[4] = 0; }  // the next pass accumulates from zero without a memset
        const uint8_t call = (A + C + G + T >= mincov && (A | C | G | T | N)) ? mmlst_majority_call(A, C, G, T, N) : 'N';
        const uint8_t db = db_base[col];
        uint8_t out;
        if (call == 'N') { out = (db >= 'A' && db <= 'Z') ? db + 32 : db; ++h; }
        else { out = call; if (call != db) ++s; }
        cons[col] = out;
    }
    __shared__ uint32_t sh[2];
    if (threadIdx.x < 2) sh[threadIdx.x] = 0;
    __syncthreads();
    h = __reduce_add_sync(0xffffffffu, h);
    s = __reduce_add_sync(0xffffffffu, s);
    if ((threadIdx.x & 31) == 0) { atomicAdd(&sh[0], h); atomicAdd(&sh[1], s); }
    __syncthreads();
    if (threadIdx.x == 0) { holes[locus] = sh[0]; snps[locus] = sh[1]; }
    tl_mark(tl, MMLST_TL_CONSENSUS, 2);
}

}  // namespace

extern "C" int mmlst_consensus_dev(const uint32_t* counts, const uint8_t* dbseq, const uint32_t* col_off, uint32_t n_loci,
                                   uint32_t mincov, uint8_t* cons, uint32_t* holes, uint32_t* snps, void* stream) {
    if (n_loci == 0) return MMLST_OK;
    if (!counts || !dbseq || !col_off || !cons || !holes || !snps) { mmlst_set_error("mmlst_consensus_dev: null pointer"); return MMLST_E_ARG; }
    static bool carve[MMLST_MAX_DEVICES] = {false};
    mmlst_prefer_max_shared(consensus_kernel<false>, carve);
    consensus_kernel<false><<<n_loci, CONS_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(const_cast<uint32_t*>(counts), dbseq, nullptr, col_off, nullptr, mincov, cons, holes, snps, mmlst_timeline_buffer());
    CUDA_TRY(cudaGetLastError());
    return MMLST_OK;
}

// device-driven variant: n_loci and the DB offsets come from mmlst_select_dev (header[0], db_start)
extern "C" int mmlst_consensus_indirect_dev(uint32_t* counts, const uint8_t* db_ascii, const uint64_t* db_start,
                                            const uint32_t* col_off, uint32_t max_loci, const uint32_t* header, uint32_t mincov,
                                            uint8_t* cons, uint32_t* holes, uint32_t* snps, uint32_t flags, void* stream) {
    if (max_loci == 0) return MMLST_OK;
    if (!counts || !db_ascii || !db_start || !col_off || !header || !cons || !holes || !snps) { mmlst_set_error("mmlst_consensus_indirect_dev: null pointer"); return MMLST_E_ARG; }
    const unsigned long long* dbs = reinterpret_cast<const unsigned long long*>(db_start);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    static bool carve_t[MMLST_MAX_DEVICES] = {false}, carve_f[MMLST_MAX_DEVICES] = {false};
    mmlst_prefer_max_shared(consensus_kernel<true>, carve_t);
    mmlst_prefer_max_shared(consensus_kernel<false>, carve_f);
    if (flags & MMLST_CONSENSUS_CONSUME) CUDA_TRY(mmlst_launch_dependent(consensus_kernel<true>, dim3(max_loci), dim3(CONS_THREADS), 0, s, counts, db_ascii, dbs, col_off, header, mincov, cons, holes, snps, mmlst_timeline_buffer()));
    else CUDA_TRY(mmlst_launch_dependent(consensus_kernel<false>, dim3(max_loci), dim3(CONS_THREADS), 0, s, counts, db_ascii, dbs, col_off, header, mincov, cons, holes, snps, mmlst_timeline_buffer()));
    return MMLST_OK;
}
