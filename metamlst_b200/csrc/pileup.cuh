// Shared declarations of the two pileup implementations.
#pragma once
#include "common.cuh"

// Consensus fused into the pileup launch (device-driven pass): the chunk list of mmlst_select_dev names, per chunk, the chosen locus it belongs to
// (reserved[0]) and how many chunks that locus has (reserved[1]); the CTA that finishes the LAST chunk of a locus (ticket counter per locus, left at
// zero) calls the consensus of that locus while its counts are still in L2 -- one launch and one cold-cache pass over the count tensor less per sample.
struct FusedConsensus {
    uint32_t* ticket;            // [max loci] zero-initialised, self-resetting; nullptr = not fused
    const uint8_t* db_ascii; const unsigned long long* db_start; const uint32_t* col_off;
    uint32_t mincov; uint8_t* cons; uint32_t* holes; uint32_t* snps; uint32_t consume;
};

struct PileupArgs {
    const mmlst_prec* recs;
    const uint32_t* planes; const mmlst_chunk* chunks; uint32_t n_chunks; uint32_t max_row_words;
    int minscore, max_xm; uint32_t* counts; uint32_t total_cols;
    const uint32_t* n_chunks_dev;  // when non-null the chunk count is read on the device (written by mmlst_select_dev)
    FusedConsensus fc;
    unsigned long long* tl = nullptr;   // profiling aid (mmlst_debug_timeline), nullptr = off
};

// majority call + comparison with the DB allele for the columns [c0, c1) of one locus, by the whole CTA (cmseq/cmseq.py:202-209,234-237,551-554,
// metaMLST_functions.py:260-276; same arithmetic as consensus_kernel).  sh: two shared words.
__device__ __forceinline__ void consensus_of_locus(uint32_t* counts, const uint8_t* db_base, uint32_t c0, uint32_t c1, uint32_t mincov, bool consume,
                                                   uint8_t* cons, uint32_t* holes_out, uint32_t* snps_out, uint32_t* sh) {
    uint32_t h = 0, s = 0;
    for (uint32_t col = c0 + threadIdx.x; col < c1; col += blockDim.x) {
        uint32_t* c = counts + static_cast<size_t>(col) * 5;
        const uint32_t A = __ldcg(c + 0), C = __ldcg(c + 1), G = __ldcg(c + 2), T = __ldcg(c + 3), N = __ldcg(c + 4);
        if (consume) { c[0] = 0; c[1] = 0; c[2] = 0; c[3] = 0; c[4] = 0; }
        const uint8_t call = (A + C + G + T >= mincov && (A | C | G | T | N)) ? mmlst_majority_call(A, C, G, T, N) : 'N';
        const uint8_t db = db_base[col];
        uint8_t out;
        if (call == 'N') { out = (db >= 'A' && db <= 'Z') ? db + 32 : db; ++h; }
        else { out = call; if (call != db) ++s; }
        cons[col] = out;
    }
    if (threadIdx.x < 2) sh[threadIdx.x] = 0;
    __syncthreads();
    h = __reduce_add_sync(0xffffffffu, h);
    s = __reduce_add_sync(0xffffffffu, s);
    if ((threadIdx.x & 31) == 0) { atomicAdd(&sh[0], h); atomicAdd(&sh[1], s); }
    __syncthreads();
    if (threadIdx.x == 0) { *holes_out = sh[0]; *snps_out = sh[1]; }
}

bool mmlst_pileup_bitsliced_fits(uint32_t max_row_words);
int launch_pileup_atomic(const PileupArgs& a, cudaStream_t stream);
int launch_pileup_bitsliced(const PileupArgs& a, cudaStream_t stream);
__device__ __forceinline__ uint32_t pileup_n_chunks(const PileupArgs& a) { return a.n_chunks_dev ? *a.n_chunks_dev : a.n_chunks; }

// words of a plane row for a record touching nw contig words: 3 planes, padded to an odd count (0 stays 0)
__host__ __device__ __forceinline__ uint32_t mmlst_row_words(uint32_t nw) {
    const uint32_t rw = 3u * nw;
    return rw + ((rw != 0u && (rw & 1u) == 0u) ? 1u : 0u);
}
__host__ __device__ __forceinline__ uint32_t mmlst_touched_words(uint32_t pos, uint32_t reflen) {
    return reflen ? (((pos & 31u) + reflen + 31u) >> 5) : 0u;
}
