// Stage 3: closest allele by zip-truncated Hamming distance (replaces metaMLST_functions.py:230-234 driven by
// metamlst-merge.py:174-181).  2-bit codes stored as two bit-planes => one 32-base mismatch mask costs
// XOR + LOP3 ((qh^rh)|(ql^rl)) and one POPC.  thread = DB row (planes held in registers, loaded coalesced from
// 32-row word-major tiles), CTA = 256 rows, queries staged in shared memory and broadcast with 128-bit LDS;
// per query a warp-level REDUX.MIN of (distance<<8 | row-in-CTA), then one 64-bit atomicMin per (CTA, query) of
// (distance<<32 | row) which also resolves ties to the lowest row.  Sequences flagged with bit 15 of their length hold
// non-ACGT characters and are left to the exact path (hamming_exact.cu, H9).
#include "common.cuh"

namespace {

constexpr int kRowsPerCta = 128;
constexpr int kQChunk = 64;
constexpr int kQSplit = 2048;  // queries handled by one CTA (gridDim.z splits longer query ranges)

struct HamArgs {
    const uint32_t* db_hi; const uint32_t* db_lo; const uint16_t* row_len; uint32_t n_rows;
    const uint32_t* q_hi; const uint32_t* q_lo; const uint16_t* q_len; uint32_t n_q;
    const uint32_t* blocks; uint32_t n_blocks; uint32_t row_index_base;
    unsigned long long* best;
};

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(static_cast<uint32_t>(__cvta_generic_to_shared(smem_dst))), "l"(gsrc) : "memory");
}
__device__ __forceinline__ uint32_t prefix_mask(int bits) {  // low `bits` bits set, clamped to [0, 32]: VIMNMX + BMSK
    uint32_t m;
    asm("bmsk.clamp.b32 %0, 0, %1;" : "=r"(m) : "r"(static_cast<uint32_t>(max(bits, 0))));
    return m;
}

// POPC runs on the XU pipe at 16 lanes/clk/SM (8 issue cycles per warp instruction and SM sub-partition) while a
// LOP3 costs 2: three mismatch words are folded by one carry-save adder (2 LOP3) into ones + twos, so 3 words cost
// 2 POPC instead of 3 and the two pipes carry about the same load (~5.3 cycles per word each).
__device__ __forceinline__ uint32_t popc3(uint32_t a, uint32_t b, uint32_t c) {
    const uint32_t u = a ^ b;
    const uint32_t ones = u ^ c;
    const uint32_t twos = (a & b) | (u & c);
    return __popc(ones) + 2u * __popc(twos);
}

template <int W>
__global__ void __launch_bounds__(kRowsPerCta, 5) hamming_min_kernel(const HamArgs a) {
    static_assert(W % 6 == 0 || W == 8 || W == 16 || W == 32, "W: 8, 16, 24 or 32 words per plane");
    constexpr int U = (W % 6 == 0) ? 6 : 4;  // words per unit: plain / masked / skipped is decided per unit (CTA-uniform)
    constexpr int NU = W / U;
    const uint32_t* blk = a.blocks + 4 * blockIdx.y;
    const uint32_t q_begin = blk[0], q_end = blk[1], r_begin = blk[2], r_end = blk[3];
    // row tiles start AT the block's first row (not at a 32-row tile boundary): only the last CTA of a block is ragged
    const uint32_t row0 = r_begin + blockIdx.x * kRowsPerCta;
    if (row0 >= r_end) return;
    const uint32_t qs = q_begin + blockIdx.z * kQSplit;
    if (qs >= q_end) return;
    const uint32_t qe = min(q_end, qs + kQSplit);

    __shared__ __align__(16) uint32_t sq_hi[2][kQChunk + 2][W];
    __shared__ __align__(16) uint32_t sq_lo[2][kQChunk + 2][W];
    __shared__ uint32_t sq_len[2][kQChunk + 2];
    __shared__ uint32_t part[kRowsPerCta / 32][kQChunk + 1];
    __shared__ uint32_t s_minl, s_maxl;

    const uint32_t lane = threadIdx.x & 31u, wib = threadIdx.x >> 5;
    const uint32_t row = row0 + threadIdx.x;
    bool valid = (row < r_end) && (row < a.n_rows);
    uint32_t rh[W], rl[W];
    uint32_t rlen = 0;
    {
        const uint32_t tile = row >> 5, r = row & 31u;
        const bool inb = row < ((a.n_rows + 31u) & ~31u);
#pragma unroll
        for (int w = 0; w < W; ++w) {
            rh[w] = inb ? a.db_hi[(static_cast<size_t>(tile) * W + w) * 32 + r] : 0u;
            rl[w] = inb ? a.db_lo[(static_cast<size_t>(tile) * W + w) * 32 + r] : 0u;
        }
        if (valid) {
            const uint32_t raw = a.row_len[row];
            rlen = raw & 0x7fffu;
            valid = !(raw & 0x8000u);  // bit 15: row holds non-ACGT characters -> exact path (hamming_exact.cu, H9)
        }
    }
    // query staging is software-pipelined with cp.async (LDGSTS, no registers): chunk c+1 travels global -> the other
    // shared-memory buffer while chunk c is compared, and the first chunk is requested together with the row planes so
    // that a CTA pays ONE memory round trip before computing
    auto fetch = [&](uint32_t qc, uint32_t buf) {
        const uint32_t nq = min(uint32_t(kQChunk), qe - qc);
        for (uint32_t i = threadIdx.x; i < nq * (W / 4); i += kRowsPerCta) {
            const uint32_t qi = i / (W / 4), w4 = i % (W / 4);
            cp_async16(&sq_hi[buf][qi][4 * w4], a.q_hi + static_cast<size_t>(qc + qi) * W + 4 * w4);
            cp_async16(&sq_lo[buf][qi][4 * w4], a.q_lo + static_cast<size_t>(qc + qi) * W + 4 * w4);
        }
        if (threadIdx.x < nq) sq_len[buf][threadIdx.x] = a.q_len[qc + threadIdx.x];
        if ((nq & 1u) && threadIdx.x < W) { sq_hi[buf][nq][threadIdx.x] = 0u; sq_lo[buf][nq][threadIdx.x] = 0u; }  // phantom partner of an odd chunk
        if ((nq & 1u) && threadIdx.x == 0) sq_len[buf][nq] = 0u;
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    auto commit = [&]() { asm volatile("cp.async.wait_group 0;" ::: "memory"); };
    fetch(qs, 0);
    if (threadIdx.x == 0) { s_minl = 0xffffffffu; s_maxl = 0u; }
    __syncthreads();
    {
        const uint32_t mn = __reduce_min_sync(0xffffffffu, valid ? rlen : 0xffffffffu);
        const uint32_t mx = __reduce_max_sync(0xffffffffu, valid ? rlen : 0u);
        if (lane == 0) { atomicMin(&s_minl, mn); atomicMax(&s_maxl, mx); }
    }
    commit();
    __syncthreads();
    const uint32_t cta_minl = s_minl, cta_maxl = s_maxl;

    uint32_t buf = 0;
    for (uint32_t qc = qs; qc < qe; qc += kQChunk, buf ^= 1u) {
        const uint32_t nq = min(uint32_t(kQChunk), qe - qc);
        if (qc + kQChunk < qe) fetch(qc + kQChunk, buf ^ 1u);  // in flight during the compare loop below
        // two queries per iteration: independent accumulators double the instruction-level parallelism and share the
        // unit classification (the union of the two queries' classes; masking a plain word is always correct)
        for (uint32_t qi = 0; qi < nq; qi += 2) {
            const uint32_t qlen0 = sq_len[buf][qi] & 0x7fffu, qlen1 = sq_len[buf][qi + 1] & 0x7fffu;
            const bool two = qi + 1 < nq;
            // CTA-uniform unit classes (sequences are zero-padded, H9 zip truncation):
            //   unit <  lo_u : inside min(len_q, len_r) for every row of the CTA      -> plain XOR/OR, carry-save, POPC
            //   unit >= hi_u : beyond max(len_q, len_r) for every row: both are zero  -> skipped
            //   between      : every mismatch word masked to min(len_q, len_r) of the pair
            const uint32_t qmin = two ? min(qlen0, qlen1) : qlen0, qmax = max(qlen0, qlen1);
            const uint32_t lo_u = (min(cta_minl, qmin) >> 5) / U;
            const uint32_t hi_u = (((max(cta_maxl, qmax) + 31u) >> 5) + U - 1) / U;
            const int minlen0 = static_cast<int>(min(qlen0, rlen)), minlen1 = static_cast<int>(min(qlen1, rlen));
            uint32_t acc0 = 0, acc1 = 0;
#pragma unroll
            for (int u = 0; u < NU; ++u) {
                if (uint32_t(u) >= hi_u) break;  // uniform
                uint32_t m0[U], m1[U];
#pragma unroll
                for (int k = 0; k < U; ++k) {
                    const int w = U * u + k;
                    m0[k] = (rh[w] ^ sq_hi[buf][qi][w]) | (rl[w] ^ sq_lo[buf][qi][w]);
                    m1[k] = (rh[w] ^ sq_hi[buf][qi + 1][w]) | (rl[w] ^ sq_lo[buf][qi + 1][w]);
                }
                if (uint32_t(u) >= lo_u) {  // uniform
#pragma unroll
                    for (int k = 0; k < U; ++k) {
                        const int w = U * u + k;
                        m0[k] &= prefix_mask(minlen0 - 32 * w);
                        m1[k] &= prefix_mask(minlen1 - 32 * w);
                    }
                }
                if (U == 6) {
                    acc0 += popc3(m0[0], m0[1], m0[2]) + popc3(m0[3], m0[4], m0[5]);
                    acc1 += popc3(m1[0], m1[1], m1[2]) + popc3(m1[3], m1[4], m1[5]);
                } else {
                    acc0 += popc3(m0[0], m0[1], m0[2]) + __popc(m0[3]);
                    acc1 += popc3(m1[0], m1[1], m1[2]) + __popc(m1[3]);
                }
            }
            uint32_t key0 = valid ? ((acc0 << 8) | threadIdx.x) : 0xffffffffu;
            uint32_t key1 = valid ? ((acc1 << 8) | threadIdx.x) : 0xffffffffu;
            key0 = __reduce_min_sync(0xffffffffu, key0);
            key1 = __reduce_min_sync(0xffffffffu, key1);
            if (lane == 0) { part[wib][qi] = key0; part[wib][qi + 1] = key1; }
        }
        __syncthreads();
        if (threadIdx.x < nq) {
            uint32_t key = 0xffffffffu;
#pragma unroll
            for (int w = 0; w < kRowsPerCta / 32; ++w) key = min(key, part[w][threadIdx.x]);
            if (key != 0xffffffffu && !(sq_len[buf][threadIdx.x] & 0x8000u)) {  // flagged queries: exact path only
                const unsigned long long v = (static_cast<unsigned long long>(key >> 8) << 32) |
                                             static_cast<unsigned long long>(a.row_index_base + row0 + (key & 255u));
                atomicMin(a.best + qc + threadIdx.x, v);
            }
        }
        __syncthreads();  // everyone is done with this chunk's queries and partial minima
        if (qc + kQChunk < qe) { commit(); __syncthreads(); }
    }
}

// Any plane width (rows longer than 1024 bases, or widths the tiled kernel has no instance for): thread = DB row, queries of the
// block in turn, word by word from global memory.  Same best[] contract; an order of magnitude slower -- MLST loci are 400-550 bp, this
// is here so that no input is refused.
__global__ void __launch_bounds__(kRowsPerCta) hamming_min_wide_kernel(const HamArgs a, uint32_t W) {
    const uint32_t* blk = a.blocks + 4 * blockIdx.y;
    const uint32_t q_begin = blk[0], q_end = blk[1], r_begin = blk[2], r_end = blk[3];
    const uint32_t row = r_begin + blockIdx.x * kRowsPerCta + threadIdx.x;
    const bool live = row < r_end && row < a.n_rows;
    const uint32_t rl_raw = live ? a.row_len[row] : 0x8000u;
    const size_t tb = static_cast<size_t>(row >> 5) * W * 32 + (row & 31u);
    for (uint32_t q = q_begin; q < q_end; ++q) {
        const uint32_t ql_raw = a.q_len[q];
        unsigned long long key = ~0ull;
        if (live && !(rl_raw & 0x8000u) && !(ql_raw & 0x8000u)) {
            const uint32_t m = min(rl_raw, ql_raw);
            uint32_t d = 0;
            for (uint32_t w = 0; 32 * w < m; ++w) {
                uint32_t x = (a.db_hi[tb + static_cast<size_t>(w) * 32] ^ a.q_hi[static_cast<size_t>(q) * W + w]) |
                             (a.db_lo[tb + static_cast<size_t>(w) * 32] ^ a.q_lo[static_cast<size_t>(q) * W + w]);
                const uint32_t left = m - 32 * w;
                if (left < 32) x &= (1u << left) - 1u;
                d += __popc(x);
            }
            key = (static_cast<unsigned long long>(d) << 32) | (row + a.row_index_base);
        }
        // warp minimum, one atomic per (warp, query)
        for (int o = 16; o > 0; o >>= 1) { const unsigned long long x = __shfl_xor_sync(0xffffffffu, key, o); key = x < key ? x : key; }
        if ((threadIdx.x & 31) == 0 && key != ~0ull) atomicMin(a.best + q, key);
    }
}

template <int W>
int launch(const HamArgs& a, uint32_t max_rows, uint32_t max_q, cudaStream_t s) {
    dim3 grid((max_rows + kRowsPerCta - 1) / kRowsPerCta, a.n_blocks, (max_q + kQSplit - 1) / kQSplit);
    hamming_min_kernel<W><<<grid, kRowsPerCta, 0, s>>>(a);
    return mmlst_cuda_fail(cudaGetLastError(), "hamming_min_kernel");
}

}  // namespace

// max_block_rows / max_block_queries size the grid (blocks with fewer rows exit early)
extern "C" int mmlst_hamming_min_dev2(const uint32_t* db_hi, const uint32_t* db_lo, const uint16_t* row_len, uint32_t n_rows,
                                      uint32_t W, const uint32_t* q_hi, const uint32_t* q_lo, const uint16_t* q_len,
                                      uint32_t n_q, const uint32_t* blocks, uint32_t n_blocks, uint32_t max_block_rows,
                                      uint32_t max_block_queries, uint32_t row_index_base, unsigned long long* best,
                                      void* stream) {
    if (n_q == 0 || n_rows == 0 || n_blocks == 0) return MMLST_OK;
    if (!db_hi || !db_lo || !row_len || !q_hi || !q_lo || !q_len || !blocks || !best) {
        mmlst_set_error("mmlst_hamming_min_dev: null pointer");
        return MMLST_E_ARG;
    }
    if ((reinterpret_cast<uintptr_t>(q_hi) & 15) || (reinterpret_cast<uintptr_t>(q_lo) & 15)) {
        mmlst_set_error("mmlst_hamming_min_dev: query planes must be 16-byte aligned");
        return MMLST_E_ARG;
    }
    // 0 = not known: every block may span all rows / all queries (as the any-width path reads it).  A call whose blocks are all
    // empty then launches CTAs that exit at once and leaves best[] at the caller's "no row" preset, instead of a grid of size 0.
    if (max_block_rows == 0) max_block_rows = n_rows;
    if (max_block_queries == 0) max_block_queries = n_q;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    for (uint32_t b0 = 0; b0 < n_blocks; b0 += 65535u) {   // gridDim.y holds 65535 blocks: more go out in slices
        const uint32_t nb = n_blocks - b0 < 65535u ? n_blocks - b0 : 65535u;
        HamArgs a{db_hi, db_lo, row_len, n_rows, q_hi, q_lo, q_len, n_q, blocks + 4 * static_cast<size_t>(b0), nb, row_index_base, best};
        int rc;
        switch (W) {
            case 8: rc = launch<8>(a, max_block_rows, max_block_queries, s); break;
            case 16: rc = launch<16>(a, max_block_rows, max_block_queries, s); break;
            case 24: rc = launch<24>(a, max_block_rows, max_block_queries, s); break;
            case 32: rc = launch<32>(a, max_block_rows, max_block_queries, s); break;
            default: {
                if (W == 0) { mmlst_set_error("mmlst_hamming_min_dev: W = 0"); return MMLST_E_ARG; }
                const uint32_t mr = max_block_rows ? max_block_rows : n_rows;
                hamming_min_wide_kernel<<<dim3((mr + kRowsPerCta - 1) / kRowsPerCta, nb), kRowsPerCta, 0, s>>>(a, W);
                rc = mmlst_cuda_fail(cudaGetLastError(), "hamming_min_wide_kernel");
            }
        }
        if (rc != MMLST_OK) return rc;
    }
    return MMLST_OK;
}

extern "C" int mmlst_hamming_min_dev(const uint32_t* db_hi, const uint32_t* db_lo, const uint16_t* row_len, uint32_t n_rows,
                                     uint32_t W, const uint32_t* q_hi, const uint32_t* q_lo, const uint16_t* q_len,
                                     uint32_t n_q, const uint32_t* blocks, uint32_t n_blocks, uint32_t row_index_base,
                                     unsigned long long* best, void* stream) {
    // conservative grid: every block may span all rows / all queries
    return mmlst_hamming_min_dev2(db_hi, db_lo, row_len, n_rows, W, q_hi, q_lo, q_len, n_q, blocks, n_blocks, n_rows, n_q,
                                  row_index_base, best, stream);
}
