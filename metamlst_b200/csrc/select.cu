// Best-allele selection ON THE DEVICE (replaces the host round trip between stage 1 and stage 2).
//
// Reference semantics (metamlst.py:133-151, 184-206, 213-220, 244):
//   per locus   maxLen = max hit count; localScore = sum(AS) - (maxLen - n) * penalty; avg = round(localScore / n, 1)
//   per locus   chosen = lowest int(allele) among the alleles whose ROUNDED average equals the locus maximum
//   per species processed only if int(detected_loci / loci_in_db * 100) >= nloci; order of species and of loci inside
//               a species = dict insertion order = ascending first passing record (H5)
// H6: Python's round(x, 1) is the correctly rounded decimal (ties on the exact binary value go to the even digit).
// Two rounded values are equal iff their integer tenths T are equal, and T is computed here exactly from the bits of
// the IEEE double x = (double)localScore / (double)n (same correctly rounded division as Python's float division).
#include <stdlib.h>

#include "common.cuh"

namespace {

constexpr unsigned long long T_BIAS = 1ull << 62;

// integer nearest to 10*x, ties to even, computed exactly (x finite)
__device__ __forceinline__ long long round_tenths(double x) {
    const unsigned long long bits = static_cast<unsigned long long>(__double_as_longlong(x));
    const bool neg = bits >> 63;
    const int ex = int((bits >> 52) & 0x7ff);
    unsigned long long m = bits & ((1ull << 52) - 1);
    int e;
    if (ex == 0) { e = -1074; } else { m |= 1ull << 52; e = ex - 1075; }
    unsigned long long t;
    const unsigned long long y = m * 10ull;  // < 2^57
    if (e >= 0) {
        t = (e >= 6) ? 0x3fffffffffffffffull : (y << e);  // |x| >= 2^58: clamp (scores never get there)
    } else {
        const int s = -e;
        if (s > 63) {
            t = 0;  // y < 2^57 <= half
        } else {
            const unsigned long long q = y >> s;
            const unsigned long long rem = y & ((1ull << s) - 1ull);
            const unsigned long long half = 1ull << (s - 1);
            t = q + ((rem > half || (rem == half && (q & 1ull))) ? 1ull : 0ull);
        }
    }
    return neg ? -static_cast<long long>(t) : static_cast<long long>(t);
}

struct SelArgs {
    long long* sum_as; uint32_t* n_hit; uint32_t* first_idx;
    const uint32_t* locus_rows; const uint32_t* locus_start; const uint32_t* allele_num; uint32_t n_ref;
    const uint32_t* species_of_locus; const uint32_t* genes_in_db; uint32_t n_loci, n_species;
    int penalty, nloci_pct;
    const unsigned long long* contig_start; const uint32_t* ref_len; const unsigned long long* db_off;
    uint32_t chunk_records, slots, flags;
    unsigned long long* counters;
    // scratch: per-locus results + the "CTAs done" ticket (left at zero by every call)
    unsigned long long* res_key;  // (allele_num << 32 | row) of the chosen allele, ~0 = locus not detected
    uint32_t* res_first;          // first passing record of the locus
    uint32_t* done;
    // outputs
    uint32_t* header;  // [0]=n_chosen [1]=n_chunks [2]=total_cols [3]=error flags [4]=chunk_records used [6..9]=counters
    uint32_t* chosen_tid; uint32_t* chosen_species; uint32_t* col_off; unsigned long long* db_start;
    mmlst_chunk* chunks; uint32_t max_chunks;
    unsigned long long* tl;  // profiling aid (mmlst_debug_timeline), nullptr = off
    uint32_t warp_final;     // finalize with ONE warp and no CTA barrier when n_loci, n_species <= 32 (mmlst_set_select_warp_finalize)
    uint32_t* chosen_first;  // optional: first passing record of every chosen locus (owner-computes merge across GPUs)
};

__device__ __forceinline__ long long tenths_of(long long score, uint32_t n, uint32_t mx, int penalty) {
    if (n != mx) score -= static_cast<long long>(mx - n) * penalty;
    return round_tenths(__ddiv_rn(static_cast<double>(score), static_cast<double>(n)));
}

constexpr int SEL_THREADS = 256;
constexpr int SEL_R = 4;  // rows per thread held in registers (1024 alleles per locus without a second trip to memory)

// block-wide reductions over 256 threads (8 warps): warp REDUX / shuffles, then one shared-memory round
__device__ __forceinline__ uint32_t block_max_u32(uint32_t v, uint32_t* sh) {
    v = __reduce_max_sync(0xffffffffu, v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    uint32_t r = sh[0];
#pragma unroll
    for (int i = 1; i < SEL_THREADS / 32; ++i) r = max(r, sh[i]);
    return r;
}
__device__ __forceinline__ unsigned long long block_reduce_u64(unsigned long long v, unsigned long long* sh, bool want_max) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long x = __shfl_xor_sync(0xffffffffu, v, o);
        v = want_max ? (x > v ? x : v) : (x < v ? x : v);
    }
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    unsigned long long r = sh[0];
#pragma unroll
    for (int i = 1; i < SEL_THREADS / 32; ++i) { const unsigned long long x = sh[i]; r = want_max ? (x > r ? x : r) : (x < r ? x : r); }
    return r;
}

// Finalization by ONE warp (n_loci <= 32, n_species <= 32: every MLST scheme set a sample is typed against): lane m owns locus m, what the CTA-wide form
// does with nine barriers and shared-memory atomics is done with shuffles, so the serial tail of the launch is two dependent reads plus warp arithmetic.
// Same outputs as the CTA-wide form below, statement for statement (gate, H5 order keys, ranks, column layout, chunk list).
__device__ void finalize_warp(const SelArgs& a, const uint32_t* s_sol, const uint32_t* s_gdb, uint32_t* sm) {
    constexpr uint32_t FULLM = 0xffffffffu;
    const uint32_t lane = threadIdx.x;   // caller: threadIdx.x < 32
    const uint32_t nl = a.n_loci;
    unsigned long long cnt0 = 0, cnt1 = 0;
    if (lane == 0 && a.counters) { cnt0 = __ldcg(a.counters); cnt1 = __ldcg(a.counters + 1); }
    if (lane == 0) *a.done = 0;
    const bool v = lane < nl;
    const unsigned long long ck = v ? __ldcg(a.res_key + lane) : ~0ull;
    const uint32_t lf = v ? __ldcg(a.res_first + lane) : 0xffffffffu;
    const bool det = v && ck != ~0ull;
    const uint32_t tid = static_cast<uint32_t>(ck & 0xffffffffull);
    const uint32_t sp = v ? s_sol[lane] : 0xffffffffu;
    // what hangs off the chosen row: requested now (the per-locus CTAs asked it into the L2), used after the ranking
    unsigned long long q0 = 0, q1 = 0, dbo = 0;
    uint32_t ln = 0;
    if (det) { q0 = a.contig_start[tid]; q1 = a.contig_start[tid + 1]; ln = a.ref_len[tid]; dbo = a.db_off[tid]; }
    tl_mark(a.tl, MMLST_TL_SELECT, 5);
    // per species: detected loci and the first passing record of the species (metamlst.py:181-206)
    uint32_t det_cnt = 0, sp_first = 0xffffffffu;
    for (uint32_t j = 0; j < nl; ++j) {
        const uint32_t spj = __shfl_sync(FULLM, sp, j), lfj = __shfl_sync(FULLM, lf, j);
        const bool dj = __shfl_sync(FULLM, det ? 1u : 0u, j) != 0u;
        if (dj && spj == sp) { ++det_cnt; sp_first = min(sp_first, lfj); }
    }
    uint32_t pass = 0, broken = 0;
    if (det) {
        const uint32_t tot = s_gdb[sp];
        if (a.flags & MMLST_SELECT_LOCAL) pass = 1;
        else if (tot < det_cnt) broken = 1;   // "Database is broken" (metamlst.py:188-190)
        else pass = int((double(det_cnt) / double(tot)) * 100.0) >= a.nloci_pct;   // metamlst.py:206
    }
    uint32_t err = __any_sync(FULLM, broken) ? 1u : 0u;
    const bool kept = det && pass;
    const unsigned long long key = kept ? ((static_cast<unsigned long long>(sp_first) << 32) | lf) + 1ull : 0ull;
    uint32_t rank = 0;
    for (uint32_t j = 0; j < nl; ++j) {
        const unsigned long long k2 = __shfl_sync(FULLM, key, j);
        rank += (k2 != 0ull) && ((k2 < key) || (k2 == key && j < lane));
    }
    const uint32_t nsel = __popc(__ballot_sync(FULLM, kept));
    // output order: lane i takes the locus whose rank is i
    uint32_t* s_inv = sm;   // [32] warp-private from here on (the other warps of the CTA have left)
    if (kept) s_inv[rank] = lane;
    __syncwarp();
    const bool o = lane < nsel;
    const uint32_t src = o ? s_inv[lane] : 0u;
    const uint32_t o_tid = __shfl_sync(FULLM, tid, src), o_sp = __shfl_sync(FULLM, sp, src), o_lf = __shfl_sync(FULLM, lf, src), o_len = __shfl_sync(FULLM, ln, src);
    const unsigned long long o_q0 = __shfl_sync(FULLM, q0, src), o_q1 = __shfl_sync(FULLM, q1, src), o_dbo = __shfl_sync(FULLM, dbo, src);
    const uint32_t o_nrec = o ? static_cast<uint32_t>(o_q1 - o_q0) : 0u;
    unsigned long long totrec = o ? (o_q1 - o_q0) : 0ull;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) totrec += __shfl_xor_sync(FULLM, totrec, d);
    tl_mark(a.tl, MMLST_TL_SELECT, 6);
    uint32_t cr = a.chunk_records;
    if (cr == 0) cr = 512u * mmlst_chunk_tiles(totrec, a.slots);   // same rule as mmlst_chunk_records()
    uint32_t nch_i = 0;
    if (o) { const uint32_t k = (o_nrec + cr - 1) / cr; nch_i = k ? k : 1u; }   // a chosen locus without pileup records still gets one (empty) chunk
    // exclusive prefixes in output order: first column and first chunk of every chosen locus
    uint32_t col_inc = o ? o_len : 0u, ch_inc = nch_i;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t c2 = __shfl_up_sync(FULLM, col_inc, d), h2 = __shfl_up_sync(FULLM, ch_inc, d);
        if (lane >= static_cast<uint32_t>(d)) { col_inc += c2; ch_inc += h2; }
    }
    const uint32_t col_ex = col_inc - (o ? o_len : 0u), ch_ex = ch_inc - nch_i;
    const uint32_t tot_cols = __shfl_sync(FULLM, col_inc, 31), tot_ch = __shfl_sync(FULLM, ch_inc, 31);
    if (tot_ch > a.max_chunks) err |= 2u;
    uint32_t* s_cbase = sm + 32;    // [33]
    uint32_t* s_q0 = s_cbase + 33;  // [32]
    uint32_t* s_nrec = s_q0 + 32;   // [32]
    uint32_t* s_col = s_nrec + 32;  // [32]
    uint32_t* s_len = s_col + 32;   // [32]
    if (o) {
        a.chosen_tid[lane] = o_tid;
        a.chosen_species[lane] = o_sp;
        if (a.chosen_first) a.chosen_first[lane] = o_lf;
        a.db_start[lane] = o_dbo;
        a.col_off[lane] = col_ex;
        s_cbase[lane] = ch_ex; s_q0[lane] = static_cast<uint32_t>(o_q0); s_nrec[lane] = o_nrec; s_col[lane] = col_ex; s_len[lane] = o_len;
    }
    if (lane == 0) {
        a.col_off[nsel] = tot_cols;
        s_cbase[nsel] = tot_ch;
        a.header[0] = nsel; a.header[1] = min(tot_ch, a.max_chunks); a.header[2] = tot_cols; a.header[3] = err; a.header[4] = cr;
        if (a.counters) {  // totalReads / ignoredReads travel with the header; consumed like the tables
            a.header[6] = static_cast<uint32_t>(cnt0); a.header[7] = static_cast<uint32_t>(cnt0 >> 32);
            a.header[8] = static_cast<uint32_t>(cnt1); a.header[9] = static_cast<uint32_t>(cnt1 >> 32);
            if (a.flags & MMLST_SELECT_CONSUME) { a.counters[0] = 0; a.counters[1] = 0; }
        }
    }
    if (lane == 0) { sm[194] = nsel; sm[195] = min(tot_ch, a.max_chunks); sm[196] = cr; }   // for the chunk list, written by the whole CTA
    tl_mark(a.tl, MMLST_TL_SELECT, 7);
}

// chunk descriptors from what finalize_warp left in shared memory (whole CTA, after one barrier): one warp needed 3.0 us for the ~300 of a capped
// configs[1] sample, 256 threads 0.9 us
__device__ void chunk_list_from_warp_layout(const SelArgs& a, const uint32_t* sm) {
    const uint32_t* s_cbase = sm + 32;
    const uint32_t* s_q0 = s_cbase + 33;
    const uint32_t* s_nrec = s_q0 + 32;
    const uint32_t* s_col = s_nrec + 32;
    const uint32_t* s_len = s_col + 32;
    const uint32_t nsel = sm[194], nch = sm[195], cr = sm[196];
    for (uint32_t c = threadIdx.x; c < nch; c += blockDim.x) {
        uint32_t lo = 0, hi = nsel;  // last i with s_cbase[i] <= c
        while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (s_cbase[mid] <= c) lo = mid; else hi = mid; }
        const unsigned long long b0 = s_q0[lo], b1 = b0 + s_nrec[lo];
        const unsigned long long b = b0 + static_cast<unsigned long long>(c - s_cbase[lo]) * cr;
        mmlst_chunk ckk;
        ckk.rec_begin = static_cast<uint32_t>(b);
        ckk.rec_end = static_cast<uint32_t>(b + cr < b1 ? b + cr : b1);
        ckk.col_base = s_col[lo]; ckk.contig_len = s_len[lo]; ckk.plane_delta = 0;
        ckk.reserved[0] = lo;
        ckk.reserved[1] = s_cbase[lo + 1] - s_cbase[lo];
        ckk.reserved[2] = 0;
        a.chunks[c] = ckk;
    }
    tl_mark(a.tl, MMLST_TL_SELECT, 4);
}

// ONE launch for the whole selection.  CTA = one locus: its allele rows (locus_rows[locus_start[l] .. locus_start[l+1]))
// are reduced three times inside the CTA (max hit count -> max rounded average -> lowest allele number), no global
// atomics and no grid barrier.  The last CTA to finish (ticket counter) applies the --nloci gate, orders species and
// loci (H5), lays out the columns and writes the pileup chunk descriptors.
__global__ void __launch_bounds__(SEL_THREADS) sel_locus(const SelArgs a) {
    extern __shared__ __align__(8) uint32_t sm[];
    __shared__ unsigned long long sh64[SEL_THREADS / 32];
    __shared__ uint32_t sh32[SEL_THREADS / 32];
    __shared__ uint32_t s_last;
    const uint32_t l = blockIdx.x;
    tl_mark(a.tl, MMLST_TL_SELECT, 0);
    const uint32_t r0 = a.locus_start[l], r1 = a.locus_start[l + 1];   // constant table: may be read before the predecessor is done
    // Any CTA may turn out to be the last one and finalize: each fetches the two small constant tables the finalization walks (species of a locus,
    // `genes` rows of a species) into shared memory NOW, so that those loads fly under its own reduction instead of opening two dependent round
    // trips to memory at the very end of the launch.
    uint32_t* const s_sol = sm + 10 * a.n_loci + 1 + 3 * a.n_species;  // [n_loci] (behind the finalization arrays)
    uint32_t* const s_gdb = s_sol + a.n_loci;                          // [n_species]
    for (uint32_t i = threadIdx.x; i < a.n_loci; i += blockDim.x) s_sol[i] = a.species_of_locus[i];
    for (uint32_t i = threadIdx.x; i < a.n_species; i += blockDim.x) s_gdb[i] = a.genes_in_db[i];
    pdl_wait();                  // the score tables are complete and visible
    pdl_launch_dependents();     // the pileup CTAs may become resident (they wait for THIS grid before reading the chunk list)
    // The first SEL_R x 256 rows of the locus live in registers: ONE round of independent loads (row id, then hit count /
    // score sum / first index / allele number together), after which the three passes are register arithmetic.  Loci
    // with more rows run the same passes over the remainder from global memory.
    uint32_t tt[SEL_R], nn[SEL_R], an[SEL_R], ff[SEL_R];
    long long ss[SEL_R];
#pragma unroll
    for (int k = 0; k < SEL_R; ++k) {
        const uint32_t i = r0 + k * SEL_THREADS + threadIdx.x;
        tt[k] = (i < r1) ? (a.locus_rows ? a.locus_rows[i] : i) : 0xffffffffu;   // no row list = allele rows already grouped by locus: one trip to memory less
    }
#pragma unroll
    for (int k = 0; k < SEL_R; ++k) {
        const bool v = tt[k] != 0xffffffffu;
        nn[k] = v ? a.n_hit[tt[k]] : 0u;
        ss[k] = v ? a.sum_as[tt[k]] : 0ll;
        ff[k] = v ? a.first_idx[tt[k]] : 0xffffffffu;
        an[k] = v ? a.allele_num[tt[k]] : 0u;
    }
    tl_mark(a.tl, MMLST_TL_SELECT, 1, nn[0] + an[SEL_R - 1]);   // the table rows have arrived
    const uint32_t rest0 = r0 + SEL_R * SEL_THREADS + threadIdx.x;  // rows beyond the register window
    // pass 1: per-locus max hit count and first passing record
    uint32_t mx = 0, fmin = 0xffffffffu;
#pragma unroll
    for (int k = 0; k < SEL_R; ++k)
        if (nn[k]) { mx = max(mx, nn[k]); fmin = min(fmin, ff[k]); }
    for (uint32_t i = rest0; i < r1; i += SEL_THREADS) {
        const uint32_t t = a.locus_rows ? a.locus_rows[i] : i;
        const uint32_t n = a.n_hit[t];
        if (n) { mx = max(mx, n); fmin = min(fmin, a.first_idx[t]); }
    }
    mx = block_max_u32(mx, sh32);
    if (mx) {  // CTA-uniform
        const uint32_t nfmax = block_max_u32(~fmin, sh32);
        // pass 2: maximum rounded average (integer tenths)
        unsigned long long best = 0, tk[SEL_R];
#pragma unroll
        for (int k = 0; k < SEL_R; ++k) {
            tk[k] = nn[k] ? static_cast<unsigned long long>(tenths_of(ss[k], nn[k], mx, a.penalty)) + T_BIAS : 0ull;
            best = tk[k] > best ? tk[k] : best;
        }
        for (uint32_t i = rest0; i < r1; i += SEL_THREADS) {
            const uint32_t t = a.locus_rows ? a.locus_rows[i] : i;
            const uint32_t n = a.n_hit[t];
            if (n) { const unsigned long long v = static_cast<unsigned long long>(tenths_of(a.sum_as[t], n, mx, a.penalty)) + T_BIAS; best = v > best ? v : best; }
        }
        best = block_reduce_u64(best, sh64, true);
        // pass 3: lowest allele number among the alleles that reach it (then lowest row)
        unsigned long long key = ~0ull;
#pragma unroll
        for (int k = 0; k < SEL_R; ++k) {
            if (!nn[k]) continue;
            if (tk[k] == best) {
                const unsigned long long kk = (static_cast<unsigned long long>(an[k]) << 32) | tt[k];
                key = kk < key ? kk : key;
            }
            if (a.flags & MMLST_SELECT_CONSUME) { a.sum_as[tt[k]] = 0; a.n_hit[tt[k]] = 0; a.first_idx[tt[k]] = 0xffffffffu; }
        }
        for (uint32_t i = rest0; i < r1; i += SEL_THREADS) {
            const uint32_t t = a.locus_rows ? a.locus_rows[i] : i;
            const uint32_t n = a.n_hit[t];
            if (!n) continue;
            if (static_cast<unsigned long long>(tenths_of(a.sum_as[t], n, mx, a.penalty)) + T_BIAS == best) {
                const unsigned long long k = (static_cast<unsigned long long>(a.allele_num[t]) << 32) | t;
                key = k < key ? k : key;
            }
            if (a.flags & MMLST_SELECT_CONSUME) { a.sum_as[t] = 0; a.n_hit[t] = 0; a.first_idx[t] = 0xffffffffu; }
        }
        key = block_reduce_u64(key, sh64, false);
        if (threadIdx.x == 0) {
            a.res_key[l] = key; a.res_first[l] = ~nfmax;
            // what the finalizing CTA will read for this locus's chosen row (record range, BAM LN, DB offset) is asked into the L2 now: it arrives while
            // the ticket travels, instead of costing the finalizer a trip to HBM on its serial path
            const uint32_t row = static_cast<uint32_t>(key & 0xffffffffull);
            if (key != ~0ull && row < a.n_ref) {
                asm volatile("prefetch.global.L2 [%0];" ::"l"(a.contig_start + row));
                asm volatile("prefetch.global.L2 [%0];" ::"l"(a.contig_start + row + 1));
                asm volatile("prefetch.global.L2 [%0];" ::"l"(a.ref_len + row));
                asm volatile("prefetch.global.L2 [%0];" ::"l"(a.db_off + row));
            }
        }
    } else if (threadIdx.x == 0) {
        a.res_key[l] = ~0ull; a.res_first[l] = 0xffffffffu;
    }
    // ticket: the last CTA finalizes
    __syncthreads();
    tl_mark(a.tl, MMLST_TL_SELECT, 2);   // the locus is reduced
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = (atomicAdd(a.done, 1u) == gridDim.x - 1u);
    }
    __syncthreads();
    tl_mark(a.tl, MMLST_TL_SELECT, 3, s_last);   // the ticket is back
    if (!s_last) return;
    __threadfence();
    if (a.warp_final && a.n_loci <= 32u && a.n_species <= 32u) {
        if (threadIdx.x < 32) finalize_warp(a, s_sol, s_gdb, sm);
        __syncthreads();   // the layout of the chosen loci is in shared memory
        chunk_list_from_warp_layout(a, sm);
        return;
    }

    // ---- last CTA: finalize.  Two dependent round trips to memory: the per-locus results, then what hangs off the chosen rows
    // (record range, BAM LN, DB offset); everything else comes from shared memory.
    unsigned long long* s_key = reinterpret_cast<unsigned long long*>(sm);   // [n_loci] order key of kept loci, 0 = not kept
    uint32_t* s_tid = sm + 2 * a.n_loci;                                     // [n_loci] chosen row of the locus
    uint32_t* s_cbase = s_tid + a.n_loci;                                    // [n_loci + 1]
    uint32_t* s_len = s_cbase + a.n_loci + 1;                                // [n_loci] BAM LN of chosen rows, output order
    uint32_t* s_nch = s_len + a.n_loci;                                      // [n_loci] chunks of chosen rows, output order
    uint32_t* s_lfirst = s_nch + a.n_loci;                                   // [n_loci]
    uint32_t* s_q0 = s_lfirst + a.n_loci;                                    // [n_loci] first pileup record of chosen rows, output order
    uint32_t* s_col = s_q0 + a.n_loci;                                       // [n_loci] first column of chosen rows, output order
    uint32_t* s_nrec = s_col + a.n_loci;                                     // [n_loci] pileup records of chosen rows, output order
    uint32_t* s_detected = s_nrec + a.n_loci;                                // [n_species]
    uint32_t* s_first = s_detected + a.n_species;                            // [n_species]
    uint32_t* s_pass = s_first + a.n_species;                                // [n_species]
    __shared__ uint32_t s_n, s_err, s_cr, s_totch;
    __shared__ unsigned long long s_totrec;
    unsigned long long cnt0 = 0, cnt1 = 0;
    if (threadIdx.x == 0 && a.counters) { cnt0 = __ldcg(a.counters); cnt1 = __ldcg(a.counters + 1); }   // in flight under everything below
    for (uint32_t i = threadIdx.x; i < a.n_species; i += blockDim.x) { s_detected[i] = 0; s_first[i] = 0xffffffffu; }
    if (threadIdx.x == 0) { s_n = 0; s_err = 0; s_totrec = 0; *a.done = 0; }
    __syncthreads();
    for (uint32_t m = threadIdx.x; m < a.n_loci; m += blockDim.x) {
        const unsigned long long ck = __ldcg(a.res_key + m);
        const uint32_t lf = __ldcg(a.res_first + m);
        s_tid[m] = static_cast<uint32_t>(ck & 0xffffffffull);
        s_lfirst[m] = lf;
        s_key[m] = (ck != ~0ull) ? 1ull : 0ull;  // provisional: detected
        if (ck != ~0ull) {
            const uint32_t sp = s_sol[m];
            atomicAdd(s_detected + sp, 1u);
            atomicMin(s_first + sp, lf);
        }
    }
    __syncthreads();
    tl_mark(a.tl, MMLST_TL_SELECT, 5);   // last CTA: per-locus results read back
    for (uint32_t sp = threadIdx.x; sp < a.n_species; sp += blockDim.x) {
        const uint32_t det = s_detected[sp], tot = s_gdb[sp];
        uint32_t pass = 0;
        if (det) {
            if (a.flags & MMLST_SELECT_LOCAL) pass = 1;  // this GPU owns a subset of the loci: the gate is applied after the merge
            else if (tot < det) atomicOr(&s_err, 1u);  // "Database is broken" (metamlst.py:188-190)
            else pass = int((double(det) / double(tot)) * 100.0) >= a.nloci_pct;  // metamlst.py:206
        }
        s_pass[sp] = pass;
    }
    __syncthreads();
    // order key of every kept locus: (species first record, locus first record) + 1 so that 0 means "not kept"
    for (uint32_t m = threadIdx.x; m < a.n_loci; m += blockDim.x) {
        unsigned long long key = 0;
        if (s_key[m]) {
            const uint32_t sp = s_sol[m];
            if (s_pass[sp]) { key = ((static_cast<unsigned long long>(s_first[sp]) << 32) | s_lfirst[m]) + 1ull; atomicAdd(&s_n, 1u); }
        }
        s_key[m] = key;
    }
    __syncthreads();
    for (uint32_t m = threadIdx.x; m < a.n_loci; m += blockDim.x) {
        const unsigned long long key = s_key[m];
        if (!key) continue;
        const uint32_t tid = s_tid[m];
        // the only loads that depend on the chosen row: issued together, before the rank is counted
        const unsigned long long q0 = a.contig_start[tid], q1 = a.contig_start[tid + 1];
        const uint32_t ln = a.ref_len[tid];
        const unsigned long long dbo = a.db_off[tid];
        uint32_t rank = 0;
        for (uint32_t j = 0; j < a.n_loci; ++j) {
            const unsigned long long k2 = s_key[j];
            rank += (k2 != 0ull) && ((k2 < key) || (k2 == key && j < m));
        }
        a.chosen_tid[rank] = tid;
        a.chosen_species[rank] = s_sol[m];
        if (a.chosen_first) a.chosen_first[rank] = s_lfirst[m];
        a.db_start[rank] = dbo;
        s_len[rank] = ln;
        s_q0[rank] = static_cast<uint32_t>(q0);
        s_nrec[rank] = static_cast<uint32_t>(q1 - q0);
        atomicAdd(&s_totrec, q1 - q0);
    }
    __syncthreads();
    tl_mark(a.tl, MMLST_TL_SELECT, 6);   // last CTA: what hangs off the chosen rows has arrived, loci ranked
    const uint32_t nsel = s_n;
    if (threadIdx.x == 0) {
        uint32_t cr = a.chunk_records;
        if (cr == 0) cr = 512u * mmlst_chunk_tiles(s_totrec, a.slots);  // same rule as mmlst_chunk_records()
        s_cr = cr;
    }
    __syncthreads();
    const uint32_t cr = s_cr;
    for (uint32_t i = threadIdx.x; i < nsel; i += blockDim.x) {
        const uint32_t k = (s_nrec[i] + cr - 1) / cr;
        s_nch[i] = k ? k : 1u;   // a chosen locus without pileup records still gets one (empty) chunk: the fused consensus hangs off the last chunk of a locus
    }
    __syncthreads();
    if (threadIdx.x == 0) {  // exclusive prefixes over shared memory (no dependent global loads)
        uint32_t col = 0, nch = 0;
        for (uint32_t i = 0; i < nsel; ++i) {
            a.col_off[i] = col;
            s_col[i] = col;
            s_cbase[i] = nch;
            nch += s_nch[i];
            col += s_len[i];
        }
        a.col_off[nsel] = col;
        s_cbase[nsel] = nch;
        s_totch = nch;
        if (nch > a.max_chunks) s_err |= 2u;
        a.header[0] = nsel; a.header[1] = min(nch, a.max_chunks); a.header[2] = col; a.header[3] = s_err; a.header[4] = cr;
        if (a.counters) {  // totalReads / ignoredReads travel with the header; consumed like the tables
            a.header[6] = static_cast<uint32_t>(cnt0); a.header[7] = static_cast<uint32_t>(cnt0 >> 32);
            a.header[8] = static_cast<uint32_t>(cnt1); a.header[9] = static_cast<uint32_t>(cnt1 >> 32);
            if (a.flags & MMLST_SELECT_CONSUME) { a.counters[0] = 0; a.counters[1] = 0; }
        }
    }
    __syncthreads();
    tl_mark(a.tl, MMLST_TL_SELECT, 7);   // last CTA: header and column layout written
    const uint32_t nch = min(s_totch, a.max_chunks);
    for (uint32_t c = threadIdx.x; c < nch; c += blockDim.x) {
        uint32_t lo = 0, hi = nsel;  // last i with s_cbase[i] <= c
        while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (s_cbase[mid] <= c) lo = mid; else hi = mid; }
        const unsigned long long q0 = s_q0[lo], q1 = q0 + s_nrec[lo];
        const unsigned long long b = q0 + static_cast<unsigned long long>(c - s_cbase[lo]) * cr;
        mmlst_chunk ck;
        ck.rec_begin = static_cast<uint32_t>(b);
        ck.rec_end = static_cast<uint32_t>(b + cr < q1 ? b + cr : q1);
        ck.col_base = s_col[lo]; ck.contig_len = s_len[lo]; ck.plane_delta = 0;
        ck.reserved[0] = lo;                              // chosen locus (output order) the chunk belongs to
        ck.reserved[1] = s_cbase[lo + 1] - s_cbase[lo];   // chunks of that locus
        ck.reserved[2] = 0;
        a.chunks[c] = ck;
    }
    tl_mark(a.tl, MMLST_TL_SELECT, 4);   // last CTA: finalization written
}

}  // namespace

static int g_select_warp = -1;
static int select_warp() {
    if (g_select_warp < 0) {
        const char* e = getenv("MMLST_SELECT_WARP");
        g_select_warp = e ? (e[0] == '1') : MMLST_SELECT_WARP_DEFAULT;
    }
    return g_select_warp;
}
// see include/mmlst.h
extern "C" int mmlst_set_select_warp_finalize(int on) {
    const int prev = select_warp();
    if (on == 0 || on == 1) g_select_warp = on;
    return prev;
}

// Dynamic shared memory of one selection launch: the finalization arrays (10 n_loci + 1 + 3 n_species words, see the kernel) + the prefetched
// species_of_locus / genes_in_db, and never less than the 193 words the one-warp finalizer lays out whatever n_loci is.
static size_t select_smem_bytes(uint32_t n_loci, uint32_t n_species) {
    const size_t smem = sizeof(uint32_t) * (static_cast<size_t>(n_loci) * 11 + 1 + 4 * static_cast<size_t>(n_species)) + 16;
    return smem < 200 * sizeof(uint32_t) ? 200 * sizeof(uint32_t) : smem;
}

// see common.cuh
int mmlst_select_fits(uint32_t n_loci, uint32_t n_species, const char* who) {
    static int max_dynamic_by_device[MMLST_MAX_DEVICES] = {0};   // 0 = not asked yet
    int& max_dynamic = max_dynamic_by_device[mmlst_current_device()];
    if (max_dynamic == 0) {
        int dev = 0, optin = 0;
        CUDA_TRY(cudaGetDevice(&dev));
        CUDA_TRY(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
        cudaFuncAttributes fa;
        CUDA_TRY(cudaFuncGetAttributes(&fa, sel_locus));
        max_dynamic = optin - static_cast<int>(fa.sharedSizeBytes);   // the kernel's static shared memory counts against the same per-block limit
    }
    const size_t smem = select_smem_bytes(n_loci, n_species);
    if (smem > static_cast<size_t>(max_dynamic)) {
        mmlst_set_error("%s: %u loci / %u species need %zu bytes of shared memory per block for the selection, the device allows %d", who, n_loci,
                        n_species, smem, max_dynamic);
        return MMLST_E_RANGE;
    }
    return MMLST_OK;
}

// see include/mmlst.h
extern "C" int mmlst_select_dev(int64_t* sum_as, uint32_t* n_hit, uint32_t* first_idx, const uint32_t* locus_rows,
                                const uint32_t* locus_start, const uint32_t* allele_num, uint32_t n_ref,
                                const uint32_t* species_of_locus, const uint32_t* genes_in_db, uint32_t n_loci, uint32_t n_species,
                                int penalty, int nloci_pct, const uint64_t* contig_start, const uint32_t* ref_len,
                                const uint64_t* db_off, uint32_t chunk_records, void* scratch, size_t scratch_bytes,
                                uint32_t* header, uint32_t* chosen_tid, uint32_t* chosen_species, uint32_t* col_off,
                                uint64_t* db_start, mmlst_chunk* chunks, uint32_t max_chunks, uint32_t flags,
                                uint64_t* counters, uint32_t* chosen_first, void* stream) {
    if (!sum_as || !n_hit || !first_idx || !locus_start || !allele_num || !species_of_locus || !genes_in_db ||
        !contig_start || !ref_len || !db_off || !scratch || !header || !chosen_tid || !chosen_species || !col_off || !db_start || !chunks) {
        mmlst_set_error("mmlst_select_dev: null pointer");
        return MMLST_E_ARG;
    }
    if (n_loci == 0) { mmlst_set_error("mmlst_select_dev: no loci"); return MMLST_E_ARG; }
    if (n_loci > 8192 || n_species > 4096) { mmlst_set_error("mmlst_select_dev: more than 8192 loci / 4096 species"); return MMLST_E_RANGE; }
    if (const int rc = mmlst_select_fits(n_loci, n_species, "mmlst_select_dev")) return rc;
    const size_t need = static_cast<size_t>(n_loci) * 12 + 16;
    if (scratch_bytes < need || (reinterpret_cast<uintptr_t>(scratch) & 7)) { mmlst_set_error("mmlst_select_dev: scratch needs %zu bytes, 8-byte aligned", need); return MMLST_E_ARG; }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    // scratch layout: res_key u64[n_loci] | res_first u32[n_loci] | (pad to 8) done u32
    uint8_t* p = static_cast<uint8_t*>(scratch);
    SelArgs a;
    a.sum_as = reinterpret_cast<long long*>(sum_as); a.n_hit = n_hit; a.first_idx = first_idx;
    a.locus_rows = locus_rows; a.locus_start = locus_start;
    a.allele_num = allele_num; a.n_ref = n_ref; a.species_of_locus = species_of_locus; a.genes_in_db = genes_in_db;
    a.n_loci = n_loci; a.n_species = n_species; a.penalty = penalty; a.nloci_pct = nloci_pct;
    a.contig_start = reinterpret_cast<const unsigned long long*>(contig_start); a.ref_len = ref_len;
    a.db_off = reinterpret_cast<const unsigned long long*>(db_off); a.chunk_records = chunk_records;
    a.flags = flags; a.counters = reinterpret_cast<unsigned long long*>(counters);
    a.res_key = reinterpret_cast<unsigned long long*>(p);
    a.res_first = reinterpret_cast<uint32_t*>(a.res_key + n_loci);
    a.done = reinterpret_cast<uint32_t*>(p + ((static_cast<size_t>(n_loci) * 12 + 7) & ~static_cast<size_t>(7)));
    a.slots = static_cast<uint32_t>(mmlst_num_sms()) * MMLST_CHUNKS_PER_SM;
    a.header = header; a.chosen_tid = chosen_tid; a.chosen_species = chosen_species; a.col_off = col_off;
    a.db_start = reinterpret_cast<unsigned long long*>(db_start); a.chunks = chunks; a.max_chunks = max_chunks;
    a.chosen_first = chosen_first;
    a.tl = mmlst_timeline_buffer();
    a.warp_final = select_warp() ? 1u : 0u;
    if (!(flags & MMLST_SELECT_SCRATCH_CLEAN)) CUDA_TRY(cudaMemsetAsync(a.done, 0, 4, s));
    const size_t smem = select_smem_bytes(n_loci, n_species);
    static size_t configured_by_device[MMLST_MAX_DEVICES] = {0};  // 0 = not asked yet
    size_t& configured = configured_by_device[mmlst_current_device()];
    if (configured == 0) {   // what every kernel starts with: 48 KB less its static shared memory
        cudaFuncAttributes fa;
        CUDA_TRY(cudaFuncGetAttributes(&fa, sel_locus));
        configured = fa.maxDynamicSharedSizeBytes;
    }
    if (smem > configured) {
        CUDA_TRY(cudaFuncSetAttribute(sel_locus, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
        configured = smem;
    }
    static bool carve[MMLST_MAX_DEVICES] = {false};
    mmlst_prefer_max_shared(sel_locus, carve);
    CUDA_TRY(mmlst_launch_dependent(sel_locus, dim3(n_loci), dim3(SEL_THREADS), smem, s, a));
    return MMLST_OK;
}
