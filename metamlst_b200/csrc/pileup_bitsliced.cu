// Stage 2, implementation 2: pileup histogram WITHOUT per-base atomics -- bit-sliced vertical counters.
//
// Why: at config-2 depth (~1.5e5 x) the histogram is 1.5 G increments into ~1e4 x 5 bins.  Shared/global atomics
// retire ~0.5-1 increment/clk/SM (B300_MICROARCH "Atomics": ATOMS 2 cyc/lane, REDG 1.29 cyc/lane), i.e. ~1e11/s
// chip-wide, two orders of magnitude under what the 6.5 TB/s HBM stream delivers (~1e13 base-increments/s).
// So the bases are never expanded: a record stays three 32-column bit-planes per word (V, B1, B0) and 32 columns
// are counted per LOP3 with carry-save adders (Harley-Seal), the same trick as a vertical popcount.
//
// Mapping
//   CTA      : persistent over chunks (records of one contig, any length; the library builds <= 63 tiles); tile = 512 consecutive
//              coordinate-sorted records.
//              Their plane rows are ONE contiguous global range and their 16-byte records another, so a tile is two
//              cp.async.bulk (TMA 1-D, SASS UBLKCP) into a double-buffered shared-memory stage, completion on one
//              mbarrier; thread 0 issues tile t+1 before tile t is counted.  No per-thread global loads at all.
//   prepass  : once per tile the 16-byte records are rewritten in place to what the inner loop needs
//              {first contig word, row offset inside the stage, words touched, tag-filter mask}.
//   warp     : owns one 32-column word w of the contig (w mod 8 == warp id inside the sliding 8-word window).
//   lane     : takes records lane, lane+32, ... of the tile (16 per tile).  Rows are already aligned to the contig's
//              words (include/mmlst.h), so a (record, word) pair costs 1 LDS.128 + 3 LDS, ~9 integer ops to form
//              five 1-bit planes (counted, ok, ok&B0, ok&B1, ok&B0&B1) and a 16-input Harley-Seal block (30 LOP3
//              per 16 inputs per counter) into private bit-sliced counters ones/twos/fours/eights, the sixteens
//              plane rippled into 6 upper planes once per tile.
//   flush    : when the warp's word changes, after 63 tiles on the same word (63 x 16 = 1008 records per lane; one more tile
//              could reach 1024, which 10 planes cannot hold) or when the chunk ends: bit-sliced add across the 32 lanes (shuffle butterfly
//              over only as many planes as the tiles accumulated so far can have set), lane i extracts column i,
//              converts to A/C/G/T/N and issues 5 coalesced RED.ADD.
#include <stdlib.h>
#include "common.cuh"
#include "pileup.cuh"

namespace {

constexpr int TR = 512;         // records per tile
constexpr int NWARP = 8;        // column words in the window
constexpr int NTHREADS = NWARP * 32;
constexpr int LOWP = 4;         // ones, twos, fours, eights
constexpr int UPP = 6;          // 16s .. 512s  => < 1024 records per lane between flushes: a warp flushes after 63 tiles on one word
constexpr int NP = LOWP + UPP;  // planes per lane counter
constexpr uint32_t kMaxAccTiles = ((1u << NP) - 1u) / 16u;   // 63 tiles of 16 records per lane fit the NP planes
constexpr int NPR = NP + 5;     // planes after the 32-lane reduction
constexpr uint32_t FULL = 0xffffffffu;

// full adder on 32 columns at once: 2 LOP3
__device__ __forceinline__ void csa(uint32_t& hi, uint32_t& lo, uint32_t a, uint32_t b, uint32_t c) {
    const uint32_t u = a ^ b;
    hi = (a & b) | (u & c);
    lo = u ^ c;
}

struct Counter {
    uint32_t p[NP];  // p[0..3] = ones, twos, fours, eights; p[4..9] = 16s..512s
};

__device__ __forceinline__ void ripple16(Counter& c, uint32_t x) {  // add the "sixteens" plane
#pragma unroll
    for (int i = LOWP; i < NP; ++i) {
        const uint32_t carry = c.p[i] & x;
        c.p[i] ^= x;
        x = carry;
    }
}

struct Contrib { uint32_t x[5]; };  // counted, ok, ok&B0, ok&B1, ok&B0&B1

// planes of tile record i (rewritten 16-byte record in shared memory: {w0, stage row offset, nw, pm}) for contig word w
__device__ __forceinline__ Contrib load_contrib(const uint32_t* __restrict__ planes, const uint4* __restrict__ meta, uint32_t i, int w) {
    const uint4 m = meta[i];
    const uint32_t j = static_cast<uint32_t>(w - static_cast<int>(m.x));
    const bool valid = j < m.z;                       // the record touches word w (records past the tile end have nw = 0)
    const uint32_t* r = planes + (valid ? m.y + 3u * j : 0u);
    const uint32_t vm = valid ? FULL : 0u;
    const uint32_t v = r[0], b1 = r[1], b0 = r[2];
    Contrib c;
    c.x[0] = (v | b0) & vm;
    c.x[1] = v & m.w & vm;
    c.x[2] = c.x[1] & b0;
    c.x[3] = c.x[1] & b1;
    c.x[4] = c.x[2] & b1;
    return c;
}

// bit-sliced sum over the 32 lanes of a counter whose planes >= P are still zero: every lane ends with the warp
// total in P + 5 planes
template <int P>
__device__ __forceinline__ void reduce_lanes(const Counter& c, uint32_t (&t)[P + 5]) {
#pragma unroll
    for (int i = 0; i < P + 5; ++i) t[i] = (i < P) ? c.p[i] : 0u;
#pragma unroll
    for (int step = 0; step < 5; ++step) {
        uint32_t carry = 0;
#pragma unroll
        for (int i = 0; i < P + 5; ++i) {
            if (i <= P + step) {  // planes that can be non-zero after this step
                const uint32_t o = __shfl_xor_sync(FULL, t[i], 1 << step);
                uint32_t hi, lo;
                csa(hi, lo, t[i], o, carry);
                t[i] = lo;
                carry = hi;
            }
        }
    }
}

template <int N>
__device__ __forceinline__ uint32_t extract(const uint32_t (&t)[N], uint32_t lane) {
    uint32_t v = 0;
#pragma unroll
    for (int i = 0; i < N; ++i) v |= ((t[i] >> lane) & 1u) << i;
    return v;
}

struct WarpAcc {
    Counter c[5];  // counted, ok, ok&B0, ok&B1, ok&B0&B1
    __device__ __forceinline__ void clear() {
#pragma unroll
        for (int k = 0; k < 5; ++k)
#pragma unroll
            for (int i = 0; i < NP; ++i) c[k].p[i] = 0u;
    }
};

template <int P>
__device__ __forceinline__ void flush_word_p(const WarpAcc& acc, int w, const mmlst_chunk& ck, uint32_t* __restrict__ counts) {
    const uint32_t lane = threadIdx.x & 31u;
    uint32_t t[P + 5];
    uint32_t n[5];
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        reduce_lanes<P>(acc.c[k], t);
        n[k] = extract<P + 5>(t, lane);
    }
    const uint32_t n_cnt = n[0], n_ok = n[1], n_p0 = n[2], n_p1 = n[3], n_p01 = n[4];
    const long long col = static_cast<long long>(w) * 32 + lane;
    if (col < 0 || col >= static_cast<long long>(ck.contig_len)) return;
    uint32_t* c = counts + (static_cast<size_t>(ck.col_base) + col) * 5;
    const uint32_t nT = n_p01, nG = n_p1 - n_p01, nC = n_p0 - n_p01, nA = n_ok - n_p0 - n_p1 + n_p01, nN = n_cnt - n_ok;
    if (nA) atomicAdd(c + 0, nA);
    if (nC) atomicAdd(c + 1, nC);
    if (nG) atomicAdd(c + 2, nG);
    if (nT) atomicAdd(c + 3, nT);
    if (nN) atomicAdd(c + 4, nN);
}

// tiles = tiles accumulated since the counters were cleared: a lane counted <= 16 * tiles records
__device__ __forceinline__ void flush_word(const WarpAcc& acc, int w, const mmlst_chunk& ck, uint32_t* __restrict__ counts, uint32_t tiles) {
    if (tiles <= 3) flush_word_p<6>(acc, w, ck, counts);        // <= 48  < 2^6
    else if (tiles <= 15) flush_word_p<8>(acc, w, ck, counts);  // <= 240 < 2^8
    else flush_word_p<NP>(acc, w, ck, counts);                  // <= 1008 < 2^10
}

template <int NS>
__global__ void __launch_bounds__(NTHREADS, 2) pileup_bitsliced_kernel(const PileupArgs a, const uint32_t stage_words) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    // stage s: planes [stage_words] u32, then TR x 16-byte records
    const size_t stage_bytes = static_cast<size_t>(stage_words) * 4 + TR * sizeof(mmlst_prec);
    uint4* loop_recs = reinterpret_cast<uint4*>(smem_raw + NS * stage_bytes);  // [2][TR], by tile parity
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + NS * stage_bytes + 2 * TR * sizeof(uint4));

    const uint32_t lane = threadIdx.x & 31u, wid = threadIdx.x >> 5;
    tl_mark(a.tl, MMLST_TL_PILEUP, 0);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < NS; ++s) mbar_init(bars + s, 1);
        fence_mbar_init();
    }
    __syncthreads();
    pdl_wait();                 // barriers are set up; now the predecessor (selection: chunk list, header) must be complete and visible
    pdl_launch_dependents();    // the consensus CTAs may become resident; they wait for this grid before reading the counts
    uint32_t phase_bits = 0;  // parity per stage
    const int max_nw = int(a.max_row_words / 3u);  // upper bound of the contig words any record touches

    // NO LOCAL MEMORY in this kernel: a grid that has touched its stack completes late -- the dependent kernel started 6.3 us after the last CTA of
    // this one had finished, 0.9 us once the last spilled word was gone (profiles/r3k_tail_timeline.json, profiles/tools/tail_timeline.py).  The chunk
    // count is therefore re-read when it is needed (a cached load) instead of being kept live across the chunk, where ptxas parked it on the stack.
    // What has to survive a whole chunk but is the same for every thread (the next chunk of this CTA, the locus of the chunk for the fused consensus)
    // lives in shared memory, by chunk parity: thread 0 writes it before the chunk's first barrier, everybody reads it after the flush.
    __shared__ uint32_t s_ctl[2][4];
    if (blockIdx.x >= pileup_n_chunks(a)) return;
    uint32_t par = 0;
    for (uint32_t ci = blockIdx.x;; par ^= 1u) {
        const mmlst_chunk ck = a.chunks[ci];
        const bool first = ci == blockIdx.x;
        if (first) tl_mark(a.tl, MMLST_TL_PILEUP, 1, ck.rec_end);
        if (threadIdx.x == 0) {   // whether another chunk follows is settled HERE, before the flush (the load flies under the chunk's first copy)
            const uint32_t nx = ci + gridDim.x;
            s_ctl[par][0] = nx < pileup_n_chunks(a) ? nx : 0xffffffffu;
            s_ctl[par][1] = ck.reserved[0];
            s_ctl[par][2] = ck.reserved[1];
        }
        const uint32_t nrec = ck.rec_end - ck.rec_begin;
        const uint32_t ntiles = (nrec + TR - 1) / TR;
        uint4 g_first = make_uint4(0, 0, 0, 0), g_last = g_first;  // thread 0: first / last record of the next tile to copy

        auto load_geo = [&](uint32_t t) {  // thread 0: two 16-byte loads, consumed one tile later
            const uint32_t r0 = ck.rec_begin + t * TR;
            const uint32_t last = min(r0 + uint32_t(TR), ck.rec_end) - 1u;
            g_first = __ldg(reinterpret_cast<const uint4*>(a.recs + r0));
            g_last = __ldg(reinterpret_cast<const uint4*>(a.recs + last));
        };
        auto issue_copy = [&](uint32_t t, int stage) {  // thread 0
            const uint32_t r0 = ck.rec_begin + t * TR;
            const uint32_t cnt = min(uint32_t(TR), ck.rec_end - r0);
            const uint32_t a0 = (g_first.y + ck.plane_delta) & ~3u;
            const uint32_t w_end = g_last.y + ck.plane_delta + mmlst_row_words(g_last.w >> 16);
            const uint32_t pbytes = (((w_end + 3u) & ~3u) - a0) * 4u;
            const uint32_t mbytes = cnt * uint32_t(sizeof(mmlst_prec));
            uint8_t* st = smem_raw + stage * stage_bytes;
            mbar_expect_tx(bars + stage, pbytes + mbytes);
            if (pbytes) bulk_g2s(st, a.planes + a0, pbytes, bars + stage);
            bulk_g2s(st + static_cast<size_t>(stage_words) * 4, a.recs + r0, mbytes, bars + stage);
        };

        WarpAcc acc;
        acc.clear();
        int cur_w = INT_MIN;
        uint32_t acc_tiles = 0;  // tiles folded into acc since the last clear

        if (threadIdx.x == 0 && ntiles) load_geo(0);
        __syncthreads();  // every warp is done with the previous chunk's stages and loop records
        if (threadIdx.x == 0 && ntiles) { issue_copy(0, 0); if (ntiles > 1) load_geo(1); }

        for (uint32_t t = 0; t < ntiles; ++t) {
            const int stage = t % NS;
            mbar_wait(bars + stage, (phase_bits >> stage) & 1u);
            phase_bits ^= 1u << stage;
            if (first && t < 3) tl_mark(a.tl, MMLST_TL_PILEUP, 3 + t);   // tiles 0..2 landed

            const uint8_t* st = smem_raw + stage * stage_bytes;
            const uint4* raw = reinterpret_cast<const uint4*>(st + static_cast<size_t>(stage_words) * 4);
            const uint32_t* planes = reinterpret_cast<const uint32_t*>(st);
            uint4* mt = loop_recs + (t & 1u) * TR;
            const uint32_t cnt = min(uint32_t(TR), ck.rec_end - (ck.rec_begin + t * TR));
            // prepass: the tile's records in the form the inner loop wants, into the loop-record buffer of this parity
            // {first contig word, row offset inside the stage, words touched, tag-filter mask}; nw = 0 past the tile end
            {
                const uint32_t soff_base = ck.plane_delta - ((raw[0].y + ck.plane_delta) & ~3u);
#pragma unroll
                for (uint32_t i = threadIdx.x; i < uint32_t(TR); i += NTHREADS) {
                    uint4 m = make_uint4(0u, 0u, 0u, 0u);
                    if (i < cnt) {
                        const uint4 r = raw[i];
                        const int as = static_cast<int>(r.z) >> 16;
                        const int xm = static_cast<int>(r.w & 0xffu);
                        m.x = static_cast<uint32_t>(static_cast<int>(r.x) >> 5);
                        m.y = r.y + soff_base;
                        m.z = r.w >> 16;
                        m.w = (as >= a.minscore && xm <= a.max_xm) ? FULL : 0u;
                    }
                    mt[i] = m;
                }
            }
            // the ONLY CTA-wide barrier of a tile: loop records visible, and every warp has finished tile t-1, so its
            // stage and the other loop-record buffer may be overwritten
            __syncthreads();
            if (threadIdx.x == 0 && t + 1 < ntiles) {
                issue_copy(t + 1, (t + 1) % NS);
                if (t + 2 < ntiles) load_geo(t + 2);
            }
            const int wlo0 = static_cast<int>(mt[0].x);  // sorted: the first record has the smallest first word
            // last word any record of the tile can touch (span bound), clipped to the contig
            const int whi = min(static_cast<int>(mt[cnt - 1].x) + max_nw - 1, (int(ck.contig_len) - 1) >> 5);
            for (int wlo = wlo0; wlo <= whi; wlo += NWARP) {
                // the word of this window that this warp owns: w == wid (mod NWARP)
                const int w = wlo + ((int(wid) - wlo) & (NWARP - 1));
                if (w > whi) continue;
                // same word for kMaxAccTiles tiles: flush anyway, the next tile could carry out of the top plane (chunks of any length)
                if (w != cur_w || acc_tiles == kMaxAccTiles) {
                    if (cur_w != INT_MIN) flush_word(acc, cur_w, ck, a.counts, acc_tiles);
                    acc.clear();
                    cur_w = w;
                    acc_tiles = 0;
                }
                ++acc_tiles;
                uint32_t t2[5][2], t4[5][2], t8[5][2];
#pragma unroll
                for (int pr = 0; pr < 8; ++pr) {
                    const Contrib xa = load_contrib(planes, mt, (2 * pr) * 32 + lane, w);
                    const Contrib xb = load_contrib(planes, mt, (2 * pr + 1) * 32 + lane, w);
#pragma unroll
                    for (int k = 0; k < 5; ++k) {
                        Counter& c = acc.c[k];
                        csa(t2[k][pr & 1], c.p[0], c.p[0], xa.x[k], xb.x[k]);
                        if (pr & 1) {
                            csa(t4[k][(pr >> 1) & 1], c.p[1], c.p[1], t2[k][0], t2[k][1]);
                            if ((pr & 3) == 3) {
                                csa(t8[k][(pr >> 2) & 1], c.p[2], c.p[2], t4[k][0], t4[k][1]);
                                if (pr == 7) {
                                    uint32_t t16;
                                    csa(t16, c.p[3], c.p[3], t8[k][0], t8[k][1]);
                                    ripple16(c, t16);
                                }
                            }
                        }
                    }
                }
            }
        }
        if (first) tl_mark(a.tl, MMLST_TL_PILEUP, 6);   // thread 0 = warp 0 is done counting
        if (cur_w != INT_MIN) flush_word(acc, cur_w, ck, a.counts, acc_tiles);
        if (a.tl && first) {   // profiling only: when the SLOWEST warp of the CTA is done flushing
            tl_mark(a.tl, MMLST_TL_PILEUP, 2);   // (re-used slot: warp 0 done flushing; the descriptor mark moves to slot 1)
            __syncthreads();
            tl_mark(a.tl, MMLST_TL_PILEUP, 7);
        }
        if (a.fc.ticket) {
            // fused consensus: the CTA that completes the last chunk of a locus calls it (release / acquire around the ticket)
            __shared__ uint32_t s_last, s_cons[2];
            __syncthreads();
            const uint32_t locus = s_ctl[par][1];
            if (threadIdx.x == 0) {
                __threadfence();
                s_last = (atomicAdd(a.fc.ticket + locus, 1u) + 1u == s_ctl[par][2]) ? 1u : 0u;
            }
            __syncthreads();
            if (s_last) {
                __threadfence();
                const uint32_t c0 = a.fc.col_off[locus], c1 = a.fc.col_off[locus + 1];
                consensus_of_locus(a.counts, a.fc.db_ascii + a.fc.db_start[locus] - c0, c0, c1, a.fc.mincov, a.fc.consume != 0, a.fc.cons,
                                   a.fc.holes + locus, a.fc.snps + locus, s_cons);
                if (threadIdx.x == 0) a.fc.ticket[locus] = 0;
            }
        }
        ci = s_ctl[par][0];
        if (ci == 0xffffffffu) break;
    }
}

}  // namespace

// does a stream whose largest row has max_row_words words fit the bit-sliced kernel's shared-memory stages?  (else: atomic kernel)
bool mmlst_pileup_bitsliced_fits(uint32_t max_row_words) {
    const uint32_t stage_words = ((TR * max_row_words + 8u) + 31u) & ~31u;
    const size_t stage_bytes = size_t(stage_words) * 4 + TR * sizeof(mmlst_prec);
    const size_t smem = 2 * stage_bytes + 2 * TR * sizeof(uint4) + 2 * sizeof(uint64_t) + 16;
    return !(max_row_words < 3 || smem > 220 * 1024);
}

int launch_pileup_bitsliced(const PileupArgs& a_in, cudaStream_t stream) {
    PileupArgs a = a_in;
    a.tl = mmlst_timeline_buffer();
    // stage = TR rows of the largest row (+ alignment slack) + TR 16-byte records; rows too long for shared memory
    // take the atomic path
    const uint32_t stage_words = ((TR * a.max_row_words + 8u) + 31u) & ~31u;
    const size_t stage_bytes = size_t(stage_words) * 4 + TR * sizeof(mmlst_prec);
    const size_t smem = 2 * stage_bytes + 2 * TR * sizeof(uint4) + 2 * sizeof(uint64_t) + 16;
    if (a.max_row_words < 3 || smem > 220 * 1024) return launch_pileup_atomic(a, stream);
    const int sms = mmlst_num_sms();
    static size_t configured_by_device[MMLST_MAX_DEVICES] = {0};
    size_t& configured = configured_by_device[mmlst_current_device()];
    if (smem > configured) {
        cudaError_t e = cudaFuncSetAttribute(pileup_bitsliced_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
        if (e != cudaSuccess) return mmlst_cuda_fail(e, "cudaFuncSetAttribute(pileup_bitsliced_kernel)");
        configured = smem;
    }
    static bool carve[MMLST_MAX_DEVICES] = {false};
    mmlst_prefer_max_shared(pileup_bitsliced_kernel<2>, carve);
    const int per_sm = smem <= 113 * 1024 ? int(MMLST_CHUNKS_PER_SM) : 1;  // 227 KB per SM, 1 KB reserved per CTA
    const uint32_t grid = a.n_chunks_dev ? uint32_t(sms * per_sm) : min(a.n_chunks, uint32_t(sms * per_sm));
    // a device-driven launch (chunk list written by the selection kernel just before) is a link of the pass's chain: programmatic dependent launch
    if (a.n_chunks_dev) return mmlst_cuda_fail(mmlst_launch_dependent(pileup_bitsliced_kernel<2>, dim3(grid), dim3(NTHREADS), smem, stream, a, stage_words), "pileup_bitsliced_kernel");
    pileup_bitsliced_kernel<2><<<grid, NTHREADS, smem, stream>>>(a, stage_words);
    return mmlst_cuda_fail(cudaGetLastError(), "pileup_bitsliced_kernel");
}
