// Kernels of the run-length score stream (included by score_runs.cu; tests/simt compiles the same text for the host,
// one std::thread per lane, to run the warp program of every kernel form without a GPU).
#pragma once
#include "common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr uint32_t FULL = 0xffffffffu;

struct RunArgs {
    const uint32_t* run_tid; const uint32_t* run_start; const uint32_t* chunk_run; uint32_t n_runs;
    const int16_t* as0; const uint8_t* xm3; const uint16_t* qlen; const uint32_t* orig_idx;
    const uint16_t* chunk_qlen;  // QC form: len(SEQ) of every record of chunk c (uniform chunks), qlen[] is not read
    uint64_t n_rec; uint64_t idx_base;
    const uint8_t* allow; uint32_t n_ref;
    int minscore, max_xm, min_read_len;
    long long* sum_as; uint32_t* n_hit; uint32_t* first_idx; unsigned long long* counters;
    int l2_hints;  // ring forms: streams evict-first, run tables / allow[] / chunk_qlen evict-last in the L2
    const uint16_t* code;  // form 7: the compact stream of score_pack16_kernel (one word per record) ...
    const uint32_t* head;  // ... and its per-chunk word (top AS | len(SEQ) << 16)
};

__device__ __forceinline__ void flush_run(const RunArgs& a, uint32_t key, long long s, uint32_t c, uint32_t mn) {
    if (c) {
        atomicAdd(reinterpret_cast<unsigned long long*>(a.sum_as + key), static_cast<unsigned long long>(s));
        atomicAdd(a.n_hit + key, c);
        atomicMin(a.first_idx + key, mn);
    }
}

template <bool OIDX> struct Loaded;  // one lane's 8 consecutive records of a chunk
template <> struct Loaded<false> { uint4 a8, q8; uint2 x8; uint32_t cq; };
template <> struct Loaded<true> { uint4 a8, q8; uint2 x8; uint32_t cq; uint4 oa, ob; };

// QC: the chunk's common len(SEQ) comes from chunk_qlen[] (one u16 per 256 records) instead of 16 B of qlen[] per lane
template <bool OIDX, bool QC>
__device__ __forceinline__ Loaded<OIDX> load_chunk(const RunArgs& a, uint64_t base_lane) {
    Loaded<OIDX> L;
    L.a8 = ld_stream_u4(a.as0 + base_lane);
    L.x8 = ld_stream_u2(a.xm3 + base_lane);
    if constexpr (QC) { L.cq = __ldg(a.chunk_qlen + (base_lane >> 8)); L.q8 = make_uint4(0, 0, 0, 0); }
    else { L.q8 = ld_stream_u4(a.qlen + base_lane); L.cq = 0; }
    if constexpr (OIDX) { L.oa = ld_stream_u4(a.orig_idx + base_lane); L.ob = ld_stream_u4(a.orig_idx + base_lane + 4); }
    return L;
}

template <bool OIDX>
__device__ __forceinline__ uint32_t rec_index(const Loaded<OIDX>& L, uint32_t idx0, int k) {
    if constexpr (OIDX) {
        const uint32_t oi[8] = {L.oa.x, L.oa.y, L.oa.z, L.oa.w, L.ob.x, L.ob.y, L.ob.z, L.ob.w};
        return oi[k];
    } else {
        return idx0 + k;
    }
}

struct WarpRun {  // warp-uniform state of the open run
    uint32_t r, key, end;  // run index, its allele, one past its last record (0xffffffff past the last run)
    bool al;               // allele passes --filter
    long long s; uint32_t c, mn;
};

__device__ __forceinline__ void open_run(const RunArgs& a, WarpRun& w, uint32_t r) {
    w.r = r;
    if (r < a.n_runs) {
        w.key = __ldg(a.run_tid + r);
        w.end = __ldg(a.run_start + r + 1);
        w.al = (w.key < a.n_ref) && a.allow[w.key];
    } else {
        w.key = 0xffffffffu; w.end = 0xffffffffu; w.al = false;
    }
    w.s = 0; w.c = 0; w.mn = 0xffffffffu;
}

__device__ __forceinline__ void close_run(const RunArgs& a, WarpRun& w, uint32_t lane) {
    if (lane == 0 && w.al) flush_run(a, w.key, w.s, w.c, w.mn);
}

// ---- the three filters of metamlst.py:115 on packed fields, without unpacking the records (SWAR)
// Unsigned lane-wise x >= t for lanes of any width with top bit H: d = (x | H) - (t & ~H) never borrows across lanes and
// its top bit says x_low >= t_low; then x >= t  <=>  (x_h & ~t_h) | (~(x_h ^ t_h) & d_h).  Signed as0 is compared
// after biasing both sides by 0x8000 (only the top bit of x changes, so the bias folds into the logic).
struct Thr {
    uint32_t as_T, as_TL;  // (minscore + 32768) in both halves; the same without the top bits
    uint32_t ql_T, ql_TL;  // min_read_len in both halves
    uint32_t xm_T, xm_TH;  // max_xm in all four bytes; the same with the top bits set
    uint32_t h8;           // 0x80808080, or 0 when a threshold lies outside its field and nothing can pass
};
constexpr uint32_t H16 = 0x80008000u, H8 = 0x80808080u;

__device__ __forceinline__ Thr make_thr(const RunArgs& a) {
    Thr t;
    const bool none = a.minscore > 32767 || a.min_read_len > 65535 || a.max_xm < 0;
    const uint32_t ts = static_cast<uint32_t>(max(a.minscore, -32768) + 32768) & 0xffffu;
    const uint32_t tq = static_cast<uint32_t>(min(max(a.min_read_len, 0), 65535));
    const uint32_t tx = static_cast<uint32_t>(min(max(a.max_xm, 0), 255));
    t.as_T = ts | (ts << 16); t.as_TL = t.as_T & ~H16;
    t.ql_T = tq | (tq << 16); t.ql_TL = t.ql_T & ~H16;
    t.xm_T = tx * 0x01010101u; t.xm_TH = t.xm_T | H8;
    t.h8 = none ? 0u : H8;
    return t;
}

// p_lo / p_hi: one byte per record (records 0-3 / 4-7 of the lane), 1 = passes all three filters
template <bool OIDX, bool QC>
__device__ __forceinline__ void lane_pass(const Loaded<OIDX>& L, const Thr& t, int min_read_len, uint32_t& p_lo, uint32_t& p_hi) {
    const uint32_t aw[4] = {L.a8.x, L.a8.y, L.a8.z, L.a8.w};
    const uint32_t qw[4] = {L.q8.x, L.q8.y, L.q8.z, L.q8.w};
    uint32_t m[4];
#pragma unroll
    for (int w = 0; w < 4; ++w) {
        const uint32_t da = (aw[w] | H16) - t.as_TL;
        const uint32_t ga = (~aw[w] & ~t.as_T) | ((aw[w] ^ t.as_T) & da);          // as0 >= minscore (signed halves)
        // only the top bit of every half is meaningful; the final `& t.h8` below keeps exactly those
        if constexpr (QC) {
            m[w] = ga;
        } else {
            const uint32_t dq = (qw[w] | H16) - t.ql_TL;
            const uint32_t gq = (qw[w] & ~t.ql_T) | (~(qw[w] ^ t.ql_T) & dq);     // qlen >= min_read_len
            m[w] = ga & gq;
        }
    }
    const uint32_t b_lo = __byte_perm(m[0], m[1], 0x7531), b_hi = __byte_perm(m[2], m[3], 0x7531);  // top byte of every half
    const uint32_t x0 = L.x8.x, x1 = L.x8.y;
    const uint32_t d0 = t.xm_TH - (x0 & ~H8), d1 = t.xm_TH - (x1 & ~H8);
    const uint32_t g0 = (t.xm_T & ~x0) | (~(t.xm_T ^ x0) & d0), g1 = (t.xm_T & ~x1) | (~(t.xm_T ^ x1) & d1);  // max_xm >= xm3
    p_lo = (b_lo & g0 & t.h8) >> 7;
    p_hi = (b_hi & g1 & t.h8) >> 7;
    if constexpr (QC) {
        if (static_cast<int>(L.cq) < min_read_len) { p_lo = 0; p_hi = 0; }  // warp-uniform: the whole chunk is too short
    }
}

// sum / count / first index of the lane's records selected by the byte masks
template <bool OIDX>
__device__ __forceinline__ void lane_sums(const Loaded<OIDX>& L, uint32_t p_lo, uint32_t p_hi, uint32_t idx0, int& s, uint32_t& c, uint32_t& mn) {
    s = __dp2a_lo(static_cast<int>(L.a8.x), static_cast<int>(p_lo), 0);   // as0[0] p[0] + as0[1] p[1]
    s = __dp2a_hi(static_cast<int>(L.a8.y), static_cast<int>(p_lo), s);
    s = __dp2a_lo(static_cast<int>(L.a8.z), static_cast<int>(p_hi), s);
    s = __dp2a_hi(static_cast<int>(L.a8.w), static_cast<int>(p_hi), s);
    c = __popc(p_lo | (p_hi << 1));
    if constexpr (OIDX) {
        mn = 0xffffffffu;
#pragma unroll
        for (int k = 0; k < 8; ++k) mn = (((k < 4 ? p_lo : p_hi) >> (8 * (k & 3))) & 1u) ? min(mn, rec_index<true>(L, idx0, k)) : mn;
    } else {
        const uint32_t k = p_lo ? (static_cast<uint32_t>(__ffs(p_lo)) - 1u) >> 3 : 4u + ((static_cast<uint32_t>(__ffs(p_hi)) - 1u) >> 3);
        mn = (p_lo | p_hi) ? idx0 + k : 0xffffffffu;
    }
}

// one 256-record chunk starting at record `base` (this lane: records base + 8 lane .. + 7)
template <bool OIDX, bool QC>
__device__ __forceinline__ void reduce_chunk(const RunArgs& a, const Thr& thr, WarpRun& w, const Loaded<OIDX>& L, uint64_t base, uint32_t lane,
                                             uint32_t& tot, uint32_t& ign) {
    constexpr uint32_t R = 8;
    const uint64_t rec0 = base + (lane << 3);
    const uint32_t idx0 = static_cast<uint32_t>(a.idx_base + rec0);
    uint32_t p_lo, p_hi;
    lane_pass<OIDX, QC>(L, thr, a.min_read_len, p_lo, p_hi);
    const uint64_t chunk_end = base + 256;
    if (chunk_end <= w.end) {  // the whole chunk lies inside the open run
        if (w.al) {
            int s; uint32_t c, mn;
            lane_sums<OIDX>(L, p_lo, p_hi, idx0, s, c, mn);
            tot += R;
            ign += R - c;
            w.s += __reduce_add_sync(FULL, s);
            w.c += __reduce_add_sync(FULL, c);
            w.mn = min(w.mn, __reduce_min_sync(FULL, mn));
        }
        if (chunk_end == w.end) { close_run(a, w, lane); open_run(a, w, w.r + 1); }
        return;
    }
    uint64_t lo = base;
    while (lo < chunk_end) {  // segment [lo, hi) of the chunk belongs to the open run
        const uint64_t hi = (w.end < chunk_end) ? static_cast<uint64_t>(w.end) : chunk_end;
        if (w.al) {
            // the lane's records inside the segment: bytes [klo, khi) of its 8
            const uint32_t klo = lo <= rec0 ? 0u : (lo - rec0 >= R ? R : static_cast<uint32_t>(lo - rec0));
            const uint32_t khi = hi <= rec0 ? 0u : (hi - rec0 >= R ? R : static_cast<uint32_t>(hi - rec0));
            const unsigned long long ones = 0x0101010101010101ull;
            const unsigned long long below_hi = khi >= 8 ? ~0ull : ((1ull << (8 * khi)) - 1ull);
            const unsigned long long below_lo = klo >= 8 ? ~0ull : ((1ull << (8 * klo)) - 1ull);
            const unsigned long long inm = khi > klo ? (below_hi & ~below_lo & ones) : 0ull;
            const uint32_t in_lo = static_cast<uint32_t>(inm), in_hi = static_cast<uint32_t>(inm >> 32);
            int s; uint32_t c, mn;
            lane_sums<OIDX>(L, p_lo & in_lo, p_hi & in_hi, idx0, s, c, mn);
            const uint32_t in = khi > klo ? khi - klo : 0u;
            tot += in;
            ign += in - c;
            w.s += __reduce_add_sync(FULL, s);
            w.c += __reduce_add_sync(FULL, c);
            w.mn = min(w.mn, __reduce_min_sync(FULL, mn));
        }
        if (hi == w.end) { close_run(a, w, lane); open_run(a, w, w.r + 1); }
        lo = hi;
    }
}

// tail (< 256 records): last warp of the grid, one record per lane per step; the run is found by walking from the
// tail chunk's entry
template <bool QC>
__device__ __forceinline__ void score_tail(const RunArgs& a, uint64_t nchunks, uint32_t lane, uint32_t& tot, uint32_t& ign) {
    uint32_t r = __ldg(a.chunk_run + nchunks);
    for (uint64_t i = (nchunks << 8) + lane; i < a.n_rec; i += 32) {
        while (r + 1 < a.n_runs && i >= a.run_start[r + 1]) ++r;
        const uint32_t key = a.run_tid[r];
        if (!((key < a.n_ref) && a.allow[key])) continue;
        ++tot;
        const int as = a.as0[i];
        const int ql = QC ? int(a.chunk_qlen[nchunks]) : int(a.qlen[i]);
        if ((as >= a.minscore) && (ql >= a.min_read_len) && (int(a.xm3[i]) <= a.max_xm)) {
            const uint32_t idx = a.orig_idx ? a.orig_idx[i] : static_cast<uint32_t>(a.idx_base + i);
            flush_run(a, key, as, 1u, idx);
        } else {
            ++ign;
        }
    }
}

template <bool OIDX, bool PIPE, bool QC>
__global__ void __launch_bounds__(kThreads, PIPE ? (OIDX ? 2 : 3) : (OIDX ? 3 : 4)) score_runs_kernel(const RunArgs a) {
    pdl_launch_dependents();  // the selection kernel may take its (few) CTAs now; it waits for this grid to finish before it reads the tables
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warp = (static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const uint64_t nwarps = (static_cast<uint64_t>(gridDim.x) * blockDim.x) >> 5;
    const uint64_t nchunks = a.n_rec >> 8;  // full 256-record chunks
    const uint64_t per = (nchunks + nwarps - 1) / nwarps;
    const uint64_t c0 = warp * per;
    const uint64_t c1 = (c0 + per < nchunks) ? c0 + per : nchunks;
    uint32_t tot = 0, ign = 0;
    const Thr thr = make_thr(a);

    if (c0 < c1) {
        // software pipeline: the loads of the NEXT pair of chunks are issued before the current pair is reduced, so every
        // warp keeps 2.5 KB in flight while it computes; the first pair is requested before the (dependent) run lookup
        uint64_t ch = c0;
        Loaded<OIDX> A0, A1;
        bool have = ch + 1 < c1;
        if (have) { A0 = load_chunk<OIDX, QC>(a, (ch << 8) + (lane << 3)); A1 = load_chunk<OIDX, QC>(a, ((ch + 1) << 8) + (lane << 3)); }
        WarpRun w;
        open_run(a, w, __ldg(a.chunk_run + c0));
        Loaded<OIDX> B0, B1;  // ping-pong register buffers: no copy between them (a copy would wait for the loads)
        if constexpr (!PIPE) {
            while (have) {
                reduce_chunk<OIDX, QC>(a, thr, w, A0, ch << 8, lane, tot, ign);
                reduce_chunk<OIDX, QC>(a, thr, w, A1, (ch + 1) << 8, lane, tot, ign);
                ch += 2;
                have = ch + 1 < c1;
                if (have) { A0 = load_chunk<OIDX, QC>(a, (ch << 8) + (lane << 3)); A1 = load_chunk<OIDX, QC>(a, ((ch + 1) << 8) + (lane << 3)); }
            }
        }
        while (have) {
            const bool moreB = ch + 3 < c1;
            if (moreB) { B0 = load_chunk<OIDX, QC>(a, ((ch + 2) << 8) + (lane << 3)); B1 = load_chunk<OIDX, QC>(a, ((ch + 3) << 8) + (lane << 3)); }
            reduce_chunk<OIDX, QC>(a, thr, w, A0, ch << 8, lane, tot, ign);
            reduce_chunk<OIDX, QC>(a, thr, w, A1, (ch + 1) << 8, lane, tot, ign);
            ch += 2;
            if (!moreB) break;
            have = ch + 3 < c1;
            if (have) { A0 = load_chunk<OIDX, QC>(a, ((ch + 2) << 8) + (lane << 3)); A1 = load_chunk<OIDX, QC>(a, ((ch + 3) << 8) + (lane << 3)); }
            reduce_chunk<OIDX, QC>(a, thr, w, B0, ch << 8, lane, tot, ign);
            reduce_chunk<OIDX, QC>(a, thr, w, B1, (ch + 1) << 8, lane, tot, ign);
            ch += 2;
        }
        if (ch < c1) {
            const uint64_t base = ch << 8;
            const Loaded<OIDX> L0 = load_chunk<OIDX, QC>(a, base + (lane << 3));
            reduce_chunk<OIDX, QC>(a, thr, w, L0, base, lane, tot, ign);
        }
        close_run(a, w, lane);
    }

    if (warp == nwarps - 1 && (a.n_rec & 255u)) score_tail<QC>(a, nchunks, lane, tot, ign);
    tot = __reduce_add_sync(FULL, tot);
    ign = __reduce_add_sync(FULL, ign);
    if (lane == 0 && tot) {
        atomicAdd(a.counters + 0, static_cast<unsigned long long>(tot));
        atomicAdd(a.counters + 1, static_cast<unsigned long long>(ign));
    }
}

// ---- variant 2: the same reduction fed through a per-warp shared-memory ring filled by TMA bulk copies.
// The register variants above keep at most two chunks (1.5 KB in the 3 B form) in flight per warp, and only while the
// warp is not reducing; at 32 resident warps per SM that is under the ~35 KB per SM the HBM stream needs (Little's law
// at ~6.4 TB/s), and ncu shows the kernel waiting on long-scoreboard stalls at 45 % DRAM throughput.  Here lane 0 of every
// warp keeps NS stages of two chunks each requested ahead (cp.async.bulk, completion on a warp-private mbarrier), so the
// bytes in flight (NS x 1.5 KB per warp, ~190 KB per SM) no longer depend on registers or on what the warp is doing;
// the lanes read their 8 records from the stage with one LDS.128 + one LDS.64.  Warps still own contiguous chunk ranges,
// so the open run stays in registers exactly as above, and no CTA-wide barrier is needed after the mbarrier set-up.
// ---- ring-kernel forms of the run state and of the chunk reduction.  Two differences from the functions above, same
// results: (1) the NEXT run's (allele, end) are requested when a run is opened, so a run boundary costs one cached
// allow[] lookup instead of two dependent trips to HBM (a warp meets a boundary every ~7 chunks at config 2);
// (2) a chunk that crosses run boundaries builds its per-lane record masks from 32-bit offsets inside the chunk.
struct WarpRunPF {
    uint32_t r, key, end;  // as WarpRun
    uint32_t nkey, nend;   // run r + 1, already requested
    bool al;
    long long s; uint32_t c, mn;
};

// table lookups of the ring forms: HINT = through the evict-last L2 policy `pol`, else the plain read-only path
template <bool HINT> __device__ __forceinline__ uint32_t tab_u32(const uint32_t* p, uint64_t pol) {
    if constexpr (HINT) return ld_table_u32(p, pol); else return __ldg(p);
}
template <bool HINT> __device__ __forceinline__ uint32_t tab_u16(const uint16_t* p, uint64_t pol) {
    if constexpr (HINT) return ld_table_u16(p, pol); else return __ldg(p);
}
template <bool HINT> __device__ __forceinline__ uint32_t tab_u8(const uint8_t* p, uint64_t pol) {
    if constexpr (HINT) return ld_table_u8(p, pol); else return *p;
}
template <bool HINT>
__device__ __forceinline__ void request_next_run(const RunArgs& a, WarpRunPF& w, uint64_t pol) {
    if (w.r + 1u < a.n_runs) { w.nkey = tab_u32<HINT>(a.run_tid + w.r + 1u, pol); w.nend = tab_u32<HINT>(a.run_start + w.r + 2u, pol); }
    else { w.nkey = 0xffffffffu; w.nend = 0xffffffffu; }
}
template <bool HINT>
__device__ __forceinline__ void open_run_pf(const RunArgs& a, WarpRunPF& w, uint32_t r, uint64_t pol) {
    w.r = r;
    if (r < a.n_runs) { w.key = tab_u32<HINT>(a.run_tid + r, pol); w.end = tab_u32<HINT>(a.run_start + r + 1u, pol); }
    else { w.key = 0xffffffffu; w.end = 0xffffffffu; }
    request_next_run<HINT>(a, w, pol);
    w.al = (w.key < a.n_ref) && tab_u8<HINT>(a.allow + w.key, pol);
    w.s = 0; w.c = 0; w.mn = 0xffffffffu;
}
template <bool HINT>
__device__ __forceinline__ void next_run_pf(const RunArgs& a, WarpRunPF& w, uint32_t lane, uint64_t pol) {
    if (lane == 0 && w.al) flush_run(a, w.key, w.s, w.c, w.mn);
    w.r += 1u; w.key = w.nkey; w.end = w.nend;  // past the last run: key = end = 0xffffffff, nothing is counted
    request_next_run<HINT>(a, w, pol);
    w.al = (w.key < a.n_ref) && tab_u8<HINT>(a.allow + w.key, pol);
    w.s = 0; w.c = 0; w.mn = 0xffffffffu;
}

// 0x01 in byte k of (in_lo | in_hi << 32) for the lane's records k in [klo, khi), 0 <= klo, khi <= 8
__device__ __forceinline__ uint32_t bytes_below(uint32_t k) { return k >= 4u ? 0xffffffffu : ((1u << (8u * k)) - 1u); }
__device__ __forceinline__ void segment_masks(uint32_t klo, uint32_t khi, uint32_t& in_lo, uint32_t& in_hi) {
    in_lo = bytes_below(min(khi, 4u)) & ~bytes_below(min(klo, 4u)) & 0x01010101u;
    in_hi = bytes_below(khi > 4u ? khi - 4u : 0u) & ~bytes_below(klo > 4u ? klo - 4u : 0u) & 0x01010101u;
}

// sum / count of the lane's records selected by the byte masks, and the index of the first selected one
__device__ __forceinline__ void lane_sums_pf(const Loaded<false>& L, uint32_t p_lo, uint32_t p_hi, int& s, uint32_t& c) {
    s = __dp2a_lo(static_cast<int>(L.a8.x), static_cast<int>(p_lo), 0);
    s = __dp2a_hi(static_cast<int>(L.a8.y), static_cast<int>(p_lo), s);
    s = __dp2a_lo(static_cast<int>(L.a8.z), static_cast<int>(p_hi), s);
    s = __dp2a_hi(static_cast<int>(L.a8.w), static_cast<int>(p_hi), s);
    c = __popc(p_lo | (p_hi << 1));
}
__device__ __forceinline__ uint32_t first_pass_index(uint32_t p_lo, uint32_t p_hi, uint32_t idx0) {
    const uint32_t k = p_lo ? (static_cast<uint32_t>(__ffs(p_lo)) - 1u) >> 3 : 4u + ((static_cast<uint32_t>(__ffs(p_hi)) - 1u) >> 3);
    return (p_lo | p_hi) ? idx0 + k : 0xffffffffu;
}

template <bool QC, bool HINT>
__device__ __forceinline__ void reduce_chunk_pf(const RunArgs& a, const Thr& thr, WarpRunPF& w, const Loaded<false>& L, uint32_t base, uint32_t lane,
                                                uint32_t& tot, uint32_t& ign, uint64_t pol) {
    constexpr uint32_t R = 8;
    const uint32_t idx0 = static_cast<uint32_t>(a.idx_base) + base + (lane << 3);
    uint32_t p_lo, p_hi;
    lane_pass<false, QC>(L, thr, a.min_read_len, p_lo, p_hi);
    const uint32_t chunk_end = base + 256u;  // n_rec < 2^32 - 256: no wrap
    if (chunk_end <= w.end) {  // the whole chunk lies inside the open run
        if (w.al) {
            int s; uint32_t c;
            lane_sums_pf(L, p_lo, p_hi, s, c);
            tot += R;
            ign += R - c;
            w.s += __reduce_add_sync(FULL, s);
            w.c += __reduce_add_sync(FULL, c);
            // record indices ascend inside a run (no file-order index here): once the run has a passing record, later
            // chunks cannot lower its first index
            if (w.mn == 0xffffffffu) w.mn = __reduce_min_sync(FULL, first_pass_index(p_lo, p_hi, idx0));
        }
        if (chunk_end == w.end) next_run_pf<HINT>(a, w, lane, pol);
        return;
    }
    const int lane0 = static_cast<int>(lane << 3);
    uint32_t lo = base;
    while (lo < chunk_end) {  // segment [lo, hi) of the chunk belongs to the open run
        const uint32_t hi = min(w.end, chunk_end);
        if (w.al) {
            const uint32_t klo = static_cast<uint32_t>(min(max(static_cast<int>(lo - base) - lane0, 0), 8));
            const uint32_t khi = static_cast<uint32_t>(min(max(static_cast<int>(hi - base) - lane0, 0), 8));
            uint32_t in_lo, in_hi;
            segment_masks(klo, khi, in_lo, in_hi);
            int s; uint32_t c;
            lane_sums_pf(L, p_lo & in_lo, p_hi & in_hi, s, c);
            const uint32_t in = khi - klo;  // hi > lo, so khi >= klo
            tot += in;
            ign += in - c;
            w.s += __reduce_add_sync(FULL, s);
            w.c += __reduce_add_sync(FULL, c);
            if (w.mn == 0xffffffffu) w.mn = __reduce_min_sync(FULL, first_pass_index(p_lo & in_lo, p_hi & in_hi, idx0));
        }
        if (hi == w.end) next_run_pf<HINT>(a, w, lane, pol);
        lo = hi;
    }
}

// CH chunks per stage, NS stages per warp, MINB resident CTAs per SM the register budget is set for
template <bool QC, int NS, int CH, int MINB, bool HINT>
__global__ void __launch_bounds__(kThreads, MINB) score_runs_ring_kernel(const RunArgs a) {
    pdl_launch_dependents();  // the selection kernel may take its (few) CTAs now; it waits for this grid to finish before it reads the tables
    extern __shared__ __align__(128) uint8_t ring_raw[];
    constexpr uint32_t AS_B = CH * 512u, QL_B = QC ? 0u : CH * 512u, XM_B = CH * 256u;
    constexpr uint32_t STAGE_B = AS_B + QL_B + XM_B;
    constexpr uint32_t CH_B = STAGE_B / CH;  // bytes one chunk brings
    constexpr int NW = kThreads / 32;
    const uint32_t lane = threadIdx.x & 31u, wid = threadIdx.x >> 5;
    uint8_t* const my = ring_raw + wid * (NS * STAGE_B);
    uint64_t* const bars = reinterpret_cast<uint64_t*>(ring_raw + NW * NS * STAGE_B) + wid * NS;
    if (threadIdx.x == 0) {
        uint64_t* all = reinterpret_cast<uint64_t*>(ring_raw + NW * NS * STAGE_B);
        for (int i = 0; i < NW * NS; ++i) mbar_init(all + i, 1);
        fence_mbar_init();
    }
    __syncthreads();

    const uint64_t warp = (static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const uint64_t nwarps = (static_cast<uint64_t>(gridDim.x) * blockDim.x) >> 5;
    const uint64_t nchunks = a.n_rec >> 8;
    const uint64_t per = (nchunks + nwarps - 1) / nwarps;
    const uint64_t c0 = warp * per;
    const uint64_t c1 = (c0 + per < nchunks) ? c0 + per : nchunks;
    uint32_t tot = 0, ign = 0;
    const Thr thr = make_thr(a);
    const uint64_t pol_s = HINT ? l2_policy(1) : 0ull, pol_t = HINT ? l2_policy(2) : 0ull;  // streams evict-first, tables evict-last

    if (c0 < c1) {
        const uint32_t ngroups = static_cast<uint32_t>((c1 - c0 + CH - 1) / CH);
        auto issue = [&](uint32_t g, int stage) {  // lane 0: request group g (1..CH chunks) into `stage`
            const uint64_t ch = c0 + static_cast<uint64_t>(g) * CH;
            const uint32_t nch = (c1 - ch < CH) ? static_cast<uint32_t>(c1 - ch) : static_cast<uint32_t>(CH);
            uint8_t* st = my + stage * STAGE_B;
            mbar_expect_tx(bars + stage, nch * CH_B);
            if constexpr (HINT) {
                bulk_g2s_hint(st, a.as0 + (ch << 8), nch * 512u, bars + stage, pol_s);
                if constexpr (!QC) bulk_g2s_hint(st + AS_B, a.qlen + (ch << 8), nch * 512u, bars + stage, pol_s);
                bulk_g2s_hint(st + AS_B + QL_B, a.xm3 + (ch << 8), nch * 256u, bars + stage, pol_s);
            } else {
                bulk_g2s(st, a.as0 + (ch << 8), nch * 512u, bars + stage);
                if constexpr (!QC) bulk_g2s(st + AS_B, a.qlen + (ch << 8), nch * 512u, bars + stage);
                bulk_g2s(st + AS_B + QL_B, a.xm3 + (ch << 8), nch * 256u, bars + stage);
            }
        };
        if (lane == 0) {
            const uint32_t pre = ngroups < static_cast<uint32_t>(NS) ? ngroups : static_cast<uint32_t>(NS);
            for (uint32_t g = 0; g < pre; ++g) issue(g, static_cast<int>(g));
        }
        WarpRunPF w;
        open_run_pf<HINT>(a, w, tab_u32<HINT>(a.chunk_run + c0, pol_t), pol_t);  // dependent lookups run under the first copies
        uint32_t phase = 0;
        int stage = 0;
        for (uint32_t g = 0; g < ngroups; ++g) {
            const uint64_t ch = c0 + static_cast<uint64_t>(g) * CH;
            const uint32_t nch = (c1 - ch < CH) ? static_cast<uint32_t>(c1 - ch) : static_cast<uint32_t>(CH);
            mbar_wait(bars + stage, (phase >> stage) & 1u);
            phase ^= 1u << stage;
            const uint8_t* st = my + stage * STAGE_B;
#pragma unroll
            for (uint32_t k = 0; k < static_cast<uint32_t>(CH); ++k) {
                if (k < nch) {  // warp-uniform
                    Loaded<false> L;
                    L.a8 = *reinterpret_cast<const uint4*>(st + k * 512u + lane * 16u);
                    L.x8 = *reinterpret_cast<const uint2*>(st + AS_B + QL_B + k * 256u + lane * 8u);
                    if constexpr (QC) { L.q8 = make_uint4(0, 0, 0, 0); L.cq = tab_u16<HINT>(a.chunk_qlen + ch + k, pol_t); }
                    else { L.q8 = *reinterpret_cast<const uint4*>(st + AS_B + k * 512u + lane * 16u); L.cq = 0; }
                    if (k + 1u == nch) {
                        __syncwarp();  // every lane has the stage's last records in registers: the stage may be refilled
                        if (lane == 0 && g + NS < ngroups) issue(g + NS, stage);
                    }
                    reduce_chunk_pf<QC, HINT>(a, thr, w, L, static_cast<uint32_t>((ch + k) << 8), lane, tot, ign, pol_t);
                }
            }
            stage = (stage + 1 == NS) ? 0 : stage + 1;
        }
        if (lane == 0 && w.al) flush_run(a, w.key, w.s, w.c, w.mn);
    }

    if (warp == nwarps - 1 && (a.n_rec & 255u)) score_tail<QC>(a, nchunks, lane, tot, ign);
    tot = __reduce_add_sync(FULL, tot);
    ign = __reduce_add_sync(FULL, ign);
    if (lane == 0 && tot) {
        atomicAdd(a.counters + 0, static_cast<unsigned long long>(tot));
        atomicAdd(a.counters + 1, static_cast<unsigned long long>(ign));
    }
}

// ---- form 6 (experimental, QC streams): form 5's ring (4 chunks x 2 stages per warp) with the chunks reduced TWO AT A TIME.
// r1s ncu of form 5: ~119 warp instructions per 256-record chunk of which the filter + sums are ~35; the rest is per-chunk
// bookkeeping (REDUX x 2-3, run-boundary tests, counters, loop).  When both chunks of a pair lie inside the open run -- 5 of 6
// pairs at config 2 -- one set of reductions and tests serves 512 records.  Same tables as every other form (tests/simt,
// tests/test_gpu_parity.py fixture kernel_form); a separate kernel so that the measured forms' code is untouched.
__device__ __forceinline__ void reduce_pair_pf(const RunArgs& a, const Thr& thr, WarpRunPF& w, const Loaded<false>& La, const Loaded<false>& Lb,
                                               uint32_t base, uint32_t lane, uint32_t& tot, uint32_t& ign, uint64_t pol) {
    if (base + 512u > w.end) {  // a run ends inside the pair: chunk by chunk
        reduce_chunk_pf<true, false>(a, thr, w, La, base, lane, tot, ign, pol);
        reduce_chunk_pf<true, false>(a, thr, w, Lb, base + 256u, lane, tot, ign, pol);
        return;
    }
    if (w.al) {
        uint32_t pa_lo, pa_hi, pb_lo, pb_hi;
        lane_pass<false, true>(La, thr, a.min_read_len, pa_lo, pa_hi);
        lane_pass<false, true>(Lb, thr, a.min_read_len, pb_lo, pb_hi);
        int s = __dp2a_lo(static_cast<int>(La.a8.x), static_cast<int>(pa_lo), 0);
        s = __dp2a_hi(static_cast<int>(La.a8.y), static_cast<int>(pa_lo), s);
        s = __dp2a_lo(static_cast<int>(La.a8.z), static_cast<int>(pa_hi), s);
        s = __dp2a_hi(static_cast<int>(La.a8.w), static_cast<int>(pa_hi), s);
        s = __dp2a_lo(static_cast<int>(Lb.a8.x), static_cast<int>(pb_lo), s);
        s = __dp2a_hi(static_cast<int>(Lb.a8.y), static_cast<int>(pb_lo), s);
        s = __dp2a_lo(static_cast<int>(Lb.a8.z), static_cast<int>(pb_hi), s);
        s = __dp2a_hi(static_cast<int>(Lb.a8.w), static_cast<int>(pb_hi), s);  // |s| <= 16 x 32768 per lane, x 32 lanes < 2^31
        const uint32_t c = __popc(pa_lo | (pa_hi << 1) | (pb_lo << 2) | (pb_hi << 3));
        tot += 16u;
        ign += 16u - c;
        w.s += __reduce_add_sync(FULL, s);
        w.c += __reduce_add_sync(FULL, c);
        if (w.mn == 0xffffffffu) {  // indices ascend inside a run: the first chunk's hits come first
            const uint32_t idx0 = static_cast<uint32_t>(a.idx_base) + base + (lane << 3);
            const uint32_t ma = first_pass_index(pa_lo, pa_hi, idx0);
            w.mn = __reduce_min_sync(FULL, ma != 0xffffffffu ? ma : first_pass_index(pb_lo, pb_hi, idx0 + 256u));
        }
    }
    if (base + 512u == w.end) next_run_pf<false>(a, w, lane, pol);
}

__global__ void __launch_bounds__(kThreads, 4) score_runs_ring_pair_kernel(const RunArgs a) {
    pdl_launch_dependents();  // the selection kernel may take its (few) CTAs now; it waits for this grid to finish before it reads the tables
    extern __shared__ __align__(128) uint8_t ring_raw[];
    constexpr int NS = 2;
    constexpr uint32_t CH = 4, AS_B = CH * 512u, XM_B = CH * 256u, STAGE_B = AS_B + XM_B, CH_B = STAGE_B / CH;
    constexpr int NW = kThreads / 32;
    const uint32_t lane = threadIdx.x & 31u, wid = threadIdx.x >> 5;
    uint8_t* const my = ring_raw + wid * (NS * STAGE_B);
    uint64_t* const bars = reinterpret_cast<uint64_t*>(ring_raw + NW * NS * STAGE_B) + wid * NS;
    if (threadIdx.x == 0) {
        uint64_t* all = reinterpret_cast<uint64_t*>(ring_raw + NW * NS * STAGE_B);
        for (int i = 0; i < NW * NS; ++i) mbar_init(all + i, 1);
        fence_mbar_init();
    }
    __syncthreads();

    const uint64_t warp = (static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const uint64_t nwarps = (static_cast<uint64_t>(gridDim.x) * blockDim.x) >> 5;
    const uint64_t nchunks = a.n_rec >> 8;
    const uint64_t per = (nchunks + nwarps - 1) / nwarps;
    const uint64_t c0 = warp * per;
    const uint64_t c1 = (c0 + per < nchunks) ? c0 + per : nchunks;
    uint32_t tot = 0, ign = 0;
    const Thr thr = make_thr(a);

    if (c0 < c1) {
        const uint32_t ngroups = static_cast<uint32_t>((c1 - c0 + CH - 1) / CH);
        auto issue = [&](uint32_t g, int stage) {  // lane 0: request group g (1..CH chunks) into `stage`
            const uint64_t ch = c0 + static_cast<uint64_t>(g) * CH;
            const uint32_t nch = (c1 - ch < CH) ? static_cast<uint32_t>(c1 - ch) : CH;
            uint8_t* st = my + stage * STAGE_B;
            mbar_expect_tx(bars + stage, nch * CH_B);
            if (a.l2_hints) {   // the stream is read once: evict-first, so that what the rest of the pass re-reads (tables, the pileup stream, kernel code) stays in the L2
                const uint64_t pol_s = l2_policy(1);   // one instruction per stage, not a register pair held across the loop
                bulk_g2s_hint(st, a.as0 + (ch << 8), nch * 512u, bars + stage, pol_s);
                bulk_g2s_hint(st + AS_B, a.xm3 + (ch << 8), nch * 256u, bars + stage, pol_s);
            } else {
                bulk_g2s(st, a.as0 + (ch << 8), nch * 512u, bars + stage);
                bulk_g2s(st + AS_B, a.xm3 + (ch << 8), nch * 256u, bars + stage);
            }
        };
        if (lane == 0) {
            const uint32_t pre = ngroups < static_cast<uint32_t>(NS) ? ngroups : static_cast<uint32_t>(NS);
            for (uint32_t g = 0; g < pre; ++g) issue(g, static_cast<int>(g));
        }
        WarpRunPF w;
        open_run_pf<false>(a, w, __ldg(a.chunk_run + c0), 0ull);
        uint32_t phase = 0;
        int stage = 0;
        auto load = [&](const uint8_t* st, uint32_t k, uint64_t ch) {
            Loaded<false> L;
            L.a8 = *reinterpret_cast<const uint4*>(st + k * 512u + lane * 16u);
            L.x8 = *reinterpret_cast<const uint2*>(st + AS_B + k * 256u + lane * 8u);
            L.q8 = make_uint4(0, 0, 0, 0);
            L.cq = __ldg(a.chunk_qlen + ch + k);
            return L;
        };
        for (uint32_t g = 0; g < ngroups; ++g) {
            const uint64_t ch = c0 + static_cast<uint64_t>(g) * CH;
            const uint32_t nch = (c1 - ch < CH) ? static_cast<uint32_t>(c1 - ch) : CH;
            mbar_wait(bars + stage, (phase >> stage) & 1u);
            phase ^= 1u << stage;
            const uint8_t* st = my + stage * STAGE_B;
#pragma unroll
            for (uint32_t k = 0; k < CH; k += 2) {
                if (k < nch) {  // warp-uniform
                    const bool two = k + 1u < nch;
                    const Loaded<false> La = load(st, k, ch);
                    Loaded<false> Lb = La;
                    if (two) Lb = load(st, k + 1u, ch);
                    if (k + 2u >= nch) {
                        __syncwarp();  // every lane has the stage's last records in registers: the stage may be refilled
                        if (lane == 0 && g + NS < ngroups) issue(g + NS, stage);
                    }
                    const uint32_t base = static_cast<uint32_t>((ch + k) << 8);
                    if (two) reduce_pair_pf(a, thr, w, La, Lb, base, lane, tot, ign, 0ull);
                    else reduce_chunk_pf<true, false>(a, thr, w, La, base, lane, tot, ign, 0ull);
                }
            }
            stage = (stage + 1 == NS) ? 0 : stage + 1;
        }
        if (lane == 0 && w.al) flush_run(a, w.key, w.s, w.c, w.mn);
    }

    if (warp == nwarps - 1 && (a.n_rec & 255u)) score_tail<true>(a, nchunks, lane, tot, ign);
    tot = __reduce_add_sync(FULL, tot);
    ign = __reduce_add_sync(FULL, ign);
    if (lane == 0 && tot) {
        atomicAdd(a.counters + 0, static_cast<unsigned long long>(tot));
        atomicAdd(a.counters + 1, static_cast<unsigned long long>(ign));
    }
}

// ---- form 7: form 6 over the COMPACT score stream, 2 B per record instead of 3.  Only the as0 of a record that passes enters a
// result, and the records of one 256-record chunk of a sorted sample lie within a few hundred AS of each other, so a record is
// stored relative to its chunk's largest score.  score_pack16_kernel is the one definition of the format:
//   head[c] = u16(top_c) | len(SEQ)_c << 16,  top_c = max as0 over chunk c,  base_c = top_c - 1023
//   code[i] = 0x8400 | x' << 11 | a   (bit 15 and bit 10: guard bits, always 1)
//     a  = clamp(as0 - base_c, 0, 1023): 1..1023 exact, 0 = "as0 <= base_c"
//     x' = 15 - min(xm3, 15):            xm3 <= 14 exact, 0 = "xm3 >= 15"
// Both filters are "field >= threshold", so one subtraction of T = A | (15 - max_xm) << 11 (A = minscore - base_c, per chunk)
// tests both fields of both records of a 32-bit word: a field passes iff the guard bit above it survives.  A passing record's
// as0 is base_c + a = minscore + (a - A), and a - A is what the subtraction leaves in bits 0..9: the sum over a lane's hits is
// the sum of those fields plus minscore times the hit count, whatever the chunk.  The code is exact except where a = 0 can pass,
// i.e. minscore <= base_c: such a chunk (decided per chunk, warp-uniformly) is reduced from the resident as0[] / xm3[] as form 6
// does.  max_xm >= 15 never reaches this kernel (the launcher sends the call to form 6), max_xm < 0 puts 16 in the x' threshold
// and min(A, 1024) = 1024 (minscore above top_c, or a chunk shorter than min_read_len) makes the c threshold fail every record.
__device__ __forceinline__ uint32_t half_masks(uint32_t p) {  // 0xffff in each 16-bit half whose top bit is set
#ifdef MMLST_HOST_EMUL
    return ((p & 0x8000u) ? 0x0000ffffu : 0u) | ((p & 0x80000000u) ? 0xffff0000u : 0u);
#else
    uint32_t m;  // PRMT sign-replicate of bytes 1 and 3 (not __byte_perm: the intrinsic ignores the sign bit of each selector nibble)
    asm("prmt.b32 %0, %1, 0, 0xbb99;" : "=r"(m) : "r"(p));
    return m;
#endif
}

// the lane's two records of word `w`: per half, 0xffff iff the record passes (m) and its a - A (v)
__device__ __forceinline__ void pass16(uint32_t w, uint32_t T, uint32_t& m, uint32_t& v) {
    const uint32_t d = w - T;  // no borrow leaves a field: every field of w is >= the matching field of T, guards included
    m = half_masks(d & (d << 5));  // bit 10 (a >= A) moved onto bit 15 (x' >= 15 - max_xm)
    v = d & m & 0x03ff03ffu;
}

// number of 0xffff halves in a sum of half masks (n_lo, n_hi <= 0x7fff): -sum = n_lo + (n_hi - n_lo) << 16 (mod 2^32)
__device__ __forceinline__ uint32_t halves_set(uint32_t sm) {
    const uint32_t u = 0u - sm;
    return ((u & 0xffffu) * 2u + (u >> 16)) & 0xffffu;
}

// index of the lane's first passing record among its 8 (half masks of words 0..3), 0xffffffff if none
__device__ __forceinline__ uint32_t first_pass16(const uint32_t m[4], uint32_t idx0) {
    uint32_t b = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) b |= (m[j] & 0x00010001u) << (2 * j);  // record 2j at bit 2j, record 2j + 1 at bit 16 + 2j
    b = (b & 0x55u) | ((b >> 15) & 0xaau);
    return b ? idx0 + static_cast<uint32_t>(__ffs(b)) - 1u : 0xffffffffu;
}

// threshold word of chunk c for the compact stream; fb = the chunk has to be reduced from the 3-byte arrays
__device__ __forceinline__ uint32_t chunk_thr16(uint32_t head, int ms, uint32_t tx, int min_read_len, bool& fb) {
    int A = ms + 1023 - static_cast<int>(static_cast<int16_t>(head & 0xffffu));  // minscore - base_c
    if (static_cast<int>(head >> 16) < min_read_len) A = 1024;                    // the whole chunk is too short
    A = min(A, 1024);
    fb = A <= 0;
    return (static_cast<uint32_t>(A) | tx) * 0x00010001u;
}

// one compact chunk (lane: records base + 8 lane .. + 7 in q), run boundaries inside it allowed
__device__ __forceinline__ void reduce_chunk16(const RunArgs& a, WarpRunPF& w, const uint4& q, uint32_t T, int ms, uint32_t base, uint32_t lane,
                                               uint32_t& tot, uint32_t& ign) {
    const uint32_t idx0 = static_cast<uint32_t>(a.idx_base) + base + (lane << 3);
    const uint32_t wv[4] = {q.x, q.y, q.z, q.w};
    uint32_t m[4], v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) pass16(wv[j], T, m[j], v[j]);
    const uint32_t chunk_end = base + 256u;
    if (chunk_end <= w.end) {  // the whole chunk lies inside the open run
        if (w.al) {
            const uint32_t acc = v[0] + v[1] + v[2] + v[3];
            const uint32_t n = halves_set(m[0] + m[1] + m[2] + m[3]);
            const int s = static_cast<int>((acc & 0xffffu) + (acc >> 16)) + ms * static_cast<int>(n);
            tot += 8u;
            ign += 8u - n;
            w.s += __reduce_add_sync(FULL, s);
            w.c += __reduce_add_sync(FULL, n);
            if (w.mn == 0xffffffffu) w.mn = __reduce_min_sync(FULL, first_pass16(m, idx0));
        }
        if (chunk_end == w.end) next_run_pf<false>(a, w, lane, 0ull);
        return;
    }
    const int lane0 = static_cast<int>(lane << 3);
    uint32_t lo = base;
    while (lo < chunk_end) {  // segment [lo, hi) of the chunk belongs to the open run
        const uint32_t hi = min(w.end, chunk_end);
        if (w.al) {
            const int klo = min(max(static_cast<int>(lo - base) - lane0, 0), 8);
            const int khi = min(max(static_cast<int>(hi - base) - lane0, 0), 8);
            uint32_t mm[4], acc = 0, sm = 0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {  // records 2j, 2j + 1 of the lane inside [klo, khi)
                const uint32_t sel = ((2 * j >= klo && 2 * j < khi) ? 0x0000ffffu : 0u) | ((2 * j + 1 >= klo && 2 * j + 1 < khi) ? 0xffff0000u : 0u);
                mm[j] = m[j] & sel;
                acc += v[j] & sel;
                sm += mm[j];
            }
            const uint32_t n = halves_set(sm);
            const int s = static_cast<int>((acc & 0xffffu) + (acc >> 16)) + ms * static_cast<int>(n);
            const uint32_t in = static_cast<uint32_t>(khi - klo);  // hi > lo, so khi >= klo
            tot += in;
            ign += in - n;
            w.s += __reduce_add_sync(FULL, s);
            w.c += __reduce_add_sync(FULL, n);
            if (w.mn == 0xffffffffu) w.mn = __reduce_min_sync(FULL, first_pass16(mm, idx0));
        }
        if (hi == w.end) next_run_pf<false>(a, w, lane, 0ull);
        lo = hi;
    }
}

// two compact chunks, neither of which falls back
__device__ __forceinline__ void reduce_pair16(const RunArgs& a, WarpRunPF& w, const uint4& qa, const uint4& qb, uint32_t Ta, uint32_t Tb, int ms,
                                              uint32_t base, uint32_t lane, uint32_t& tot, uint32_t& ign) {
    if (base + 512u > w.end) {  // a run ends inside the pair: chunk by chunk
        reduce_chunk16(a, w, qa, Ta, ms, base, lane, tot, ign);
        reduce_chunk16(a, w, qb, Tb, ms, base + 256u, lane, tot, ign);
        return;
    }
    if (w.al) {
        const uint32_t wa[4] = {qa.x, qa.y, qa.z, qa.w}, wb[4] = {qb.x, qb.y, qb.z, qb.w};
        uint32_t ma[4], mb[4], va[4], vb[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) { pass16(wa[j], Ta, ma[j], va[j]); pass16(wb[j], Tb, mb[j], vb[j]); }
        const uint32_t acc = (va[0] + va[1] + va[2] + va[3]) + (vb[0] + vb[1] + vb[2] + vb[3]);  // <= 8 x 1022 per half
        const uint32_t n = halves_set((ma[0] + ma[1] + ma[2] + ma[3]) + (mb[0] + mb[1] + mb[2] + mb[3]));
        const int s = static_cast<int>((acc & 0xffffu) + (acc >> 16)) + ms * static_cast<int>(n);  // |s| <= 16 x 32768 per lane
        tot += 16u;
        ign += 16u - n;
        w.s += __reduce_add_sync(FULL, s);
        w.c += __reduce_add_sync(FULL, n);
        if (w.mn == 0xffffffffu) {  // indices ascend inside a run: the first chunk's hits come first
            const uint32_t idx0 = static_cast<uint32_t>(a.idx_base) + base + (lane << 3);
            const uint32_t fa = first_pass16(ma, idx0);
            w.mn = __reduce_min_sync(FULL, fa != 0xffffffffu ? fa : first_pass16(mb, idx0 + 256u));
        }
    }
    if (base + 512u == w.end) next_run_pf<false>(a, w, lane, 0ull);
}

// a chunk whose code 0 would be ambiguous: form 6's chunk reduction over the resident 3-byte arrays
__device__ __forceinline__ void reduce_chunk_fallback(const RunArgs& a, const Thr& thr, WarpRunPF& w, uint32_t head, uint32_t base, uint32_t lane,
                                                      uint32_t& tot, uint32_t& ign) {
    Loaded<false> L;
    L.a8 = ld_stream_u4(a.as0 + base + (lane << 3));
    L.x8 = ld_stream_u2(a.xm3 + base + (lane << 3));
    L.q8 = make_uint4(0, 0, 0, 0);
    L.cq = head >> 16;
    reduce_chunk_pf<true, false>(a, thr, w, L, base, lane, tot, ign, 0ull);
}

__global__ void __launch_bounds__(kThreads, 4) score_runs_ring_pair16_kernel(const RunArgs a) {
    pdl_launch_dependents();  // the selection kernel may take its (few) CTAs now; it waits for this grid to finish before it reads the tables
    extern __shared__ __align__(128) uint8_t ring_raw[];
    constexpr int NS = 3;
    constexpr uint32_t CH = 4, CH_B = 512u, STAGE_B = CH * CH_B;
    constexpr int NW = kThreads / 32;
    const uint32_t lane = threadIdx.x & 31u, wid = threadIdx.x >> 5;
    uint8_t* const my = ring_raw + wid * (NS * STAGE_B);
    uint64_t* const bars = reinterpret_cast<uint64_t*>(ring_raw + NW * NS * STAGE_B) + wid * NS;
    if (threadIdx.x == 0) {
        uint64_t* all = reinterpret_cast<uint64_t*>(ring_raw + NW * NS * STAGE_B);
        for (int i = 0; i < NW * NS; ++i) mbar_init(all + i, 1);
        fence_mbar_init();
    }
    __syncthreads();

    const uint64_t warp = (static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const uint64_t nwarps = (static_cast<uint64_t>(gridDim.x) * blockDim.x) >> 5;
    const uint64_t nchunks = a.n_rec >> 8;
    const uint64_t per = (nchunks + nwarps - 1) / nwarps;
    const uint64_t c0 = warp * per;
    const uint64_t c1 = (c0 + per < nchunks) ? c0 + per : nchunks;
    uint32_t tot = 0, ign = 0;
    const Thr thr = make_thr(a);
    const int ms = min(max(a.minscore, -32768), 32768);                               // same filter on an int16 as0
    const uint32_t tx = static_cast<uint32_t>(a.max_xm < 0 ? 16 : 15 - a.max_xm) << 11;  // 0 <= max_xm <= 14, or nothing passes

    if (c0 < c1) {
        const uint32_t ngroups = static_cast<uint32_t>((c1 - c0 + CH - 1) / CH);
        auto issue = [&](uint32_t g, int stage) {  // lane 0: request group g (1..CH chunks) into `stage`
            const uint64_t ch = c0 + static_cast<uint64_t>(g) * CH;
            const uint32_t nch = (c1 - ch < CH) ? static_cast<uint32_t>(c1 - ch) : CH;
            uint8_t* st = my + stage * STAGE_B;
            mbar_expect_tx(bars + stage, nch * CH_B);
            if (a.l2_hints) bulk_g2s_hint(st, a.code + (ch << 8), nch * CH_B, bars + stage, l2_policy(1));  // read once: evict-first
            else bulk_g2s(st, a.code + (ch << 8), nch * CH_B, bars + stage);
        };
        if (lane == 0) {
            const uint32_t pre = ngroups < static_cast<uint32_t>(NS) ? ngroups : static_cast<uint32_t>(NS);
            for (uint32_t g = 0; g < pre; ++g) issue(g, static_cast<int>(g));
        }
        WarpRunPF w;
        open_run_pf<false>(a, w, __ldg(a.chunk_run + c0), 0ull);
        uint32_t phase = 0;
        int stage = 0;
        for (uint32_t g = 0; g < ngroups; ++g) {
            const uint64_t ch = c0 + static_cast<uint64_t>(g) * CH;
            const uint32_t nch = (c1 - ch < CH) ? static_cast<uint32_t>(c1 - ch) : CH;
            mbar_wait(bars + stage, (phase >> stage) & 1u);
            phase ^= 1u << stage;
            const uint8_t* st = my + stage * STAGE_B;
#pragma unroll
            for (uint32_t k = 0; k < CH; k += 2) {
                if (k < nch) {  // warp-uniform
                    const bool two = k + 1u < nch;
                    const uint32_t ha = __ldg(a.head + ch + k), hb = two ? __ldg(a.head + ch + k + 1u) : 0u;
                    const uint4 qa = *reinterpret_cast<const uint4*>(st + k * CH_B + lane * 16u);
                    const uint4 qb = two ? *reinterpret_cast<const uint4*>(st + (k + 1u) * CH_B + lane * 16u) : qa;
                    if (k + 2u >= nch) {
                        __syncwarp();  // every lane has the stage's last records in registers: the stage may be refilled
                        if (lane == 0 && g + NS < ngroups) issue(g + NS, stage);
                    }
                    bool fa, fb;
                    const uint32_t Ta = chunk_thr16(ha, ms, tx, a.min_read_len, fa), Tb = chunk_thr16(hb, ms, tx, a.min_read_len, fb);
                    const uint32_t base = static_cast<uint32_t>((ch + k) << 8);
                    if (two && !fa && !fb) {
                        reduce_pair16(a, w, qa, qb, Ta, Tb, ms, base, lane, tot, ign);
                    } else {
                        if (fa) reduce_chunk_fallback(a, thr, w, ha, base, lane, tot, ign);
                        else reduce_chunk16(a, w, qa, Ta, ms, base, lane, tot, ign);
                        if (two) {
                            if (fb) reduce_chunk_fallback(a, thr, w, hb, base + 256u, lane, tot, ign);
                            else reduce_chunk16(a, w, qb, Tb, ms, base + 256u, lane, tot, ign);
                        }
                    }
                }
            }
            stage = (stage + 1 == NS) ? 0 : stage + 1;
        }
        if (lane == 0 && w.al) flush_run(a, w.key, w.s, w.c, w.mn);
    }

    if (warp == nwarps - 1 && (a.n_rec & 255u)) score_tail<true>(a, nchunks, lane, tot, ign);
    tot = __reduce_add_sync(FULL, tot);
    ign = __reduce_add_sync(FULL, ign);
    if (lane == 0 && tot) {
        atomicAdd(a.counters + 0, static_cast<unsigned long long>(tot));
        atomicAdd(a.counters + 1, static_cast<unsigned long long>(ign));
    }
}

// the compact stream of form 7 (format above) from the resident 3-byte form: one warp per 256-record chunk, every chunk
// including the partial last one (the kernel reduces that one from the 3-byte arrays)
__global__ void __launch_bounds__(256) score_pack16_kernel(const int16_t* __restrict__ as0, const uint8_t* __restrict__ xm3,
                                                           const uint16_t* __restrict__ chunk_qlen, uint64_t n_rec, uint16_t* __restrict__ code,
                                                           uint32_t* __restrict__ head) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t nwarps = (static_cast<uint64_t>(gridDim.x) * blockDim.x) >> 5;
    const uint64_t nch = (n_rec + 255u) >> 8;
    for (uint64_t c = (static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; c < nch; c += nwarps) {
        const uint64_t i0 = (c << 8) + (lane << 3);
        const bool full = (c << 8) + 256u <= n_rec;  // warp-uniform
        int as[8];
        uint32_t xm[8];
        if (full) {
            const uint4 a8 = ld_stream_u4(as0 + i0);
            const uint2 x8 = ld_stream_u2(xm3 + i0);
            const uint32_t aw[4] = {a8.x, a8.y, a8.z, a8.w};
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                as[k] = static_cast<int16_t>((aw[k >> 1] >> (16 * (k & 1))) & 0xffffu);
                xm[k] = ((k < 4 ? x8.x : x8.y) >> (8 * (k & 3))) & 0xffu;
            }
        } else {
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const bool in = i0 + k < n_rec;
                as[k] = in ? static_cast<int>(as0[i0 + k]) : -32768;  // outside the stream: raises no maximum, stored nowhere
                xm[k] = in ? static_cast<uint32_t>(xm3[i0 + k]) : 255u;
            }
        }
        int mx = as[0];
#pragma unroll
        for (int k = 1; k < 8; ++k) mx = max(mx, as[k]);
        const int top = static_cast<int>(__reduce_max_sync(FULL, static_cast<uint32_t>(mx + 32768))) - 32768;
        const int base = top - 1023;
        uint32_t w16[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) w16[k] = 0x8400u | ((15u - min(xm[k], 15u)) << 11) | static_cast<uint32_t>(max(as[k] - base, 0));
        if (full) {
            *reinterpret_cast<uint4*>(code + i0) = make_uint4(w16[0] | (w16[1] << 16), w16[2] | (w16[3] << 16), w16[4] | (w16[5] << 16), w16[6] | (w16[7] << 16));
        } else {
#pragma unroll
            for (int k = 0; k < 8; ++k)
                if (i0 + k < n_rec) code[i0 + k] = static_cast<uint16_t>(w16[k]);
        }
        if (lane == 0) head[c] = (static_cast<uint32_t>(top) & 0xffffu) | (static_cast<uint32_t>(__ldg(chunk_qlen + c)) << 16);
    }
}

// the ring configurations a launch can ask for (variant 2..5): {chunks per stage, stages, CTAs per SM}
struct RingCfg { void (*kern)(const RunArgs); uint32_t ch, ns; };
template <bool QC, bool HINT>
inline RingCfg ring_config(int variant) {
    if constexpr (QC) {  // 768 B per chunk
        switch (variant) {
            case 3: return {score_runs_ring_kernel<true, 3, 4, 3, HINT>, 4, 3};   // 72 KB per CTA
            case 4: return {score_runs_ring_kernel<true, 2, 8, 2, HINT>, 8, 2};   // 96 KB
            case 5: return {score_runs_ring_kernel<true, 2, 4, 4, HINT>, 4, 2};   // 48 KB
            default: return {score_runs_ring_kernel<true, 4, 2, 4, HINT>, 2, 4};  // 48 KB
        }
    } else {  // 1280 B per chunk
        switch (variant) {
            case 3: case 4: case 5: return {score_runs_ring_kernel<false, 2, 4, 2, HINT>, 4, 2};  // 80 KB
            default: return {score_runs_ring_kernel<false, 3, 2, 3, HINT>, 2, 3};                  // 60 KB
        }
    }
}

// tid[i] of every record from the run arrays (the coverage kernel and tests want the explicit form)
__global__ void __launch_bounds__(256) expand_runs_kernel(const uint32_t* __restrict__ run_tid, const uint32_t* __restrict__ run_start,
                                                          const uint32_t* __restrict__ chunk_run, uint32_t n_runs, uint64_t n_rec,
                                                          uint32_t* __restrict__ tid) {
    const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
    for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n_rec; i += stride) {
        uint32_t r = __ldg(chunk_run + (i >> 8));
        while (r + 1 < n_runs && i >= __ldg(run_start + r + 1)) ++r;
        tid[i] = __ldg(run_tid + r);
    }
}

__global__ void __launch_bounds__(256) expand_chunk_qlen_kernel(const uint16_t* __restrict__ chunk_qlen, uint64_t n_rec, uint16_t* __restrict__ qlen) {
    const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
    for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n_rec; i += stride) qlen[i] = __ldg(chunk_qlen + (i >> 8));
}

}  // namespace
