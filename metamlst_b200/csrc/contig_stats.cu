// cmseq's per-column selection and per-contig summaries over the count tensor of a BATCH of contigs (cmseq_api bulk methods).
// Replaces the column loops of cmseq/cmseq.py:507-569 (get_base_stats), :226-241 (reference_free_consensus), :430-456
// (polymorphism_rate) and :459-490 (breadth_and_depth_of_coverage).  Everything the reference computes in floating point except
// the low-dominance test stays on the host; this pass only selects, counts and compacts.
//
// Three launches over the batch's columns, cut into tiles of CS_TILE columns:
//   cs_tile_kernel  : per tile, the number of selected columns, of low-dominance columns and the sum of their depths;
//   cs_scan_kernel  : one CTA, exclusive scan of the tile sums (every compacted position below comes from this scan, no atomics);
//   cs_emit_kernel  : per tile again, a block scan on top of the tile's prefix: the per-contig prefix at every contig's first column,
//                     the compacted columns in ascending order, the consensus byte of every column.
// Algorithmic bytes: 20 B / column in (the tile pass reads 16 of them again, an L2 hit at batch sizes under the L2), 1 B / column of
// consensus out when asked for, 8 + 4 * width B per compacted column, 16 B per contig.
#include "common.cuh"

namespace {

constexpr uint32_t CS_THREADS = 256;
constexpr uint32_t CS_ROUNDS = 16;
constexpr uint32_t CS_TILE = CS_THREADS * CS_ROUNDS;
constexpr uint32_t CS_SCAN_THREADS = 1024;

struct TileSum {
    uint32_t sel, low;
    unsigned long long depth;
};

struct Params {
    uint32_t mode, mincov, trunc, none_char;
    double thr;
};

// largest c in [lo, hi] with col_off[c] <= col: the contig holding `col` (contigs of length 0 are skipped over)
__device__ __forceinline__ uint32_t contig_of(const uint32_t* __restrict__ col_off, uint32_t col, uint32_t lo, uint32_t hi) {
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1) >> 1;
        if (__ldg(col_off + mid) <= col) lo = mid; else hi = mid - 1;
    }
    return lo;
}

struct Column {
    uint32_t A, C, G, T, N, depth, bmax;
    bool sel, low;
};

// cmseq's column rule: selected when A+C+G+T >= mincov inside the contig's window ([trunc, len - trunc) when len > 2 trunc, else the
// whole contig); low-dominance when selected and max/sum < thr as an IEEE double quotient, exactly the host's `base_max / base_sum`
template <bool WITH_N>
__device__ __forceinline__ Column eval_column(const uint32_t* __restrict__ counts, const uint32_t* __restrict__ col_off, uint32_t col,
                                              uint32_t c, const Params& p) {
    Column r;
    const uint32_t* q = counts + 5u * col;   // 5 * col < 2^32: MMLST_CONTIG_STATS_MAX_COLS
    r.A = q[0]; r.C = q[1]; r.G = q[2]; r.T = q[3]; r.N = WITH_N ? q[4] : 0u;
    r.depth = r.A + r.C + r.G + r.T;
    r.bmax = max(max(r.A, r.C), max(r.G, r.T));
    const uint32_t c0 = __ldg(col_off + c), len = __ldg(col_off + c + 1) - c0, local = col - c0;
    const bool cut = static_cast<unsigned long long>(len) > 2ull * p.trunc;
    const bool in_window = !cut || (local >= p.trunc && local < len - p.trunc);
    r.sel = in_window && r.depth >= p.mincov;
    r.low = r.sel && static_cast<double>(r.bmax) / static_cast<double>(r.depth) < p.thr;
    return r;
}

__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__global__ void __launch_bounds__(CS_THREADS) cs_tile_kernel(const uint32_t* __restrict__ counts, const uint32_t* __restrict__ col_off, uint32_t n,
                                                             uint32_t total_cols, Params p, TileSum* __restrict__ tiles) {
    __shared__ uint32_t s_c[2];
    __shared__ uint32_t s_w[CS_THREADS / 32];
    __shared__ unsigned long long s_d[CS_THREADS / 32];
    const uint32_t t0 = blockIdx.x * CS_TILE, t1 = min(total_cols, t0 + CS_TILE);
    if (threadIdx.x == 0) { s_c[0] = contig_of(col_off, t0, 0, n - 1); s_c[1] = contig_of(col_off, t1 - 1, 0, n - 1); }
    __syncthreads();
    const uint32_t clo = s_c[0], chi = s_c[1];
    uint32_t sel = 0, low = 0;
    unsigned long long depth = 0;
    for (uint32_t col = t0 + threadIdx.x; col < t1; col += CS_THREADS) {
        const Column r = eval_column<false>(counts, col_off, col, contig_of(col_off, col, clo, chi), p);
        sel += r.sel; low += r.low; depth += r.sel ? r.depth : 0u;
    }
    const uint32_t packed = __reduce_add_sync(0xffffffffu, sel | (low << 16));   // <= 4096 each per warp
    depth = warp_sum_u64(depth);
    if ((threadIdx.x & 31) == 0) { s_w[threadIdx.x >> 5] = packed; s_d[threadIdx.x >> 5] = depth; }
    __syncthreads();
    if (threadIdx.x == 0) {
        TileSum ts{0, 0, 0ull};
        for (uint32_t w = 0; w < CS_THREADS / 32; ++w) { ts.sel += s_w[w] & 0xffffu; ts.low += s_w[w] >> 16; ts.depth += s_d[w]; }
        tiles[blockIdx.x] = ts;
    }
}

// exclusive scan of the tile sums in place; contigs that start at total_cols (length 0 at the end of the batch) and the closing entry
// [n] get the totals
__global__ void __launch_bounds__(CS_SCAN_THREADS) cs_scan_kernel(TileSum* __restrict__ tiles, uint32_t n_tiles, const uint32_t* __restrict__ col_off,
                                                                  uint32_t n, uint32_t total_cols, uint32_t* __restrict__ sel_off,
                                                                  uint32_t* __restrict__ low_off, unsigned long long* __restrict__ depth_off) {
    __shared__ uint32_t s_sel[CS_SCAN_THREADS], s_low[CS_SCAN_THREADS];
    __shared__ unsigned long long s_dep[CS_SCAN_THREADS];
    const uint32_t per = (n_tiles + CS_SCAN_THREADS - 1) / CS_SCAN_THREADS;
    const uint32_t b0 = min(n_tiles, threadIdx.x * per), b1 = min(n_tiles, b0 + per);
    uint32_t sel = 0, low = 0;
    unsigned long long dep = 0;
    for (uint32_t i = b0; i < b1; ++i) { const TileSum t = tiles[i]; sel += t.sel; low += t.low; dep += t.depth; }
    s_sel[threadIdx.x] = sel; s_low[threadIdx.x] = low; s_dep[threadIdx.x] = dep;
    __syncthreads();
    for (uint32_t o = 1; o < CS_SCAN_THREADS; o <<= 1) {   // Hillis-Steele inclusive scan of the per-thread sums
        uint32_t a = 0, b = 0;
        unsigned long long d = 0;
        if (threadIdx.x >= o) { a = s_sel[threadIdx.x - o]; b = s_low[threadIdx.x - o]; d = s_dep[threadIdx.x - o]; }
        __syncthreads();
        s_sel[threadIdx.x] += a; s_low[threadIdx.x] += b; s_dep[threadIdx.x] += d;
        __syncthreads();
    }
    sel = s_sel[threadIdx.x] - sel; low = s_low[threadIdx.x] - low; dep = s_dep[threadIdx.x] - dep;
    for (uint32_t i = b0; i < b1; ++i) {
        const TileSum t = tiles[i];
        tiles[i] = TileSum{sel, low, dep};
        sel += t.sel; low += t.low; dep += t.depth;
    }
    const uint32_t tsel = s_sel[CS_SCAN_THREADS - 1], tlow = s_low[CS_SCAN_THREADS - 1];
    const unsigned long long tdep = s_dep[CS_SCAN_THREADS - 1];
    for (uint32_t i = threadIdx.x; i <= n; i += CS_SCAN_THREADS)
        if (col_off[i] >= total_cols) { sel_off[i] = tsel; low_off[i] = tlow; depth_off[i] = tdep; }
}

// block-wide exclusive scan of (sel | low << 16, depth); returns the round totals through the references
__device__ __forceinline__ void block_scan(uint32_t& packed, unsigned long long& depth, uint32_t* s_w, unsigned long long* s_d,
                                           uint32_t& tot_packed, unsigned long long& tot_depth) {
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t ip = packed;
    unsigned long long id = depth;
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t a = __shfl_up_sync(0xffffffffu, ip, o);
        const unsigned long long d = __shfl_up_sync(0xffffffffu, id, o);
        if (lane >= static_cast<uint32_t>(o)) { ip += a; id += d; }
    }
    __syncthreads();   // the previous round's readers are done with s_w / s_d
    if (lane == 31) { s_w[warp] = ip; s_d[warp] = id; }
    __syncthreads();
    uint32_t wp = 0, tp = 0;
    unsigned long long wd = 0, td = 0;
    for (uint32_t w = 0; w < CS_THREADS / 32; ++w) {
        if (w < warp) { wp += s_w[w]; wd += s_d[w]; }
        tp += s_w[w]; td += s_d[w];
    }
    packed = wp + ip - packed; depth = wd + id - depth;
    tot_packed = tp; tot_depth = td;
}

__global__ void __launch_bounds__(CS_THREADS) cs_emit_kernel(uint32_t* __restrict__ counts, const uint32_t* __restrict__ col_off, uint32_t n,
                                                             uint32_t total_cols, Params p, const TileSum* __restrict__ tiles,
                                                             uint32_t* __restrict__ sel_off, uint32_t* __restrict__ low_off,
                                                             unsigned long long* __restrict__ depth_off, uint32_t* __restrict__ out_col,
                                                             uint32_t* __restrict__ out_val, uint8_t* __restrict__ cons, uint32_t consume) {
    __shared__ uint32_t s_c[2];
    __shared__ uint32_t s_w[CS_THREADS / 32];
    __shared__ unsigned long long s_d[CS_THREADS / 32];
    const uint32_t t0 = blockIdx.x * CS_TILE, t1 = min(total_cols, t0 + CS_TILE);
    if (threadIdx.x == 0) { s_c[0] = contig_of(col_off, t0, 0, n - 1); s_c[1] = contig_of(col_off, t1 - 1, 0, n - 1); }
    const TileSum base = tiles[blockIdx.x];
    __syncthreads();
    const uint32_t clo = s_c[0], chi = s_c[1];
    uint32_t sel_base = base.sel, low_base = base.low;
    unsigned long long dep_base = base.depth;
    for (uint32_t r0 = t0; r0 < t1; r0 += CS_THREADS) {   // uniform trip count: every thread reaches the barriers of block_scan
        const uint32_t col = r0 + threadIdx.x;
        const bool live = col < t1;
        Column r{};
        uint32_t c = 0;
        if (live) { c = contig_of(col_off, col, clo, chi); r = eval_column<true>(counts, col_off, col, c, p); }
        uint32_t packed = static_cast<uint32_t>(r.sel) | (static_cast<uint32_t>(r.low) << 16), tp;
        unsigned long long depth = r.sel ? r.depth : 0u, td;
        block_scan(packed, depth, s_w, s_d, tp, td);
        const uint32_t sel_rank = sel_base + (packed & 0xffffu), low_rank = low_base + (packed >> 16);
        const unsigned long long dep_rank = dep_base + depth;
        if (live) {
            const uint32_t c0 = __ldg(col_off + c);
            if (c0 == col) {   // first column of contig c (and of the empty contigs just before it): its prefix
                for (uint32_t k = c + 1; k-- > 0 && __ldg(col_off + k) == col;) { sel_off[k] = sel_rank; low_off[k] = low_rank; depth_off[k] = dep_rank; }
            }
            if (p.mode == MMLST_STATS_COLUMNS && r.sel) {
                out_col[sel_rank] = col - c0;
                uint32_t* v = out_val + 5u * sel_rank;
                v[0] = r.A; v[1] = r.C; v[2] = r.G; v[3] = r.T; v[4] = r.N;
            } else if (p.mode == MMLST_STATS_DEPTH && r.sel) {
                out_col[sel_rank] = col - c0;
                out_val[sel_rank] = r.depth;
            } else if (p.mode == MMLST_STATS_LOWDOM && r.low) {
                out_col[low_rank] = col - c0;
                out_val[2u * low_rank] = r.bmax;
                out_val[2u * low_rank + 1u] = r.depth;
            }
            if (cons) cons[col] = r.sel ? mmlst_majority_call(r.A, r.C, r.G, r.T, r.N) : static_cast<uint8_t>(p.none_char);
            if (consume) { uint32_t* q = counts + 5u * col; q[0] = 0; q[1] = 0; q[2] = 0; q[3] = 0; q[4] = 0; }
        }
        sel_base += tp & 0xffffu; low_base += tp >> 16; dep_base += td;
    }
}

}  // namespace

extern "C" size_t mmlst_contig_stats_scratch_bytes(uint32_t total_cols) {
    return ((size_t)total_cols + CS_TILE - 1) / CS_TILE * sizeof(TileSum) + sizeof(TileSum);
}

extern "C" int mmlst_contig_stats_dev(uint32_t* counts, const uint32_t* col_off, uint32_t n, uint32_t total_cols, const mmlst_contig_stats_params* prm,
                                      void* scratch, size_t scratch_bytes, uint32_t* sel_off, uint32_t* low_off, uint64_t* depth_off,
                                      uint32_t* out_col, uint32_t* out_val, uint8_t* cons, uint32_t flags, void* stream) {
    if (total_cols > MMLST_CONTIG_STATS_MAX_COLS) {
        mmlst_set_error("mmlst_contig_stats_dev: %u columns in one batch, at most %u (5 * column in 32 bits)", total_cols, (uint32_t)MMLST_CONTIG_STATS_MAX_COLS);
        return MMLST_E_RANGE;
    }
    if (!prm || !col_off || !sel_off || !low_off || !depth_off) { mmlst_set_error("mmlst_contig_stats_dev: null pointer"); return MMLST_E_ARG; }
    if (prm->mode > MMLST_STATS_LOWDOM || prm->mincov == 0 || prm->none_char > 255) { mmlst_set_error("mmlst_contig_stats_dev: mode %u / mincov %u / none_char %u out of range", prm->mode, prm->mincov, prm->none_char); return MMLST_E_ARG; }
    if (n == 0) return MMLST_OK;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (total_cols == 0) {   // every contig is empty: all prefixes are 0
        CUDA_TRY(cudaMemsetAsync(sel_off, 0, ((size_t)n + 1) * 4, s)); CUDA_TRY(cudaMemsetAsync(low_off, 0, ((size_t)n + 1) * 4, s));
        CUDA_TRY(cudaMemsetAsync(depth_off, 0, ((size_t)n + 1) * 8, s));
        return MMLST_OK;
    }
    if (!counts || !scratch || !out_col || !out_val) { mmlst_set_error("mmlst_contig_stats_dev: null pointer"); return MMLST_E_ARG; }
    const uint32_t n_tiles = (total_cols + CS_TILE - 1) / CS_TILE;
    if (scratch_bytes < mmlst_contig_stats_scratch_bytes(total_cols)) { mmlst_set_error("mmlst_contig_stats_dev: scratch of %zu bytes, %zu needed", scratch_bytes, mmlst_contig_stats_scratch_bytes(total_cols)); return MMLST_E_ARG; }
    const Params p{prm->mode, prm->mincov, prm->trunc, prm->none_char, prm->dominant_frq_thrsh};
    TileSum* tiles = static_cast<TileSum*>(scratch);
    unsigned long long* dof = reinterpret_cast<unsigned long long*>(depth_off);
    static bool carve_t[MMLST_MAX_DEVICES] = {false}, carve_s[MMLST_MAX_DEVICES] = {false}, carve_e[MMLST_MAX_DEVICES] = {false};
    mmlst_prefer_max_shared(cs_tile_kernel, carve_t);
    mmlst_prefer_max_shared(cs_scan_kernel, carve_s);
    mmlst_prefer_max_shared(cs_emit_kernel, carve_e);
    cs_tile_kernel<<<n_tiles, CS_THREADS, 0, s>>>(counts, col_off, n, total_cols, p, tiles);
    CUDA_TRY(cudaGetLastError());
    cs_scan_kernel<<<1, CS_SCAN_THREADS, 0, s>>>(tiles, n_tiles, col_off, n, total_cols, sel_off, low_off, dof);
    CUDA_TRY(cudaGetLastError());
    cs_emit_kernel<<<n_tiles, CS_THREADS, 0, s>>>(counts, col_off, n, total_cols, p, tiles, sel_off, low_off, dof, out_col, out_val, cons,
                                                  (flags & MMLST_CONSENSUS_CONSUME) ? 1u : 0u);
    CUDA_TRY(cudaGetLastError());
    return MMLST_OK;
}
