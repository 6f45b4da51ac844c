// Stage 1 over the RUN-LENGTH score stream (replaces metamlst.py:101-151, integer half) -- the form a coordinate-sorted BAM
// is shipped in.  The allele id of a record is not stored per record: the stream is cut into runs of equal tid
// (run_tid[r], run_start[r] .. run_start[r+1]) and every 256-record chunk carries the index of the run its first record
// belongs to (chunk_run[c]), so any chunk can be entered without a search.  What crosses PCIe and HBM per record is
// as0 i16 + xm3 u8 + qlen u16 = 5 B (the explicit-tid form of score.cu moves 9 B); the run arrays add 8 B per run and
// 4 B per 256 records.
//
// HBM-bound streaming segmented reduction: each warp owns a contiguous range of chunks, issues the loads of TWO chunks
// (6 fully coalesced 128/64-bit streaming loads per lane) before reducing either, and carries the running (allele, sum,
// hits, first index) of the open run in registers -- one atomic triple per (run, warp).  A chunk that lies inside one run
// takes the uniform path (three REDUX); a chunk crossing run boundaries is reduced segment by segment.
#include <stdlib.h>

#include "score_runs_kernels.cuh"


// Which form of the run-length kernel a launch takes: 0 = registers, two chunks in flight per warp; 1 = registers,
// software-pipelined (the next pair is requested before the current one is reduced); 2 = per-warp shared-memory ring fed
// by TMA bulk copies (3..5: the same with other stage sizes / depths, see ring_config); 6 = form 5 with pairs of chunks reduced together; 7 = form 6
// over the compact 2 B / record stream (mmlst_score_runs16_dev; the 3-byte entries take form 6 under it).  Same arithmetic, same results;
// MMLST_SCORE_VARIANT presets it, mmlst_set_score_variant changes it.
static int g_score_variant = -1;
static int score_variant() {
    if (g_score_variant < 0) {
        const char* e = getenv("MMLST_SCORE_VARIANT");
        g_score_variant = (e && e[0] >= '0' && e[0] <= '7' && !e[1]) ? e[0] - '0' : MMLST_SCORE_VARIANT_DEFAULT;
    }
    return g_score_variant;
}
extern "C" int mmlst_set_score_variant(int v) {
    const int prev = score_variant();
    if (v >= 0 && v <= 7) g_score_variant = v;
    return prev;
}

static int g_score_l2_hints = -1;
static int score_l2_hints() {
    if (g_score_l2_hints < 0) {
        const char* e = getenv("MMLST_SCORE_L2_HINTS");
        g_score_l2_hints = e ? (e[0] == '1') : MMLST_SCORE_L2_HINTS_DEFAULT;
    }
    return g_score_l2_hints;
}
extern "C" int mmlst_set_score_l2_hints(int on) {
    const int prev = score_l2_hints();
    if (on == 0 || on == 1) g_score_l2_hints = on;
    return prev;
}

// Grid of the ring forms in eighths of one resident wave (8 = exactly one wave, the blocked distribution without a tail; more = the hardware
// hands the extra CTAs to whichever SM finishes first).  MMLST_SCORE_GRID presets it, mmlst_set_score_grid_scale changes it.
static int g_score_grid8 = -1;
static int score_grid8() {
    if (g_score_grid8 < 0) {
        const char* e = getenv("MMLST_SCORE_GRID");
        const int v = e ? atoi(e) : 0;
        g_score_grid8 = (v >= 1 && v <= 64) ? v : MMLST_SCORE_GRID_DEFAULT;
    }
    return g_score_grid8;
}
extern "C" int mmlst_set_score_grid_scale(int eighths) {
    const int prev = score_grid8();
    if (eighths >= 1 && eighths <= 64) g_score_grid8 = eighths;
    return prev;
}

static int score_runs_launch(const uint32_t* run_tid, const uint32_t* run_start, uint32_t n_runs, const uint32_t* chunk_run,
                             const int16_t* as0, const uint8_t* xm3, const uint16_t* qlen, const uint16_t* chunk_qlen, const uint32_t* orig_idx,
                             uint64_t n_rec, uint64_t idx_base, const uint8_t* allow, uint32_t n_ref, int minscore,
                             int max_xm, int min_read_len, int64_t* sum_as, uint32_t* n_hit, uint32_t* first_idx,
                             uint64_t* counters, void* stream) {
    if (n_rec == 0) return MMLST_OK;
    if (!run_tid || !run_start || !chunk_run || !n_runs || !as0 || !xm3 || (!qlen && !chunk_qlen) || !allow || !sum_as || !n_hit || !first_idx || !counters) {
        mmlst_set_error("mmlst_score_runs_dev: null pointer");
        return MMLST_E_ARG;
    }
    if (n_rec >= 0xffffff00ull) { mmlst_set_error("mmlst_score_runs_dev: %llu records do not fit 32-bit run offsets", (unsigned long long)n_rec); return MMLST_E_RANGE; }
    if ((reinterpret_cast<uintptr_t>(as0) & 15) || (reinterpret_cast<uintptr_t>(xm3) & 7) || (!chunk_qlen && (reinterpret_cast<uintptr_t>(qlen) & 15)) ||
        (orig_idx && (reinterpret_cast<uintptr_t>(orig_idx) & 15))) {
        mmlst_set_error("mmlst_score_runs_dev: record arrays must be 16-byte aligned (as0/qlen/orig_idx), 8 (xm3)");
        return MMLST_E_ARG;
    }
    RunArgs a{run_tid, run_start, chunk_run, n_runs, as0, xm3, qlen, orig_idx, chunk_qlen, n_rec, idx_base, allow, n_ref, minscore, max_xm,
              min_read_len, reinterpret_cast<long long*>(sum_as), n_hit, first_idx, reinterpret_cast<unsigned long long*>(counters), score_l2_hints()};
    const uint64_t nchunks = n_rec >> 8;
    uint64_t want = (nchunks + 15) / 16;  // CTAs if every warp took two chunks
    const int variant = score_variant();
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool tma_ok = !orig_idx && !(reinterpret_cast<uintptr_t>(xm3) & 15);  // cp.async.bulk wants 16-byte aligned sources
    if (variant >= 6 && tma_ok && chunk_qlen) {  // form 5's ring with pairs of chunks reduced together (form 7 without its compact stream)
        static int pair_resident_by_device[MMLST_MAX_DEVICES] = {0};
        int& pair_resident = pair_resident_by_device[mmlst_current_device()];
        const size_t smem = (kThreads / 32) * 2u * (4u * 768u + sizeof(uint64_t));
        if (!pair_resident) {
            CUDA_TRY(cudaFuncSetAttribute(score_runs_ring_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
            CUDA_TRY(cudaFuncSetAttribute(score_runs_ring_pair_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
            int r = 0;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&r, score_runs_ring_pair_kernel, kThreads, smem) != cudaSuccess || r < 1) r = 1;
            pair_resident = r;
        }
        const uint64_t cap = static_cast<uint64_t>(mmlst_num_sms()) * pair_resident * score_grid8() / 8;
        if (want > cap) want = cap;
        if (want < 1) want = 1;
        score_runs_ring_pair_kernel<<<static_cast<unsigned>(want), kThreads, smem, st>>>(a);
        CUDA_TRY(cudaGetLastError());
        return MMLST_OK;
    }
    if (variant >= 2 && tma_ok) {
        // one resident wave of the ring kernel: NS stages of CH chunks per warp in dynamic shared memory
        static int ring_resident_by_device[MMLST_MAX_DEVICES][4][8] = {{{0}}};
        int (&ring_resident)[4][8] = ring_resident_by_device[mmlst_current_device()];
        const int hint = a.l2_hints ? 1 : 0;
        const int q = (chunk_qlen ? 1 : 0) + 2 * hint;
        const int rv = variant >= 6 ? 5 : variant;  // forms 6 and 7 exist for the per-chunk len(SEQ) stream only
        const RingCfg cfg = chunk_qlen ? (hint ? ring_config<true, true>(rv) : ring_config<true, false>(rv))
                                       : (hint ? ring_config<false, true>(rv) : ring_config<false, false>(rv));
        const size_t smem = (kThreads / 32) * static_cast<size_t>(cfg.ns) * (cfg.ch * (chunk_qlen ? 768u : 1280u) + sizeof(uint64_t));
        if (!ring_resident[q][rv]) {
            CUDA_TRY(cudaFuncSetAttribute(cfg.kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
            CUDA_TRY(cudaFuncSetAttribute(cfg.kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
            int r = 0;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&r, cfg.kern, kThreads, smem) != cudaSuccess || r < 1) r = 1;
            ring_resident[q][rv] = r;
        }
        const uint64_t cap = static_cast<uint64_t>(mmlst_num_sms()) * ring_resident[q][rv];
        if (want > cap) want = cap;
        if (want < 1) want = 1;
        cfg.kern<<<static_cast<unsigned>(want), kThreads, smem, st>>>(a);
        CUDA_TRY(cudaGetLastError());
        return MMLST_OK;
    }
    static int resident_by_device[MMLST_MAX_DEVICES][8] = {{0}};  // one wave exactly: the blocked chunk distribution has no tail
    int (&resident)[8] = resident_by_device[mmlst_current_device()];
    const int v = (orig_idx ? 1 : 0) + 2 * (variant == 1 ? 1 : 0) + (chunk_qlen ? 4 : 0);
    void (*const kerns[8])(const RunArgs) = {score_runs_kernel<false, false, false>, score_runs_kernel<true, false, false>,
                                             score_runs_kernel<false, true, false>, score_runs_kernel<true, true, false>,
                                             score_runs_kernel<false, false, true>, score_runs_kernel<true, false, true>,
                                             score_runs_kernel<false, true, true>, score_runs_kernel<true, true, true>};
    void (*kern)(const RunArgs) = kerns[v];
    if (!resident[v]) {
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident[v], kern, kThreads, 0) != cudaSuccess || resident[v] < 1) resident[v] = 3;
    }
    const uint64_t cap = static_cast<uint64_t>(mmlst_num_sms()) * resident[v];
    if (want > cap) want = cap;
    if (want < 1) want = 1;
    kern<<<static_cast<unsigned>(want), kThreads, 0, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    return MMLST_OK;
}

extern "C" int mmlst_score_runs_dev(const uint32_t* run_tid, const uint32_t* run_start, uint32_t n_runs, const uint32_t* chunk_run,
                                    const int16_t* as0, const uint8_t* xm3, const uint16_t* qlen, const uint32_t* orig_idx,
                                    uint64_t n_rec, uint64_t idx_base, const uint8_t* allow, uint32_t n_ref, int minscore,
                                    int max_xm, int min_read_len, int64_t* sum_as, uint32_t* n_hit, uint32_t* first_idx,
                                    uint64_t* counters, void* stream) {
    if (n_rec && !qlen) { mmlst_set_error("mmlst_score_runs_dev: null pointer"); return MMLST_E_ARG; }
    return score_runs_launch(run_tid, run_start, n_runs, chunk_run, as0, xm3, qlen, nullptr, orig_idx, n_rec, idx_base, allow, n_ref, minscore,
                             max_xm, min_read_len, sum_as, n_hit, first_idx, counters, stream);
}

extern "C" int mmlst_score_runs_qc_dev(const uint32_t* run_tid, const uint32_t* run_start, uint32_t n_runs, const uint32_t* chunk_run,
                                       const uint16_t* chunk_qlen, const int16_t* as0, const uint8_t* xm3, const uint32_t* orig_idx,
                                       uint64_t n_rec, uint64_t idx_base, const uint8_t* allow, uint32_t n_ref, int minscore,
                                       int max_xm, int min_read_len, int64_t* sum_as, uint32_t* n_hit, uint32_t* first_idx,
                                       uint64_t* counters, void* stream) {
    if (n_rec && !chunk_qlen) { mmlst_set_error("mmlst_score_runs_qc_dev: null pointer"); return MMLST_E_ARG; }
    return score_runs_launch(run_tid, run_start, n_runs, chunk_run, as0, xm3, nullptr, chunk_qlen, orig_idx, n_rec, idx_base, allow, n_ref,
                             minscore, max_xm, min_read_len, sum_as, n_hit, first_idx, counters, stream);
}

// Form 7: the run-length stream with len(SEQ) per chunk, scored from its compact form (code[], head[] of mmlst_score_pack16_dev).  as0[] /
// xm3[] stay resident: the chunks whose code 0 would be ambiguous (minscore <= top - 1023) and the partial last chunk are reduced from
// them.  Another form selected, max_xm >= 15 (outside the 4-bit XM field) or no compact stream: the 3-byte call, same tables.
extern "C" int mmlst_score_runs16_dev(const uint32_t* run_tid, const uint32_t* run_start, uint32_t n_runs, const uint32_t* chunk_run,
                                      const uint16_t* chunk_qlen, const int16_t* as0, const uint8_t* xm3, const uint16_t* code, const uint32_t* head,
                                      uint64_t n_rec, uint64_t idx_base, const uint8_t* allow, uint32_t n_ref, int minscore, int max_xm,
                                      int min_read_len, int64_t* sum_as, uint32_t* n_hit, uint32_t* first_idx, uint64_t* counters, void* stream) {
    if (n_rec && !chunk_qlen) { mmlst_set_error("mmlst_score_runs16_dev: null pointer"); return MMLST_E_ARG; }
    const bool compact = code && head && !(reinterpret_cast<uintptr_t>(code) & 15) && !(reinterpret_cast<uintptr_t>(xm3) & 15);
    if (score_variant() != 7 || !compact || max_xm >= 15 || n_rec < 256)
        return score_runs_launch(run_tid, run_start, n_runs, chunk_run, as0, xm3, nullptr, chunk_qlen, nullptr, n_rec, idx_base, allow, n_ref,
                                 minscore, max_xm, min_read_len, sum_as, n_hit, first_idx, counters, stream);
    if (!run_tid || !run_start || !chunk_run || !n_runs || !as0 || !xm3 || !allow || !sum_as || !n_hit || !first_idx || !counters) {
        mmlst_set_error("mmlst_score_runs16_dev: null pointer");
        return MMLST_E_ARG;
    }
    if (n_rec >= 0xffffff00ull) { mmlst_set_error("mmlst_score_runs16_dev: %llu records do not fit 32-bit run offsets", (unsigned long long)n_rec); return MMLST_E_RANGE; }
    if (reinterpret_cast<uintptr_t>(as0) & 15) { mmlst_set_error("mmlst_score_runs16_dev: as0 / xm3 / code must be 16-byte aligned"); return MMLST_E_ARG; }
    RunArgs a{run_tid, run_start, chunk_run, n_runs, as0, xm3, nullptr, nullptr, chunk_qlen, n_rec, idx_base, allow, n_ref, minscore, max_xm,
              min_read_len, reinterpret_cast<long long*>(sum_as), n_hit, first_idx, reinterpret_cast<unsigned long long*>(counters), score_l2_hints(),
              code, head};
    static int resident_by_device[MMLST_MAX_DEVICES] = {0};
    int& resident = resident_by_device[mmlst_current_device()];
    const size_t smem = (kThreads / 32) * 3u * (4u * 512u + sizeof(uint64_t));  // 3 stages of 4 chunks per warp
    if (!resident) {
        CUDA_TRY(cudaFuncSetAttribute(score_runs_ring_pair16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
        CUDA_TRY(cudaFuncSetAttribute(score_runs_ring_pair16_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        int r = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&r, score_runs_ring_pair16_kernel, kThreads, smem) != cudaSuccess || r < 1) r = 1;
        resident = r;
    }
    uint64_t want = ((n_rec >> 8) + 15) / 16;  // CTAs if every warp took two chunks
    const uint64_t cap = static_cast<uint64_t>(mmlst_num_sms()) * resident * score_grid8() / 8;
    if (want > cap) want = cap;
    if (want < 1) want = 1;
    score_runs_ring_pair16_kernel<<<static_cast<unsigned>(want), kThreads, smem, static_cast<cudaStream_t>(stream)>>>(a);
    CUDA_TRY(cudaGetLastError());
    return MMLST_OK;
}

extern "C" int mmlst_score_pack16_dev(const int16_t* as0, const uint8_t* xm3, const uint16_t* chunk_qlen, uint64_t n_rec, uint16_t* code,
                                      uint32_t* head, void* stream) {
    if (n_rec == 0) return MMLST_OK;
    if (!as0 || !xm3 || !chunk_qlen || !code || !head) { mmlst_set_error("mmlst_score_pack16_dev: null pointer"); return MMLST_E_ARG; }
    if ((reinterpret_cast<uintptr_t>(as0) & 15) || (reinterpret_cast<uintptr_t>(xm3) & 7) || (reinterpret_cast<uintptr_t>(code) & 15)) {
        mmlst_set_error("mmlst_score_pack16_dev: as0 / code must be 16-byte aligned, xm3 8");
        return MMLST_E_ARG;
    }
    uint64_t blocks = (((n_rec + 255) >> 8) + 7) / 8;  // one warp per chunk
    const uint64_t cap = static_cast<uint64_t>(mmlst_num_sms()) * 16;
    if (blocks > cap) blocks = cap;
    score_pack16_kernel<<<static_cast<unsigned>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(as0, xm3, chunk_qlen, n_rec, code, head);
    CUDA_TRY(cudaGetLastError());
    return MMLST_OK;
}

// qlen[i] of every record from the per-chunk form (the coverage kernel wants it per record)
extern "C" int mmlst_expand_chunk_qlen_dev(const uint16_t* chunk_qlen, uint64_t n_rec, uint16_t* qlen, void* stream) {
    if (n_rec == 0) return MMLST_OK;
    if (!chunk_qlen || !qlen) { mmlst_set_error("mmlst_expand_chunk_qlen_dev: null pointer"); return MMLST_E_ARG; }
    uint64_t blocks = (n_rec + 255) / 256;
    const uint64_t cap = static_cast<uint64_t>(mmlst_num_sms()) * 16;
    if (blocks > cap) blocks = cap;
    expand_chunk_qlen_kernel<<<static_cast<unsigned>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(chunk_qlen, n_rec, qlen);
    CUDA_TRY(cudaGetLastError());
    return MMLST_OK;
}

extern "C" int mmlst_expand_runs_dev(const uint32_t* run_tid, const uint32_t* run_start, uint32_t n_runs, const uint32_t* chunk_run,
                                     uint64_t n_rec, uint32_t* tid, void* stream) {
    if (n_rec == 0) return MMLST_OK;
    if (!run_tid || !run_start || !chunk_run || !n_runs || !tid) { mmlst_set_error("mmlst_expand_runs_dev: null pointer"); return MMLST_E_ARG; }
    uint64_t blocks = (n_rec + 255) / 256;
    const uint64_t cap = static_cast<uint64_t>(mmlst_num_sms()) * 16;
    if (blocks > cap) blocks = cap;
    expand_runs_kernel<<<static_cast<unsigned>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(run_tid, run_start, chunk_run, n_runs, n_rec, tid);
    CUDA_TRY(cudaGetLastError());
    return MMLST_OK;
}

// as0[i] -= coeff * xm3[i]: eight records per thread (one 128-bit and one 64-bit access each way), the last n % 8 by one thread
namespace {
__global__ void __launch_bounds__(256) as_untransform_kernel(int16_t* __restrict__ as0, const uint8_t* __restrict__ xm3, uint64_t n, int coeff) {
    const uint64_t n8 = n >> 3;
    const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
    for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n8; i += stride) {
        uint4 a = reinterpret_cast<uint4*>(as0)[i];
        const uint2 x = ld_stream_u2(xm3 + (i << 3));
        uint32_t aw[4] = {a.x, a.y, a.z, a.w};
        const uint32_t xw[2] = {x.x, x.y};
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            const uint32_t xb = xw[w >> 1] >> ((w & 1) * 16);
            const int lo = static_cast<int16_t>(aw[w] & 0xffffu) - coeff * static_cast<int>(xb & 0xffu);
            const int hi = static_cast<int16_t>(aw[w] >> 16) - coeff * static_cast<int>((xb >> 8) & 0xffu);
            aw[w] = (static_cast<uint32_t>(lo) & 0xffffu) | (static_cast<uint32_t>(hi) << 16);
        }
        reinterpret_cast<uint4*>(as0)[i] = make_uint4(aw[0], aw[1], aw[2], aw[3]);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (uint64_t i = n8 << 3; i < n; ++i) as0[i] = static_cast<int16_t>(as0[i] - coeff * static_cast<int>(xm3[i]));
}
}  // namespace

extern "C" int mmlst_as_untransform_dev(int16_t* as0, const uint8_t* xm3, uint64_t n, int coeff, void* stream) {
    if (n == 0 || coeff == 0) return MMLST_OK;
    if (!as0 || !xm3) { mmlst_set_error("mmlst_as_untransform_dev: null pointer"); return MMLST_E_ARG; }
    if ((reinterpret_cast<uintptr_t>(as0) & 15) || (reinterpret_cast<uintptr_t>(xm3) & 7)) { mmlst_set_error("mmlst_as_untransform_dev: as0 must be 16-byte aligned, xm3 8"); return MMLST_E_ARG; }
    uint64_t blocks = ((n >> 3) + 255) / 256;
    const uint64_t cap = static_cast<uint64_t>(mmlst_num_sms()) * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    as_untransform_kernel<<<static_cast<unsigned>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(as0, xm3, n, coeff);
    CUDA_TRY(cudaGetLastError());
    return MMLST_OK;
}
