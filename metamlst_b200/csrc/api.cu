// C-ABI plumbing: error text, context (stream + grow-only device buffers), host-buffer entry points.
#include <stdarg.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "common.cuh"
#include "de.h"
#include "pileup.cuh"

static thread_local char g_err[512] = "";

void mmlst_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int mmlst_cuda_fail(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return MMLST_OK;
    mmlst_set_error("CUDA error in %s: %s", what, cudaGetErrorString(e));
    return MMLST_E_CUDA;
}

namespace {
struct TraceBuf { const char* label[32]; double t[32]; int n = 0; };
thread_local TraceBuf g_trace;
bool trace_on() { static const bool on = [] { const char* e = getenv("MMLST_TRACE"); return e && *e && *e != '0'; }(); return on; }
double now_us() { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
}  // namespace
void mmlst_trace_mark(const char* label) {
    if (!trace_on() || g_trace.n >= 32) return;
    g_trace.label[g_trace.n] = label; g_trace.t[g_trace.n++] = now_us();
}
void mmlst_trace_flush(const char* call) {
    if (!trace_on()) return;
    fprintf(stderr, "[mmlst trace] %s:", call);
    for (int i = 1; i < g_trace.n; ++i) fprintf(stderr, " %s=%.0fus", g_trace.label[i], g_trace.t[i] - g_trace.t[i - 1]);
    if (g_trace.n > 1) fprintf(stderr, " total=%.0fus", g_trace.t[g_trace.n - 1] - g_trace.t[0]);
    fprintf(stderr, "\n");
    g_trace.n = 0;
}

static unsigned long long* g_timeline = nullptr;
unsigned long long* mmlst_timeline_buffer() { return g_timeline; }
// see include/mmlst.h
extern "C" int mmlst_debug_timeline(uint64_t* dev_buf) { g_timeline = reinterpret_cast<unsigned long long*>(dev_buf); return MMLST_OK; }

int mmlst_uniform_carveout() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("MMLST_UNIFORM_CARVEOUT"); v = (e && e[0] == '0') ? 0 : 1; }
    return v;
}

int mmlst_num_sms() {
    static int by_device[MMLST_MAX_DEVICES] = {0};  // per device: one process may drive several GPUs (sample.type_cohort)
    int& n = by_device[mmlst_current_device()];
    if (n == 0) {
        int dev = 0, v = 0;
        if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && v > 0) n = v;
        else n = MMLST_NUM_SMS_DEFAULT;
    }
    return n;
}

static int g_pdl = -1;
int mmlst_pdl_enabled() {
    if (g_pdl < 0) { const char* e = getenv("MMLST_PDL"); g_pdl = (e && e[0] == '1') ? 1 : 0; }
    return g_pdl;
}
extern "C" int mmlst_set_pdl(int on) { const int prev = mmlst_pdl_enabled(); if (on == 0 || on == 1) g_pdl = on; return prev; }

extern "C" const char* mmlst_last_error(void) { return g_err; }
extern "C" int mmlst_version(void) { return MMLST_VERSION; }
extern "C" int mmlst_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

extern "C" void* mmlst_pinned_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
        mmlst_set_error("cudaHostAlloc(%zu) failed", bytes);
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
extern "C" void mmlst_pinned_free(void* p) { if (p) cudaFreeHost(p); }

// ---------------------------------------------------------------------------------------------------------------
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return MMLST_OK;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { cudaGetLastError(); mmlst_set_error("cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e)); return MMLST_E_NOMEM; }
        cap = want;
        return MMLST_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T* as() { return static_cast<T*>(p); }
};

struct mmlst_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    // score stream
    DevBuf tid, as0, xm3, qlen, oidx, allow, locus_of, sum_as, n_hit, first_idx, counters;
    DevBuf run_tid, run_start, chunk_run;  // run-length form (mmlst_score_runs_dev)
    DevBuf chunk_qlen;                     // + len(SEQ) per chunk (mmlst_score_runs_qc_dev)
    bool resident_qlen = false;            // explicit qlen[] present (false after a QC upload until mmlst_coverage expands it)
    uint64_t resident_n = 0;     // records of the score stream currently in (tid/)as0/xm3/qlen(/oidx)
    bool resident_oidx = false;
    bool resident_tid = false;   // explicit tid[] present (false after a run-length upload until mmlst_coverage expands it)
    uint32_t resident_runs = 0;
    // coverage (H7)
    DevBuf qhash, cov_table, cov;
    // pileup stream (chosen contigs only)
    DevBuf p_recs, planes, chunks, counts, dbseq, col_off, cons, holes, snps;
    DevBuf cs_scratch, cs_off, cs_out;   // contig statistics (mmlst_contig_stats): tile sums, the three prefixes, compacted columns
    // hamming
    DevBuf db_hi, db_lo, db_len, q_hi, q_lo, q_len, blocks, best;
    DevBuf xr_ids, xr_x, xr_bytes, xq_ids, xq_x, xq_bytes;  // flagged (non-ACGT) rows / queries, H9
    uint32_t db_rows = 0, db_W = 0, db_n_xr = 0;
    // ST assignment (defineProfile): the `profiles` table grouped by profile, resident across queries
    DevBuf zbuf, zact;                     // compressed score stream + the sizes the decompression engine reports
    std::vector<uint32_t> zlen; uint32_t z_pending = 0;
    DevBuf zpbuf, zpact;                   // compressed pileup stream of the chosen contigs (mmlst_soa.zp) + the sizes the engine reports
    std::vector<uint32_t> zplen; uint32_t zp_pending = 0;
    DevBuf prof_start, prof_allele, st_q, st_qn, st_count, st_best, st_nbest, st_out, first_row, row_key;
    uint32_t n_st = 0;
    bool has_row_key = false;
    // resident allele index + result staging of mmlst_sample (mmlst_index_upload)
    DevBuf ix_locus_of, ix_locus_rows, ix_locus_start, ix_allele_num, ix_species_of_locus, ix_genes_in_db, ix_db_ascii, ix_db_off, ix_bam_ln, ix_zero64, ix_scratch,
           ix_out, ix_db_start, ix_chunks;
    uint32_t ix_n_ref = 0, ix_n_loci = 0, ix_n_species = 0;
    bool ix_rows_identity = false;   // allele rows already grouped by locus: mmlst_select_dev gets no row list
    std::vector<uint32_t> ix_bam_ln_h; std::vector<uint64_t> ix_db_off_h;
    // copy lanes: the pileup records of the chosen contigs are ~2 ranges per contig; spread over a few streams their DMA set-up overlaps
    static constexpr int kLanes = 3;
    cudaStream_t lane[kLanes] = {nullptr, nullptr, nullptr};
    cudaEvent_t lane_ev[kLanes + 1] = {nullptr, nullptr, nullptr, nullptr};
    int lanes_init() {
        if (lane[0]) return MMLST_OK;
        for (int i = 0; i < kLanes; ++i) CUDA_TRY(cudaStreamCreateWithFlags(&lane[i], cudaStreamNonBlocking));
        for (int i = 0; i <= kLanes; ++i) CUDA_TRY(cudaEventCreateWithFlags(&lane_ev[i], cudaEventDisableTiming));
        return MMLST_OK;
    }
    void* pin = nullptr; size_t pin_cap = 0;   // page-locked staging for the results of mmlst_sample
    int pin_reserve(size_t bytes) {
        if (bytes <= pin_cap) return MMLST_OK;
        if (pin) cudaFreeHost(pin);
        pin = nullptr; pin_cap = 0;
        cudaError_t e = cudaHostAlloc(&pin, bytes + bytes / 8 + 256, cudaHostAllocDefault);
        if (e != cudaSuccess) { cudaGetLastError(); mmlst_set_error("cudaHostAlloc(%zu) failed: %s", bytes, cudaGetErrorString(e)); return MMLST_E_NOMEM; }
        pin_cap = bytes + bytes / 8 + 256;
        return MMLST_OK;
    }
    DevBuf* all[80];
    int n_all = 0;
    mmlst_ctx() {
        DevBuf* l[] = {&tid, &as0, &xm3, &qlen, &oidx, &allow, &locus_of, &sum_as, &n_hit, &first_idx, &counters, &p_recs,
                       &planes, &chunks, &counts, &dbseq, &col_off, &cons, &holes, &snps, &db_hi,
                       &db_lo, &db_len, &q_hi, &q_lo, &q_len, &blocks, &best, &qhash, &cov_table, &cov, &xr_ids, &xr_x, &xr_bytes, &xq_ids, &xq_x, &xq_bytes,
                       &run_tid, &run_start, &chunk_run, &chunk_qlen, &prof_start, &prof_allele, &st_q, &st_qn, &st_count, &st_best, &st_nbest, &st_out,
                       &first_row, &row_key, &zbuf, &zact, &zpbuf, &zpact, &ix_locus_of, &ix_locus_rows, &ix_locus_start, &ix_allele_num, &ix_species_of_locus, &ix_genes_in_db, &ix_db_ascii,
                       &ix_db_off, &ix_bam_ln, &ix_zero64, &ix_scratch, &ix_out, &ix_db_start, &ix_chunks, &cs_scratch, &cs_off, &cs_out};
        for (DevBuf* b : l) all[n_all++] = b;
    }
};

#define CTX_ENTER(ctx)                                                        \
    if (!(ctx)) { mmlst_set_error("null context"); return MMLST_E_ARG; }      \
    CUDA_TRY(cudaSetDevice((ctx)->device))
#define TRY(expr) do { int _r = (expr); if (_r != MMLST_OK) return _r; } while (0)

extern "C" int mmlst_create(int device, mmlst_ctx** out) {
    if (!out) { mmlst_set_error("mmlst_create: null out"); return MMLST_E_ARG; }
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        mmlst_set_error("no CUDA device available (%s); libmmlst has no CPU fallback", e == cudaSuccess ? "count=0" : cudaGetErrorString(e));
        return MMLST_E_CUDA;
    }
    if (device < 0 || device >= n) { mmlst_set_error("device %d out of range (0..%d)", device, n - 1); return MMLST_E_ARG; }
    CUDA_TRY(cudaSetDevice(device));
    mmlst_ctx* c = new mmlst_ctx();
    c->device = device;
    e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { delete c; return mmlst_cuda_fail(e, "cudaStreamCreate"); }
    *out = c;
    return MMLST_OK;
}

extern "C" void mmlst_destroy(mmlst_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    for (int i = 0; i < c->n_all; ++i) c->all[i]->release();
    if (c->pin) cudaFreeHost(c->pin);
    for (int i = 0; i < mmlst_ctx::kLanes; ++i) if (c->lane[i]) cudaStreamDestroy(c->lane[i]);
    for (int i = 0; i <= mmlst_ctx::kLanes; ++i) if (c->lane_ev[i]) cudaEventDestroy(c->lane_ev[i]);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}
extern "C" void* mmlst_stream(mmlst_ctx* c) { return c ? c->stream : nullptr; }
extern "C" int mmlst_sync(mmlst_ctx* c) {
    CTX_ENTER(c);
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return MMLST_OK;
}

template <class T>
static int h2d(DevBuf& b, const T* src, size_t n, cudaStream_t s) {
    TRY(b.reserve(n * sizeof(T)));
    if (n) CUDA_TRY(cudaMemcpyAsync(b.p, src, n * sizeof(T), cudaMemcpyHostToDevice, s));
    return MMLST_OK;
}

// score stream host -> device: the run-length form (5 B / record + run arrays) when the caller provides it, else explicit tid
static int upload_score_stream(mmlst_ctx* c, const mmlst_soa* soa) {
    cudaStream_t s = c->stream;
    const size_t n = soa->n_rec;
    const bool runs = soa->run_tid != nullptr && n != 0;
    if (runs) {
        if (!soa->run_start || !soa->chunk_run || !soa->n_runs) { mmlst_set_error("mmlst_soa: run_tid without run_start / chunk_run / n_runs"); return MMLST_E_ARG; }
        if (soa->run_start[0] != 0 || soa->run_start[soa->n_runs] != n) { mmlst_set_error("mmlst_soa: run_start does not span the %zu records", n); return MMLST_E_ARG; }
        TRY(h2d(c->run_tid, soa->run_tid, (size_t)soa->n_runs, s));
        TRY(h2d(c->run_start, soa->run_start, (size_t)soa->n_runs + 1, s));
        TRY(h2d(c->chunk_run, soa->chunk_run, (n + 255) / 256, s));
    } else {
        if (n && !soa->tid) { mmlst_set_error("mmlst_soa: neither tid nor run arrays given"); return MMLST_E_ARG; }
        TRY(h2d(c->tid, soa->tid, n, s));
    }
    const bool qc = runs && soa->chunk_qlen != nullptr;
    if (runs && soa->z && soa->z->n_blocks) {
        // compressed form: the DEFLATE blocks cross PCIe, the hardware decompression engine writes as0[] / xm3[] in HBM (csrc/de.cu)
        const mmlst_zstream* z = soa->z;
        if (!z->bytes || !z->table) { mmlst_set_error("mmlst_soa.z: null pointer"); return MMLST_E_ARG; }
        TRY(c->as0.reserve(n * 2)); TRY(c->xm3.reserve(n)); TRY(c->zbuf.reserve(z->n_bytes + 64)); TRY(c->zact.reserve((size_t)z->n_blocks * 4));
        std::vector<CUmemDecompressParams> prm(z->n_blocks);
        std::vector<uint64_t> src_off(z->n_blocks);
        memset(prm.data(), 0, sizeof(CUmemDecompressParams) * z->n_blocks);
        c->zlen.resize(z->n_blocks);
        uint64_t covered[2] = {0, 0};   // the blocks of an array tile a PREFIX of it, in order; the rest of the array ships plain
        for (uint32_t b = 0; b < z->n_blocks; ++b) {
            const uint64_t* t = z->table + 4 * (size_t)b;
            const uint64_t clen = t[3] >> 32, ulen = t[3] & 0xffffffffull;
            const size_t cap = t[0] == 0 ? n * 2 : n;
            if (t[0] > 1 || t[1] != covered[t[0] & 1] || t[1] + ulen > cap || t[2] + clen > z->n_bytes || (b && t[2] < z->table[4 * (size_t)(b - 1) + 2]) || ulen > (4u << 20)) {
                mmlst_set_error("mmlst_soa.z: block %u out of range / out of order (the blocks of an array must tile a prefix of it)", b);
                return MMLST_E_ARG;
            }
            covered[t[0]] += ulen;
            prm[b].srcNumBytes = clen; prm[b].dstNumBytes = ulen; prm[b].dstActBytes = c->zact.as<cuuint32_t>() + b;
            prm[b].src = c->zbuf.as<uint8_t>() + t[2];
            prm[b].dst = (t[0] == 0 ? c->as0.as<uint8_t>() : c->xm3.as<uint8_t>()) + t[1];
            prm[b].algo = CU_MEM_DECOMPRESS_ALGORITHM_DEFLATE;
            src_off[b] = t[2];
            c->zlen[b] = (uint32_t)ulen;
        }
        std::vector<MmlstPlainCopy> plain;
        if (covered[0] < n * 2) {
            if (!soa->as0) { mmlst_set_error("mmlst_soa.z covers %llu of %llu bytes of as0[] and as0 is NULL", (unsigned long long)covered[0], (unsigned long long)(n * 2)); return MMLST_E_ARG; }
            plain.push_back({c->as0.as<uint8_t>() + covered[0], reinterpret_cast<const uint8_t*>(soa->as0) + covered[0], (size_t)(n * 2 - covered[0])});
        }
        if (covered[1] < n) {
            if (!soa->xm3) { mmlst_set_error("mmlst_soa.z covers %llu of %llu bytes of xm3[] and xm3 is NULL", (unsigned long long)covered[1], (unsigned long long)n); return MMLST_E_ARG; }
            plain.push_back({c->xm3.as<uint8_t>() + covered[1], soa->xm3 + covered[1], (size_t)(n - covered[1])});
        }
        mmlst_trace_mark("params_built");
        TRY(mmlst_h2d_inflate(c->device, s, c->zbuf.as<uint8_t>(), z->bytes, z->n_bytes, prm, src_off, &plain, 3));
        c->z_pending = z->n_blocks;
        if (z->as_xm_coeff) {   // the blocks hold as0 + coeff * xm3 over the covered prefix: back to as0 once both arrays are complete on the device
            if (z->as_xm_coeff < -256 || z->as_xm_coeff > 256) { mmlst_set_error("mmlst_soa.z: as_xm_coeff %d out of range", z->as_xm_coeff); return MMLST_E_ARG; }
            TRY(mmlst_as_untransform_dev(c->as0.as<int16_t>(), c->xm3.as<uint8_t>(), covered[0] / 2, z->as_xm_coeff, s));
        }
    } else {
        TRY(h2d(c->as0, soa->as0, n, s));
        TRY(h2d(c->xm3, soa->xm3, n, s));
    }
    if (qc) TRY(h2d(c->chunk_qlen, soa->chunk_qlen, (n + 255) / 256, s));
    else TRY(h2d(c->qlen, soa->qlen, n, s));
    c->resident_qlen = !qc;
    if (soa->orig_idx) TRY(h2d(c->oidx, soa->orig_idx, n, s));
    c->resident_n = n; c->resident_oidx = soa->orig_idx != nullptr;
    c->resident_tid = !runs; c->resident_runs = runs ? soa->n_runs : 0;
    return MMLST_OK;
}

// HOST: run arrays of a tid[] (include/mmlst.h, mmlst_score_runs_dev)
extern "C" int mmlst_build_runs(const uint32_t* tid, uint64_t n_rec, uint32_t* run_tid, uint32_t* run_start, uint32_t* chunk_run,
                                uint32_t* n_runs) {
    if (!n_runs || (n_rec && !tid)) { mmlst_set_error("mmlst_build_runs: null pointer"); return MMLST_E_ARG; }
    if (n_rec >= 0xffffff00ull) { mmlst_set_error("mmlst_build_runs: %llu records do not fit 32-bit run offsets", (unsigned long long)n_rec); return MMLST_E_RANGE; }
    if (!run_tid) {
        uint64_t r = n_rec ? 1 : 0;
        for (uint64_t i = 1; i < n_rec; ++i) r += tid[i] != tid[i - 1];
        *n_runs = (uint32_t)r;
        return MMLST_OK;
    }
    if (!run_start || !chunk_run) { mmlst_set_error("mmlst_build_runs: null pointer"); return MMLST_E_ARG; }
    const uint32_t cap = *n_runs;
    uint32_t r = 0;
    for (uint64_t i = 0; i < n_rec; ++i) {
        if (i == 0 || tid[i] != tid[i - 1]) {
            if (r >= cap) { mmlst_set_error("mmlst_build_runs: more than %u runs", cap); return MMLST_E_ARG; }
            run_tid[r] = tid[i]; run_start[r] = (uint32_t)i; ++r;
        }
        if ((i & 255u) == 0) chunk_run[i >> 8] = r - 1;
    }
    run_start[r] = (uint32_t)n_rec;
    *n_runs = r;
    return MMLST_OK;
}

// HOST: len(SEQ) per 256-record chunk when every chunk is uniform (include/mmlst.h, mmlst_score_runs_qc_dev)
extern "C" int mmlst_chunk_qlen(const uint16_t* qlen, uint64_t n_rec, uint16_t* chunk_qlen, int* uniform) {
    if (!uniform || (n_rec && (!qlen || !chunk_qlen))) { mmlst_set_error("mmlst_chunk_qlen: null pointer"); return MMLST_E_ARG; }
    *uniform = 1;
    for (uint64_t c0 = 0; c0 < n_rec; c0 += 256) {
        const uint64_t c1 = c0 + 256 < n_rec ? c0 + 256 : n_rec;
        const uint16_t q = qlen[c0];
        unsigned diff = 0;
        for (uint64_t i = c0 + 1; i < c1; ++i) diff |= (unsigned)(qlen[i] ^ q);
        if (diff) { *uniform = 0; return MMLST_OK; }
        chunk_qlen[c0 >> 8] = q;
    }
    return MMLST_OK;
}

// the score kernel over the stream upload_score_stream() left in the context (the form follows what was uploaded), tables zeroed first
static int launch_resident_score(mmlst_ctx* c, const mmlst_soa* soa, const mmlst_score_params* prm, const uint32_t* locus_of_dev) {
    cudaStream_t s = c->stream;
    const size_t n = soa->n_rec, nr = soa->n_ref;
    TRY(c->sum_as.reserve(nr * 8)); TRY(c->n_hit.reserve(nr * 4)); TRY(c->first_idx.reserve(nr * 4 + 4)); TRY(c->counters.reserve(16));
    CUDA_TRY(cudaMemsetAsync(c->sum_as.p, 0, nr * 8, s));
    CUDA_TRY(cudaMemsetAsync(c->n_hit.p, 0, nr * 4, s));
    CUDA_TRY(cudaMemsetAsync(c->first_idx.p, 0xff, nr * 4, s));
    CUDA_TRY(cudaMemsetAsync(c->counters.p, 0, 16, s));
    if (c->resident_runs && !c->resident_qlen) {
        TRY(mmlst_score_runs_qc_dev(c->run_tid.as<uint32_t>(), c->run_start.as<uint32_t>(), c->resident_runs, c->chunk_run.as<uint32_t>(),
                                    c->chunk_qlen.as<uint16_t>(), c->as0.as<int16_t>(), c->xm3.as<uint8_t>(),
                                    soa->orig_idx ? c->oidx.as<uint32_t>() : nullptr, n, 0, c->allow.as<uint8_t>(), (uint32_t)nr,
                                    prm->minscore, prm->max_xm, prm->min_read_len, c->sum_as.as<int64_t>(), c->n_hit.as<uint32_t>(),
                                    c->first_idx.as<uint32_t>(), c->counters.as<uint64_t>(), s));
    } else if (c->resident_runs) {
        TRY(mmlst_score_runs_dev(c->run_tid.as<uint32_t>(), c->run_start.as<uint32_t>(), c->resident_runs, c->chunk_run.as<uint32_t>(),
                                 c->as0.as<int16_t>(), c->xm3.as<uint8_t>(), c->qlen.as<uint16_t>(),
                                 soa->orig_idx ? c->oidx.as<uint32_t>() : nullptr, n, 0, c->allow.as<uint8_t>(), (uint32_t)nr,
                                 prm->minscore, prm->max_xm, prm->min_read_len, c->sum_as.as<int64_t>(), c->n_hit.as<uint32_t>(),
                                 c->first_idx.as<uint32_t>(), c->counters.as<uint64_t>(), s));
    } else {
        TRY(mmlst_score_dev(c->tid.as<uint32_t>(), c->as0.as<int16_t>(), c->xm3.as<uint8_t>(), c->qlen.as<uint16_t>(),
                            soa->orig_idx ? c->oidx.as<uint32_t>() : nullptr, n, 0, c->allow.as<uint8_t>(),
                            locus_of_dev, (uint32_t)nr, prm->minscore, prm->max_xm, prm->min_read_len,
                            c->sum_as.as<int64_t>(), c->n_hit.as<uint32_t>(), c->first_idx.as<uint32_t>(),
                            c->counters.as<uint64_t>(), s));
    }
    return MMLST_OK;
}

// ---------------------------------------------------------------------------------------------------------------
extern "C" int mmlst_score(mmlst_ctx* c, const mmlst_soa* soa, const uint8_t* allow, const uint32_t* locus_of,
                           uint32_t n_loci, const mmlst_score_params* prm, int64_t* sum_as, uint32_t* n_hit,
                           uint32_t* first_idx, uint64_t* counters) {
    CTX_ENTER(c);
    if (!soa || !allow || !locus_of || !prm || !sum_as || !n_hit || !first_idx || !counters) { mmlst_set_error("mmlst_score: null pointer"); return MMLST_E_ARG; }
    cudaStream_t s = c->stream;
    const size_t n = soa->n_rec, nr = soa->n_ref;
    mmlst_trace_mark("enter");
    TRY(upload_score_stream(c, soa));
    mmlst_trace_mark("upload_enqueued");
    TRY(h2d(c->allow, allow, nr, s));
    TRY(h2d(c->locus_of, locus_of, nr, s));
    TRY(launch_resident_score(c, soa, prm, c->locus_of.as<uint32_t>()));
    CUDA_TRY(cudaMemcpyAsync(sum_as, c->sum_as.p, nr * 8, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(n_hit, c->n_hit.p, nr * 4, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(first_idx, c->first_idx.p, nr * 4, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(counters, c->counters.p, 16, cudaMemcpyDeviceToHost, s));
    std::vector<uint32_t> zact;
    if (c->z_pending) {
        zact.resize(c->z_pending);
        CUDA_TRY(cudaMemcpyAsync(zact.data(), c->zact.p, (size_t)c->z_pending * 4, cudaMemcpyDeviceToHost, s));
    }
    mmlst_trace_mark("kernel_d2h_enqueued");
    CUDA_TRY(cudaStreamSynchronize(s));
    mmlst_trace_mark("sync");
    mmlst_trace_flush("mmlst_score");
    for (uint32_t b = 0; b < c->z_pending; ++b) {
        if (zact[b] != c->zlen[b]) {
            c->z_pending = 0;
            mmlst_set_error("mmlst_score: block %u of the compressed score stream inflated to %u bytes, %u expected (corrupt mmlst_soa.z)", b, zact[b], c->zlen[b]);
            return MMLST_E_ARG;
        }
    }
    c->z_pending = 0;
    return MMLST_OK;
}

// ---------------------------------------------------------------------------------------------------------------
extern "C" int mmlst_coverage(mmlst_ctx* c, const mmlst_soa* soa, const uint64_t* qhash, const uint8_t* allow,
                              const uint32_t* locus_of, uint32_t n_loci, const mmlst_score_params* prm, uint32_t flags,
                              uint64_t* cov) {
    CTX_ENTER(c);
    if (!soa || !qhash || !allow || !locus_of || !prm || !cov) { mmlst_set_error("mmlst_coverage: null pointer"); return MMLST_E_ARG; }
    cudaStream_t s = c->stream;
    const size_t n = soa->n_rec, nr = soa->n_ref;
    if (flags & MMLST_COVERAGE_STREAM_RESIDENT) {
        if (c->resident_n != n || c->resident_oidx != (soa->orig_idx != nullptr)) {
            mmlst_set_error("mmlst_coverage: MMLST_COVERAGE_STREAM_RESIDENT but the context holds %llu records, the stream has %llu",
                            (unsigned long long)c->resident_n, (unsigned long long)n);
            return MMLST_E_ARG;
        }
    } else {
        TRY(upload_score_stream(c, soa));
    }
    if (!c->resident_tid && n) {  // run-length upload: the coverage kernel wants the explicit allele id per record
        TRY(c->tid.reserve(n * 4));
        TRY(mmlst_expand_runs_dev(c->run_tid.as<uint32_t>(), c->run_start.as<uint32_t>(), c->resident_runs, c->chunk_run.as<uint32_t>(),
                                  n, c->tid.as<uint32_t>(), s));
        c->resident_tid = true;
    }
    if (!c->resident_qlen && n) {  // QC upload: the coverage kernel sums len(SEQ) per record
        TRY(c->qlen.reserve(n * 2));
        TRY(mmlst_expand_chunk_qlen_dev(c->chunk_qlen.as<uint16_t>(), n, c->qlen.as<uint16_t>(), s));
        c->resident_qlen = true;
    }
    TRY(h2d(c->qhash, qhash, 2 * n, s));
    TRY(h2d(c->allow, allow, nr, s));
    TRY(h2d(c->locus_of, locus_of, nr, s));
    const uint64_t slots = mmlst_coverage_table_slots(n);
    TRY(c->cov_table.reserve(slots * 24));
    TRY(c->cov.reserve((size_t)n_loci * 8 + 8));
    CUDA_TRY(cudaMemsetAsync(c->cov_table.p, 0, slots * 24, s));
    CUDA_TRY(cudaMemsetAsync(c->cov.p, 0, (size_t)n_loci * 8 + 8, s));
    TRY(mmlst_coverage_dev(c->tid.as<uint32_t>(), c->as0.as<int16_t>(), c->xm3.as<uint8_t>(), c->qlen.as<uint16_t>(),
                           soa->orig_idx ? c->oidx.as<uint32_t>() : nullptr, c->qhash.as<uint64_t>(), n, 0, c->allow.as<uint8_t>(),
                           c->locus_of.as<uint32_t>(), (uint32_t)nr, prm->minscore, prm->max_xm, prm->min_read_len,
                           c->cov_table.p, slots, c->cov.as<uint64_t>(), s));
    CUDA_TRY(cudaMemcpyAsync(cov, c->cov.p, (size_t)n_loci * 8, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return MMLST_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Chunk length (records) for a launch over n_rec records: two chunks per SM (one resident wave of the bit-sliced kernel --
// every (chunk, column word) pair costs one cross-lane flush, so chunks are as long as a full wave allows), whole
// 512-record tiles.
extern "C" uint32_t mmlst_chunk_records(uint64_t n_rec) {
    return 512u * mmlst_chunk_tiles(n_rec, (uint32_t)mmlst_num_sms() * MMLST_CHUNKS_PER_SM);
}

extern "C" int mmlst_pileup_dev(const mmlst_prec* recs, const uint32_t* planes, const mmlst_chunk* chunks, uint32_t n_chunks,
                                uint32_t max_row_words, int minscore, int max_xm, uint32_t* counts, uint32_t total_cols,
                                int impl, void* stream) {
    if (n_chunks == 0) return MMLST_OK;
    if (!recs || !planes || !chunks || !counts) { mmlst_set_error("mmlst_pileup_dev: null pointer"); return MMLST_E_ARG; }
    if ((reinterpret_cast<uintptr_t>(recs) & 15) || (reinterpret_cast<uintptr_t>(planes) & 15)) { mmlst_set_error("mmlst_pileup_dev: recs and planes must be 16-byte aligned"); return MMLST_E_ARG; }
    PileupArgs a{recs, planes, chunks, n_chunks, max_row_words, minscore, max_xm, counts, total_cols, nullptr};
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (impl == 1) return launch_pileup_atomic(a, s);
    if (impl == 0 || impl == 2) return launch_pileup_bitsliced(a, s);
    mmlst_set_error("mmlst_pileup_dev: impl %d unknown", impl);
    return MMLST_E_ARG;
}

// chunk list and count produced on the device by mmlst_select_dev (header[1] = n_chunks)
extern "C" int mmlst_pileup_indirect_dev(const mmlst_prec* recs, const uint32_t* planes, const mmlst_chunk* chunks,
                                         const uint32_t* header, uint32_t max_row_words, int minscore, int max_xm, uint32_t* counts,
                                         int impl, void* stream) {
    if (!recs || !planes || !chunks || !header || !counts) { mmlst_set_error("mmlst_pileup_indirect_dev: null pointer"); return MMLST_E_ARG; }
    if ((reinterpret_cast<uintptr_t>(recs) & 15) || (reinterpret_cast<uintptr_t>(planes) & 15)) { mmlst_set_error("mmlst_pileup_indirect_dev: recs and planes must be 16-byte aligned"); return MMLST_E_ARG; }
    PileupArgs a{recs, planes, chunks, 0, max_row_words, minscore, max_xm, counts, 0, header + 1, FusedConsensus{}};
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (impl == 1) return launch_pileup_atomic(a, s);
    if (impl == 0 || impl == 2) return launch_pileup_bitsliced(a, s);
    mmlst_set_error("mmlst_pileup_indirect_dev: impl %d unknown", impl);
    return MMLST_E_ARG;
}

// pileup AND consensus of a device-driven pass in one launch (see FusedConsensus in pileup.cuh); falls back to the two launches when the rows do not
// fit the bit-sliced kernel's shared memory.  ticket: device u32[max_loci], zeroed once by the caller (every call leaves it zeroed).
extern "C" int mmlst_consensus_indirect_dev(uint32_t*, const uint8_t*, const uint64_t*, const uint32_t*, uint32_t, const uint32_t*, uint32_t, uint8_t*, uint32_t*,
                                            uint32_t*, uint32_t, void*);
extern "C" int mmlst_pileup_consensus_indirect_dev(const mmlst_prec* recs, const uint32_t* planes, const mmlst_chunk* chunks, const uint32_t* header,
                                                   uint32_t max_row_words, int minscore, int max_xm, uint32_t* counts, const uint8_t* db_ascii,
                                                   const uint64_t* db_start, const uint32_t* col_off, uint32_t max_loci, uint32_t mincov, uint8_t* cons,
                                                   uint32_t* holes, uint32_t* snps, uint32_t flags, uint32_t* ticket, void* stream) {
    if (!recs || !planes || !chunks || !header || !counts || !db_ascii || !db_start || !col_off || !cons || !holes || !snps || !ticket) {
        mmlst_set_error("mmlst_pileup_consensus_indirect_dev: null pointer");
        return MMLST_E_ARG;
    }
    if ((reinterpret_cast<uintptr_t>(recs) & 15) || (reinterpret_cast<uintptr_t>(planes) & 15)) { mmlst_set_error("mmlst_pileup_consensus_indirect_dev: recs and planes must be 16-byte aligned"); return MMLST_E_ARG; }
    PileupArgs a{recs, planes, chunks, 0, max_row_words, minscore, max_xm, counts, 0, header + 1,
                 FusedConsensus{ticket, db_ascii, reinterpret_cast<const unsigned long long*>(db_start), col_off, mincov, cons, holes, snps,
                                (flags & MMLST_CONSENSUS_CONSUME) ? 1u : 0u}};
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (mmlst_pileup_bitsliced_fits(max_row_words)) return launch_pileup_bitsliced(a, s);
    a.fc = FusedConsensus{};
    TRY(launch_pileup_atomic(a, s));
    return mmlst_consensus_indirect_dev(counts, db_ascii, db_start, col_off, max_loci, header, mincov, cons, holes, snps, flags, stream);
}

// The pileup records and plane rows of the chosen contigs (contiguous ranges of the coordinate-sorted stream) host -> device, packed one after the
// other, plus the chunk list over them.  The copies are dealt over the context's copy lanes; `s` continues when all of them have landed.
// `runs`: a run of consecutive tids is one record range and one plane range of the stream and crosses the bus as one copy of each (plain
// stream only; its chunks share the run's plane_delta).
static int upload_chosen_contigs(mmlst_ctx* c, const mmlst_soa* soa, const uint32_t* chosen_tid, uint32_t n_loci, const uint32_t* col_off,
                                 std::vector<mmlst_chunk>& chunks, bool use_zp = false, bool runs = false) {
    cudaStream_t s = c->stream;
    auto row_end = [&](uint64_t r) { return soa->p_recs[r].row_off + mmlst_row_words(soa->p_recs[r].nw); };
    // end of the run that starts at chosen_tid[l] (exclusive index into chosen_tid)
    auto run_end = [&](uint32_t l) { uint32_t e = l + 1; while (runs && e < n_loci && chosen_tid[e] == chosen_tid[e - 1] + 1) ++e; return e; };
    size_t n_rec = 0, n_words = 0;
    for (uint32_t l = 0; l < n_loci; ++l) {
        const uint32_t t = chosen_tid[l];
        if (t >= soa->n_ref) { mmlst_set_error("chosen_tid[%u]=%u out of range", l, t); return MMLST_E_ARG; }
    }
    for (uint32_t l = 0, e; l < n_loci; l = e) {
        e = run_end(l);
        const uint64_t r0 = soa->contig_start[chosen_tid[l]], r1 = soa->contig_start[chosen_tid[e - 1] + 1];
        if (r1 <= r0) continue;
        n_rec += r1 - r0;
        n_words += (size_t)row_end(r1 - 1) - soa->p_recs[r0].row_off + 4;  // +4: every range starts 16-byte aligned on the device
    }
    TRY(c->p_recs.reserve(n_rec * sizeof(mmlst_prec) + 64)); TRY(c->planes.reserve(n_words * 4 + 64));
    c->zp_pending = 0;
    if (use_zp && soa->zp && soa->zp->n_blocks && mmlst_de_available(c->device) == MMLST_OK) {
        // compressed form: the chosen contigs' DEFLATE blocks cross the bus, the hardware decompression engine writes the records and plane rows in HBM
        const mmlst_zpileup* z = soa->zp;
        if (!z->bytes || !z->table || !z->contig_block) { mmlst_set_error("mmlst_soa.zp: null pointer"); return MMLST_E_ARG; }
        std::vector<MmlstSegment> segs;
        std::vector<uint32_t> first_block(1, 0u);
        std::vector<CUmemDecompressParams> prm;
        size_t zbytes = 0, nb = 0;
        for (uint32_t l = 0; l < n_loci; ++l) {
            const uint32_t t = chosen_tid[l];
            if (soa->contig_start[t + 1] <= soa->contig_start[t]) continue;
            const uint32_t b0 = z->contig_block[t], b1 = z->contig_block[t + 1];
            if (b0 >= b1 || b1 > z->n_blocks) { mmlst_set_error("mmlst_soa.zp: contig %u has records but no blocks", t); return MMLST_E_ARG; }
            const uint64_t s0 = z->table[2 * (size_t)b0], s1 = z->table[2 * (size_t)(b1 - 1)] + ((z->table[2 * (size_t)(b1 - 1) + 1] >> 32) & 0x7fffffffull);
            if (s1 < s0 || s1 > z->n_bytes) { mmlst_set_error("mmlst_soa.zp: blocks of contig %u out of range", t); return MMLST_E_ARG; }
            zbytes += ((s1 - s0) + 63) & ~(size_t)63;
            nb += b1 - b0;
        }
        TRY(c->zpbuf.reserve(zbytes + 64)); TRY(c->zpact.reserve(nb * 4 + 4));
        prm.resize(nb);
        memset(prm.data(), 0, sizeof(CUmemDecompressParams) * nb);
        c->zplen.resize(nb);
        chunks.clear();
        const uint32_t kChunkRecords = mmlst_chunk_records(n_rec);
        size_t rbase = 0, wbase = 0, zoff = 0, q = 0;
        for (uint32_t l = 0; l < n_loci; ++l) {
            const uint32_t t = chosen_tid[l];
            const uint64_t r0 = soa->contig_start[t], r1 = soa->contig_start[t + 1];
            const size_t nr = r1 - r0;
            if (nr == 0) continue;
            const uint32_t w0 = soa->p_recs[r0].row_off, w1 = row_end(r1 - 1);
            const uint32_t b0 = z->contig_block[t], b1 = z->contig_block[t + 1];
            const uint64_t s0 = z->table[2 * (size_t)b0], s1 = z->table[2 * (size_t)(b1 - 1)] + ((z->table[2 * (size_t)(b1 - 1) + 1] >> 32) & 0x7fffffffull);
            segs.push_back({c->zpbuf.as<uint8_t>() + zoff, z->bytes + s0, (size_t)(s1 - s0)});
            size_t done[2] = {0, 0};   // inflated bytes of the contig's plane rows / records placed so far
            for (uint32_t b = b0; b < b1; ++b, ++q) {
                const uint64_t off = z->table[2 * (size_t)b], w = z->table[2 * (size_t)b + 1];
                const unsigned kind = (unsigned)(w >> 63);
                const uint64_t clen = (w >> 32) & 0x7fffffffull, ulen = w & 0xffffffffull;
                const size_t cap = kind ? nr * sizeof(mmlst_prec) : (size_t)(w1 - w0) * 4;
                if (off < s0 || off + clen > s1 || (b > b0 && off < z->table[2 * (size_t)(b - 1)]) || done[kind] + ulen > cap || ulen > (4u << 20)) {
                    mmlst_set_error("mmlst_soa.zp: block %u of contig %u out of range / out of order", b, t);
                    return MMLST_E_ARG;
                }
                prm[q].srcNumBytes = clen; prm[q].dstNumBytes = ulen; prm[q].dstActBytes = c->zpact.as<cuuint32_t>() + q;
                prm[q].src = c->zpbuf.as<uint8_t>() + zoff + (off - s0);
                prm[q].dst = kind ? reinterpret_cast<uint8_t*>(c->p_recs.as<mmlst_prec>() + rbase) + done[1] : reinterpret_cast<uint8_t*>(c->planes.as<uint32_t>() + wbase) + done[0];
                prm[q].algo = CU_MEM_DECOMPRESS_ALGORITHM_DEFLATE;
                c->zplen[q] = (uint32_t)ulen;
                done[kind] += ulen;
            }
            if (done[0] != (size_t)(w1 - w0) * 4 || done[1] != nr * sizeof(mmlst_prec)) {
                mmlst_set_error("mmlst_soa.zp: the blocks of contig %u inflate to %zu + %zu bytes, the stream has %zu + %zu", t, done[0], done[1], (size_t)(w1 - w0) * 4, nr * sizeof(mmlst_prec));
                return MMLST_E_ARG;
            }
            first_block.push_back((uint32_t)q);
            zoff += ((size_t)(s1 - s0) + 63) & ~(size_t)63;
            for (size_t b = 0; b < nr; b += kChunkRecords) {
                mmlst_chunk ck{};
                ck.rec_begin = (uint32_t)(rbase + b);
                ck.rec_end = (uint32_t)(rbase + std::min(nr, b + kChunkRecords));
                ck.col_base = col_off[l];
                ck.contig_len = col_off[l + 1] - col_off[l];
                ck.plane_delta = (uint32_t)wbase - w0;
                chunks.push_back(ck);
            }
            rbase += nr;
            wbase += (size_t)(w1 - w0);
            wbase = (wbase + 3) & ~(size_t)3;
        }
        TRY(h2d(c->chunks, chunks.data(), chunks.size(), s));   // ahead of the blocks on `s`: tiny, and `s` is idle until the first group lands
        TRY(mmlst_h2d_inflate_segments(c->device, s, segs, prm, first_block, 6));
        c->zp_pending = (uint32_t)nb;
        return MMLST_OK;
    }
    TRY(c->lanes_init());
    CUDA_TRY(cudaEventRecord(c->lane_ev[mmlst_ctx::kLanes], s));   // the buffers may still be read by earlier work of `s`
    for (int i = 0; i < mmlst_ctx::kLanes; ++i) CUDA_TRY(cudaStreamWaitEvent(c->lane[i], c->lane_ev[mmlst_ctx::kLanes], 0));
    chunks.clear();
    const uint32_t kChunkRecords = mmlst_chunk_records(n_rec);
    size_t rbase = 0, wbase = 0;
    int k = 0;
    for (uint32_t l = 0, e; l < n_loci; l = e) {
        e = run_end(l);
        const uint64_t r0 = soa->contig_start[chosen_tid[l]], r1 = soa->contig_start[chosen_tid[e - 1] + 1];
        const size_t nr = r1 - r0;
        if (nr == 0) continue;
        const uint32_t w0 = soa->p_recs[r0].row_off, w1 = row_end(r1 - 1);
        CUDA_TRY(cudaMemcpyAsync(c->p_recs.as<mmlst_prec>() + rbase, soa->p_recs + r0, nr * sizeof(mmlst_prec), cudaMemcpyHostToDevice, c->lane[k]));
        k = (k + 1) % mmlst_ctx::kLanes;
        CUDA_TRY(cudaMemcpyAsync(c->planes.as<uint32_t>() + wbase, soa->planes + w0, (size_t)(w1 - w0) * 4, cudaMemcpyHostToDevice, c->lane[k]));
        k = (k + 1) % mmlst_ctx::kLanes;
        for (uint32_t m = l; m < e; ++m) {
            const uint64_t q0 = soa->contig_start[chosen_tid[m]], q1 = soa->contig_start[chosen_tid[m] + 1];
            for (uint64_t b = q0; b < q1; b += kChunkRecords) {
                mmlst_chunk ck{};
                ck.rec_begin = (uint32_t)(rbase + (b - r0));
                ck.rec_end = (uint32_t)(rbase + (std::min<uint64_t>(q1, b + kChunkRecords) - r0));
                ck.col_base = col_off[m];
                ck.contig_len = col_off[m + 1] - col_off[m];
                ck.plane_delta = (uint32_t)wbase - w0;
                chunks.push_back(ck);
            }
        }
        rbase += nr;
        wbase += (size_t)(w1 - w0);
        wbase = (wbase + 3) & ~(size_t)3;
    }
    for (int i = 0; i < mmlst_ctx::kLanes; ++i) {
        CUDA_TRY(cudaEventRecord(c->lane_ev[i], c->lane[i]));
        CUDA_TRY(cudaStreamWaitEvent(s, c->lane_ev[i], 0));
    }
    TRY(h2d(c->chunks, chunks.data(), chunks.size(), s));
    return MMLST_OK;
}

extern "C" int mmlst_pileup_consensus(mmlst_ctx* c, const mmlst_soa* soa, const uint32_t* chosen_tid, uint32_t n_loci,
                                      const uint8_t* dbseq, const uint32_t* col_off, int minscore, int max_xm,
                                      uint32_t mincov, int impl, uint32_t* counts, uint8_t* cons, uint32_t* holes,
                                      uint32_t* snps) {
    CTX_ENTER(c);
    if (!soa || !chosen_tid || !dbseq || !col_off || !cons || !holes || !snps) { mmlst_set_error("mmlst_pileup_consensus: null pointer"); return MMLST_E_ARG; }
    if (n_loci == 0) return MMLST_OK;
    cudaStream_t s = c->stream;
    mmlst_trace_mark("enter");
    const uint32_t total_cols = col_off[n_loci];
    std::vector<mmlst_chunk> chunks;
    TRY(upload_chosen_contigs(c, soa, chosen_tid, n_loci, col_off, chunks));
    mmlst_trace_mark("stream_h2d_enqueued");
    TRY(h2d(c->dbseq, dbseq, total_cols, s));
    TRY(h2d(c->col_off, col_off, (size_t)n_loci + 1, s));
    TRY(c->counts.reserve((size_t)total_cols * 20 + 16)); TRY(c->cons.reserve(total_cols + 16));
    TRY(c->holes.reserve(n_loci * 4)); TRY(c->snps.reserve(n_loci * 4));
    CUDA_TRY(cudaMemsetAsync(c->counts.p, 0, (size_t)total_cols * 20, s));
    TRY(mmlst_pileup_dev(c->p_recs.as<mmlst_prec>(), c->planes.as<uint32_t>(), c->chunks.as<mmlst_chunk>(), (uint32_t)chunks.size(),
                         soa->max_row_words, minscore, max_xm, c->counts.as<uint32_t>(), total_cols, impl, s));
    TRY(mmlst_consensus_dev(c->counts.as<uint32_t>(), c->dbseq.as<uint8_t>(), c->col_off.as<uint32_t>(), n_loci, mincov,
                            c->cons.as<uint8_t>(), c->holes.as<uint32_t>(), c->snps.as<uint32_t>(), s));
    if (counts) CUDA_TRY(cudaMemcpyAsync(counts, c->counts.p, (size_t)total_cols * 20, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(cons, c->cons.p, total_cols, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(holes, c->holes.p, n_loci * 4, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(snps, c->snps.p, n_loci * 4, cudaMemcpyDeviceToHost, s));
    mmlst_trace_mark("kernels_d2h_enqueued");
    CUDA_TRY(cudaStreamSynchronize(s));
    mmlst_trace_mark("sync");
    mmlst_trace_flush("mmlst_pileup_consensus");
    return MMLST_OK;
}

extern "C" int mmlst_contig_stats(mmlst_ctx* c, const mmlst_soa* soa, const uint32_t* tid, uint32_t n, const uint32_t* col_off, int minscore,
                                  int max_xm, const mmlst_contig_stats_params* prm, mmlst_contig_stats_out* out) {
    if (!soa || !tid || !col_off || !prm || !out || !out->sel_off || !out->low_off || !out->depth_off) { mmlst_set_error("mmlst_contig_stats: null pointer"); return MMLST_E_ARG; }
    if (col_off[0] != 0) { mmlst_set_error("mmlst_contig_stats: col_off[0] = %u, not 0", col_off[0]); return MMLST_E_ARG; }
    for (uint32_t i = 0; i < n; ++i) {
        if (col_off[i + 1] < col_off[i]) { mmlst_set_error("mmlst_contig_stats: col_off not ascending at %u", i); return MMLST_E_ARG; }
        if (i && tid[i] <= tid[i - 1]) { mmlst_set_error("mmlst_contig_stats: tid not ascending at %u", i); return MMLST_E_ARG; }
    }
    const uint32_t total_cols = col_off[n];
    if (total_cols > MMLST_CONTIG_STATS_MAX_COLS) {
        mmlst_set_error("mmlst_contig_stats: %u columns in one batch, at most %u (5 * column in 32 bits)", total_cols, (uint32_t)MMLST_CONTIG_STATS_MAX_COLS);
        return MMLST_E_RANGE;
    }
    if (prm->mode > MMLST_STATS_LOWDOM || prm->mincov == 0 || prm->none_char > 255) { mmlst_set_error("mmlst_contig_stats: mode %u / mincov %u / none_char %u out of range", prm->mode, prm->mincov, prm->none_char); return MMLST_E_ARG; }
    const uint32_t width = prm->mode == MMLST_STATS_COLUMNS ? 5u : prm->mode == MMLST_STATS_DEPTH ? 1u : 2u;
    if (out->capacity && (!out->out_col || !out->out_val)) { mmlst_set_error("mmlst_contig_stats: null pointer"); return MMLST_E_ARG; }
    out->n_out = 0;
    if (n == 0) { out->sel_off[0] = 0; out->low_off[0] = 0; out->depth_off[0] = 0; return MMLST_OK; }
    CTX_ENTER(c);
    cudaStream_t s = c->stream;
    mmlst_trace_mark("enter");
    std::vector<mmlst_chunk> chunks;
    TRY(upload_chosen_contigs(c, soa, tid, n, col_off, chunks, false, true));
    TRY(h2d(c->col_off, col_off, (size_t)n + 1, s));
    const size_t scratch = mmlst_contig_stats_scratch_bytes(total_cols);
    TRY(c->counts.reserve((size_t)total_cols * 20 + 16)); TRY(c->cs_scratch.reserve(scratch));
    TRY(c->cs_off.reserve(((size_t)n + 1) * 16 + 16)); TRY(c->cs_out.reserve((size_t)total_cols * 4 * (1 + width) + 16));
    if (out->cons) TRY(c->cons.reserve((size_t)total_cols + 16));
    uint32_t* d_sel = c->cs_off.as<uint32_t>(); uint32_t* d_low = d_sel + n + 1;
    uint64_t* d_dep = reinterpret_cast<uint64_t*>(c->cs_off.as<uint8_t>() + (((size_t)n + 1) * 8 + 15) / 16 * 16);
    uint32_t* d_col = c->cs_out.as<uint32_t>(); uint32_t* d_val = d_col + total_cols;
    CUDA_TRY(cudaMemsetAsync(c->counts.p, 0, (size_t)total_cols * 20, s));
    TRY(mmlst_pileup_dev(c->p_recs.as<mmlst_prec>(), c->planes.as<uint32_t>(), c->chunks.as<mmlst_chunk>(), (uint32_t)chunks.size(),
                         soa->max_row_words, minscore, max_xm, c->counts.as<uint32_t>(), total_cols, 0, s));
    TRY(mmlst_contig_stats_dev(c->counts.as<uint32_t>(), c->col_off.as<uint32_t>(), n, total_cols, prm, c->cs_scratch.p, scratch, d_sel, d_low, d_dep,
                               d_col, d_val, out->cons ? c->cons.as<uint8_t>() : nullptr, 0, s));
    CUDA_TRY(cudaMemcpyAsync(out->sel_off, d_sel, ((size_t)n + 1) * 4, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(out->low_off, d_low, ((size_t)n + 1) * 4, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(out->depth_off, d_dep, ((size_t)n + 1) * 8, cudaMemcpyDeviceToHost, s));
    if (out->cons && total_cols) CUDA_TRY(cudaMemcpyAsync(out->cons, c->cons.p, total_cols, cudaMemcpyDeviceToHost, s));
    mmlst_trace_mark("summaries_enqueued");
    CUDA_TRY(cudaStreamSynchronize(s));
    const uint64_t n_out = prm->mode == MMLST_STATS_LOWDOM ? out->low_off[n] : out->sel_off[n];
    if (n_out > out->capacity) { mmlst_set_error("mmlst_contig_stats: %llu compacted columns, capacity %llu", (unsigned long long)n_out, (unsigned long long)out->capacity); return MMLST_E_ARG; }
    if (n_out) {
        CUDA_TRY(cudaMemcpyAsync(out->out_col, d_col, n_out * 4, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaMemcpyAsync(out->out_val, d_val, n_out * 4 * width, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaStreamSynchronize(s));
    }
    out->n_out = n_out;
    mmlst_trace_mark("sync");
    mmlst_trace_flush("mmlst_contig_stats");
    return MMLST_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// One call per sample over HOST buffers: score -> selection (on the device) -> pileup of the chosen contigs -> consensus.
extern "C" int mmlst_index_upload(mmlst_ctx* c, const mmlst_index* ix) {
    CTX_ENTER(c);
    if (!ix || !ix->locus_of || !ix->allele_num || !ix->species_of_locus || !ix->genes_in_db || !ix->db_ascii || !ix->db_off || !ix->bam_ln) {
        mmlst_set_error("mmlst_index_upload: null pointer");
        return MMLST_E_ARG;
    }
    const uint32_t nr = ix->n_ref, nl = ix->n_loci, ns = ix->n_species;
    if (nr == 0 || nl == 0 || ns == 0) { mmlst_set_error("mmlst_index_upload: empty index"); return MMLST_E_ARG; }
    if (nl > 8192 || ns > 4096) { mmlst_set_error("mmlst_index_upload: more than 8192 loci / 4096 species"); return MMLST_E_RANGE; }
    TRY(mmlst_select_fits(nl, ns, "mmlst_index_upload"));   // refused here, not by the first mmlst_sample
    // allele rows grouped by locus (counting sort, stable: ascending row inside a locus)
    std::vector<uint32_t> start(nl + 1, 0), rows(nr);
    for (uint32_t t = 0; t < nr; ++t) {
        if (ix->locus_of[t] >= nl) { mmlst_set_error("mmlst_index_upload: locus_of[%u]=%u out of range", t, ix->locus_of[t]); return MMLST_E_ARG; }
        ++start[ix->locus_of[t] + 1];
    }
    for (uint32_t l = 0; l < nl; ++l) {
        if (ix->species_of_locus[l] >= ns) { mmlst_set_error("mmlst_index_upload: species_of_locus[%u] out of range", l); return MMLST_E_ARG; }
        start[l + 1] += start[l];
    }
    { std::vector<uint32_t> fill(start.begin(), start.end() - 1); for (uint32_t t = 0; t < nr; ++t) rows[fill[ix->locus_of[t]]++] = t; }
    for (uint32_t t = 0; t < nr; ++t)
        if (ix->db_off[t + 1] < ix->db_off[t]) { mmlst_set_error("mmlst_index_upload: db_off not ascending at row %u", t); return MMLST_E_ARG; }
    cudaStream_t s = c->stream;
    TRY(h2d(c->ix_locus_of, ix->locus_of, nr, s));
    TRY(h2d(c->ix_locus_rows, rows.data(), nr, s));
    c->ix_rows_identity = true;
    for (uint32_t t = 0; t < nr; ++t) if (rows[t] != t) { c->ix_rows_identity = false; break; }
    TRY(h2d(c->ix_locus_start, start.data(), (size_t)nl + 1, s));
    TRY(h2d(c->ix_allele_num, ix->allele_num, nr, s));
    TRY(h2d(c->ix_species_of_locus, ix->species_of_locus, nl, s));
    TRY(h2d(c->ix_genes_in_db, ix->genes_in_db, ns, s));
    TRY(c->ix_db_ascii.reserve(ix->db_off[nr] + 16));
    if (ix->db_off[nr]) CUDA_TRY(cudaMemcpyAsync(c->ix_db_ascii.p, ix->db_ascii, ix->db_off[nr], cudaMemcpyHostToDevice, s));
    TRY(h2d(c->ix_db_off, ix->db_off, (size_t)nr + 1, s));
    TRY(h2d(c->ix_bam_ln, ix->bam_ln, nr, s));
    TRY(c->ix_zero64.reserve(((size_t)nr + 1) * 8));
    CUDA_TRY(cudaMemsetAsync(c->ix_zero64.p, 0, ((size_t)nr + 1) * 8, s));
    TRY(c->ix_scratch.reserve((size_t)nl * 12 + 64));
    CUDA_TRY(cudaMemsetAsync(c->ix_scratch.p, 0, (size_t)nl * 12 + 64, s));
    TRY(c->ix_out.reserve((16 + 5 * (size_t)nl + 8) * 4));
    TRY(c->ix_db_start.reserve(((size_t)nl + 1) * 8));
    TRY(c->ix_chunks.reserve(((size_t)nl + 1) * sizeof(mmlst_chunk)));
    CUDA_TRY(cudaStreamSynchronize(s));   // `rows` / `start` are locals
    c->ix_bam_ln_h.assign(ix->bam_ln, ix->bam_ln + nr);
    c->ix_db_off_h.assign(ix->db_off, ix->db_off + nr + 1);
    c->ix_n_ref = nr; c->ix_n_loci = nl; c->ix_n_species = ns;
    return MMLST_OK;
}

extern "C" int mmlst_sample(mmlst_ctx* c, const mmlst_soa* soa, const uint8_t* allow, const mmlst_sample_params* prm, mmlst_sample_result* res) {
    CTX_ENTER(c);
    if (!soa || !allow || !prm || !res || !res->chosen_tid || !res->chosen_species || !res->col_off || !res->cons || !res->holes || !res->snps) {
        mmlst_set_error("mmlst_sample: null pointer");
        return MMLST_E_ARG;
    }
    if (!c->ix_n_ref) { mmlst_set_error("mmlst_sample: no index in the context (mmlst_index_upload)"); return MMLST_E_ARG; }
    if (soa->n_ref != c->ix_n_ref) { mmlst_set_error("mmlst_sample: the stream has %u references, the index %u", soa->n_ref, c->ix_n_ref); return MMLST_E_ARG; }
    cudaStream_t s = c->stream;
    const size_t nr = soa->n_ref;
    const uint32_t nl = c->ix_n_loci;
    const bool want_tables = res->sum_as && res->n_hit && res->first_idx;
    mmlst_trace_mark("enter");
    // ---- stage 1: score stream up (DEFLATE blocks inflated by the hardware engine when the sample carries them), score, select
    TRY(upload_score_stream(c, soa));
    TRY(h2d(c->allow, allow, nr, s));
    const mmlst_score_params sp{prm->minscore, prm->max_xm, prm->min_read_len};
    TRY(launch_resident_score(c, soa, &sp, c->ix_locus_of.as<uint32_t>()));
    // output block: header[16] | chosen_tid[nl] | chosen_species[nl] | col_off[nl+1] | holes[nl] | snps[nl]
    uint32_t* out = c->ix_out.as<uint32_t>();
    uint32_t* d_hdr = out; uint32_t* d_tid = out + 16; uint32_t* d_sp = d_tid + nl; uint32_t* d_col = d_sp + nl; uint32_t* d_holes = d_col + nl + 1; uint32_t* d_snps = d_holes + nl;
    const size_t out_words = 16 + 5 * (size_t)nl + 1;
    const size_t tab_bytes = want_tables ? nr * 16 : 0;
    const size_t stage1_bytes = (out_words * 4 + tab_bytes + (size_t)c->z_pending * 4 + 63) & ~(size_t)63;
    TRY(c->pin_reserve(stage1_bytes + res->cons_capacity + 8 * (size_t)nl + (soa->zp ? (size_t)soa->zp->n_blocks * 4 : 0) + 256));   // one reservation: the staging block does not move inside the call
    uint32_t* h_out = static_cast<uint32_t*>(c->pin);
    uint8_t* h_tab = reinterpret_cast<uint8_t*>(h_out + out_words);
    if (want_tables) {   // the selection below does not consume them
        CUDA_TRY(cudaMemcpyAsync(h_tab, c->sum_as.p, nr * 8, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaMemcpyAsync(h_tab + nr * 8, c->n_hit.p, nr * 4, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaMemcpyAsync(h_tab + nr * 12, c->first_idx.p, nr * 4, cudaMemcpyDeviceToHost, s));
    }
    uint32_t* h_zact = reinterpret_cast<uint32_t*>(h_tab + tab_bytes);
    if (c->z_pending) CUDA_TRY(cudaMemcpyAsync(h_zact, c->zact.p, (size_t)c->z_pending * 4, cudaMemcpyDeviceToHost, s));
    TRY(mmlst_select_dev(c->sum_as.as<int64_t>(), c->n_hit.as<uint32_t>(), c->first_idx.as<uint32_t>(), c->ix_rows_identity ? nullptr : c->ix_locus_rows.as<uint32_t>(),
                         c->ix_locus_start.as<uint32_t>(), c->ix_allele_num.as<uint32_t>(), (uint32_t)nr, c->ix_species_of_locus.as<uint32_t>(),
                         c->ix_genes_in_db.as<uint32_t>(), nl, c->ix_n_species, prm->penalty, prm->nloci_pct, c->ix_zero64.as<uint64_t>(),
                         c->ix_bam_ln.as<uint32_t>(), c->ix_db_off.as<uint64_t>(), 512, c->ix_scratch.p, (size_t)nl * 12 + 64, d_hdr, d_tid, d_sp, d_col,
                         c->ix_db_start.as<uint64_t>(), c->ix_chunks.as<mmlst_chunk>(), nl, 0, c->counters.as<uint64_t>(), nullptr, s));
    CUDA_TRY(cudaMemcpyAsync(h_out, out, (16 + 3 * (size_t)nl + 1) * 4, cudaMemcpyDeviceToHost, s));
    mmlst_trace_mark("stage1_enqueued");
    CUDA_TRY(cudaStreamSynchronize(s));
    mmlst_trace_mark("stage1_sync");
    for (uint32_t b = 0; b < c->z_pending; ++b) {
        if (h_zact[b] != c->zlen[b]) {
            c->z_pending = 0;
            mmlst_set_error("mmlst_sample: block %u of the compressed score stream inflated to %u bytes, %u expected (corrupt mmlst_soa.z)", b, h_zact[b], c->zlen[b]);
            return MMLST_E_ARG;
        }
    }
    c->z_pending = 0;
    if (want_tables) { memcpy(res->sum_as, h_tab, nr * 8); memcpy(res->n_hit, h_tab + nr * 8, nr * 4); memcpy(res->first_idx, h_tab + nr * 12, nr * 4); }
    const uint32_t n = h_out[0];
    res->n_chosen = n; res->error_bits = h_out[3] & 1u;
    res->total_reads = (uint64_t)h_out[6] | ((uint64_t)h_out[7] << 32);
    res->ignored_reads = (uint64_t)h_out[8] | ((uint64_t)h_out[9] << 32);
    if (n > nl) { mmlst_set_error("mmlst_sample: selection returned %u loci of %u", n, nl); return MMLST_E_CUDA; }
    const uint32_t* h_tid = h_out + 16; const uint32_t* h_sp = h_tid + nl; const uint32_t* h_col = h_sp + nl;
    memcpy(res->chosen_tid, h_tid, (size_t)n * 4); memcpy(res->chosen_species, h_sp, (size_t)n * 4); memcpy(res->col_off, h_col, ((size_t)n + 1) * 4);
    if (n == 0 || res->error_bits) { mmlst_trace_flush("mmlst_sample"); return MMLST_OK; }
    const uint32_t total_cols = h_col[n];
    if (total_cols > res->cons_capacity) { mmlst_set_error("mmlst_sample: %u consensus bytes, capacity %llu", total_cols, (unsigned long long)res->cons_capacity); return MMLST_E_ARG; }
    for (uint32_t l = 0; l < n; ++l) {   // H10: metaMLST_functions.py:267/269 index dbSequen[i] for i < BAM LN
        const uint32_t t = h_tid[l];
        if (c->ix_bam_ln_h[t] > c->ix_db_off_h[t + 1] - c->ix_db_off_h[t]) {
            mmlst_set_error("string index out of range: BAM LN %u > DB sequence length %llu for reference %u", c->ix_bam_ln_h[t],
                            (unsigned long long)(c->ix_db_off_h[t + 1] - c->ix_db_off_h[t]), t);
            res->bad_len_tid = t;
            return MMLST_E_RANGE;
        }
    }
    // ---- stage 2: only the chosen contigs' records and plane rows cross the bus (contiguous ranges of the coordinate-sorted stream)
    std::vector<mmlst_chunk> chunks;
    TRY(upload_chosen_contigs(c, soa, h_tid, n, h_col, chunks, true));
    TRY(c->counts.reserve((size_t)total_cols * 20 + 16)); TRY(c->cons.reserve(total_cols + 16));
    CUDA_TRY(cudaMemsetAsync(c->counts.p, 0, (size_t)total_cols * 20, s));
    TRY(mmlst_pileup_dev(c->p_recs.as<mmlst_prec>(), c->planes.as<uint32_t>(), c->chunks.as<mmlst_chunk>(), (uint32_t)chunks.size(),
                         soa->max_row_words, prm->minscore, prm->max_xm, c->counts.as<uint32_t>(), total_cols, prm->pileup_impl, s));
    TRY(mmlst_consensus_indirect_dev(c->counts.as<uint32_t>(), c->ix_db_ascii.as<uint8_t>(), c->ix_db_start.as<uint64_t>(), d_col, n, d_hdr, prm->mincov,
                                     c->cons.as<uint8_t>(), d_holes, d_snps, 0, s));
    const size_t hs_off = stage1_bytes + (((size_t)total_cols + 15) & ~(size_t)15);
    uint8_t* h_cons = static_cast<uint8_t*>(c->pin) + stage1_bytes;
    uint32_t* h_hs = reinterpret_cast<uint32_t*>(static_cast<uint8_t*>(c->pin) + hs_off);
    uint32_t* h_zpact = h_hs + 2 * (size_t)nl;
    CUDA_TRY(cudaMemcpyAsync(h_cons, c->cons.p, total_cols, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(h_hs, d_holes, 2 * (size_t)nl * 4, cudaMemcpyDeviceToHost, s));
    if (c->zp_pending) CUDA_TRY(cudaMemcpyAsync(h_zpact, c->zpact.p, (size_t)c->zp_pending * 4, cudaMemcpyDeviceToHost, s));
    mmlst_trace_mark("stage2_enqueued");
    CUDA_TRY(cudaStreamSynchronize(s));
    mmlst_trace_mark("stage2_sync");
    for (uint32_t b = 0; b < c->zp_pending; ++b) {
        if (h_zpact[b] != c->zplen[b]) {
            c->zp_pending = 0;
            mmlst_set_error("mmlst_sample: block %u of the compressed pileup stream inflated to %u bytes, %u expected (corrupt mmlst_soa.zp)", b, h_zpact[b], c->zplen[b]);
            return MMLST_E_ARG;
        }
    }
    c->zp_pending = 0;
    memcpy(res->cons, h_cons, total_cols);
    memcpy(res->holes, h_hs, (size_t)n * 4);
    memcpy(res->snps, h_hs + nl, (size_t)n * 4);
    mmlst_trace_flush("mmlst_sample");
    return MMLST_OK;
}

// ---------------------------------------------------------------------------------------------------------------
extern "C" int mmlst_hamming_min_dev2(const uint32_t*, const uint32_t*, const uint16_t*, uint32_t, uint32_t, const uint32_t*,
                                      const uint32_t*, const uint16_t*, uint32_t, const uint32_t*, uint32_t, uint32_t, uint32_t,
                                      uint32_t, unsigned long long*, void*);

extern "C" int mmlst_hamming_exact_dev(const uint32_t*, const uint32_t*, const uint16_t*, uint32_t, uint32_t, const uint32_t*, const uint32_t*,
                                       const uint16_t*, uint32_t, const uint32_t*, uint32_t, uint32_t, const uint32_t*, const uint32_t*,
                                       const uint8_t*, uint32_t, const uint32_t*, const uint32_t*, const uint8_t*, uint32_t,
                                       unsigned long long*, void*);

extern "C" int mmlst_db_upload_x(mmlst_ctx* c, const uint32_t* db_hi, const uint32_t* db_lo, const uint16_t* row_len,
                                 uint32_t n_rows, uint32_t W, const uint32_t* xr_ids, const uint32_t* xr_x,
                                 const uint8_t* xr_bytes, uint32_t n_xr) {
    CTX_ENTER(c);
    if (!db_hi || !db_lo || !row_len || (n_xr && (!xr_ids || !xr_x || !xr_bytes))) { mmlst_set_error("mmlst_db_upload: null pointer"); return MMLST_E_ARG; }
    for (uint32_t i = 0; i < n_xr; ++i) {
        if (xr_ids[i] >= n_rows || (i && xr_ids[i] <= xr_ids[i - 1]) || !(row_len[xr_ids[i]] & 0x8000u)) {
            mmlst_set_error("mmlst_db_upload: flagged-row list must be ascending, in range, and every listed row flagged (bit 15 of row_len)");
            return MMLST_E_ARG;
        }
    }
    const size_t words = (size_t)((n_rows + 31) / 32) * 32 * W;
    TRY(h2d(c->db_hi, db_hi, words, c->stream));
    TRY(h2d(c->db_lo, db_lo, words, c->stream));
    TRY(h2d(c->db_len, row_len, n_rows, c->stream));
    TRY(h2d(c->xr_ids, xr_ids, n_xr, c->stream));
    TRY(h2d(c->xr_x, xr_x, (size_t)n_xr * W, c->stream));
    TRY(h2d(c->xr_bytes, xr_bytes, (size_t)n_xr * W * 32, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    c->db_rows = n_rows; c->db_W = W; c->db_n_xr = n_xr; c->has_row_key = false;
    return MMLST_OK;
}

extern "C" int mmlst_db_upload(mmlst_ctx* c, const uint32_t* db_hi, const uint32_t* db_lo, const uint16_t* row_len,
                               uint32_t n_rows, uint32_t W) {
    return mmlst_db_upload_x(c, db_hi, db_lo, row_len, n_rows, W, nullptr, nullptr, nullptr, 0);
}

extern "C" int mmlst_hamming_min_x(mmlst_ctx* c, const uint32_t* q_hi, const uint32_t* q_lo, const uint16_t* q_len, uint32_t n_q,
                                   const uint32_t* xq_ids, const uint32_t* xq_x, const uint8_t* xq_bytes, uint32_t n_xq,
                                   const uint32_t* blocks, uint32_t n_blocks, uint32_t* min_dist, uint32_t* argmin_row) {
    CTX_ENTER(c);
    if (!c->db_rows) { mmlst_set_error("mmlst_hamming_min: no DB uploaded"); return MMLST_E_ARG; }
    if (!q_hi || !q_lo || !q_len || !blocks || !min_dist || !argmin_row || (n_xq && (!xq_ids || !xq_x || !xq_bytes))) {
        mmlst_set_error("mmlst_hamming_min: null pointer");
        return MMLST_E_ARG;
    }
    if (n_q == 0) return MMLST_OK;
    for (uint32_t i = 0; i < n_xq; ++i) {
        if (xq_ids[i] >= n_q || (i && xq_ids[i] <= xq_ids[i - 1]) || !(q_len[xq_ids[i]] & 0x8000u)) {
            mmlst_set_error("mmlst_hamming_min: flagged-query list must be ascending, in range, and every listed query flagged (bit 15 of q_len)");
            return MMLST_E_ARG;
        }
    }
    cudaStream_t s = c->stream;
    const uint32_t W = c->db_W;
    TRY(h2d(c->q_hi, q_hi, (size_t)n_q * W, s));
    TRY(h2d(c->q_lo, q_lo, (size_t)n_q * W, s));
    TRY(h2d(c->q_len, q_len, n_q, s));
    TRY(h2d(c->blocks, blocks, (size_t)n_blocks * 4, s));
    TRY(h2d(c->xq_ids, xq_ids, n_xq, s));
    TRY(h2d(c->xq_x, xq_x, (size_t)n_xq * W, s));
    TRY(h2d(c->xq_bytes, xq_bytes, (size_t)n_xq * W * 32, s));
    TRY(c->best.reserve((size_t)n_q * 8));
    CUDA_TRY(cudaMemsetAsync(c->best.p, 0xff, (size_t)n_q * 8, s));
    uint32_t max_rows = 0, max_q = 0;
    for (uint32_t b = 0; b < n_blocks; ++b) {
        if (blocks[4 * b + 1] < blocks[4 * b] || blocks[4 * b + 3] < blocks[4 * b + 2] || blocks[4 * b + 1] > n_q || blocks[4 * b + 3] > c->db_rows) {
            mmlst_set_error("mmlst_hamming_min: block %u out of range", b);
            return MMLST_E_ARG;
        }
        max_q = std::max(max_q, blocks[4 * b + 1] - blocks[4 * b]);
        max_rows = std::max(max_rows, blocks[4 * b + 3] - blocks[4 * b + 2]);
    }
    for (uint32_t b0 = 0; b0 < n_blocks; b0 += 65535) {
        const uint32_t nb = std::min(65535u, n_blocks - b0);
        TRY(mmlst_hamming_min_dev2(c->db_hi.as<uint32_t>(), c->db_lo.as<uint32_t>(), c->db_len.as<uint16_t>(), c->db_rows, W,
                                   c->q_hi.as<uint32_t>(), c->q_lo.as<uint32_t>(), c->q_len.as<uint16_t>(), n_q,
                                   c->blocks.as<uint32_t>() + 4 * (size_t)b0, nb, max_rows, max_q, 0,
                                   c->best.as<unsigned long long>(), s));
        TRY(mmlst_hamming_exact_dev(c->db_hi.as<uint32_t>(), c->db_lo.as<uint32_t>(), c->db_len.as<uint16_t>(), c->db_rows, W,
                                    c->q_hi.as<uint32_t>(), c->q_lo.as<uint32_t>(), c->q_len.as<uint16_t>(), n_q,
                                    c->blocks.as<uint32_t>() + 4 * (size_t)b0, nb, 0,
                                    c->xr_ids.as<uint32_t>(), c->xr_x.as<uint32_t>(), c->xr_bytes.as<uint8_t>(), c->db_n_xr,
                                    c->xq_ids.as<uint32_t>(), c->xq_x.as<uint32_t>(), c->xq_bytes.as<uint8_t>(), n_xq,
                                    c->best.as<unsigned long long>(), s));
    }
    std::vector<unsigned long long> best(n_q);
    CUDA_TRY(cudaMemcpyAsync(best.data(), c->best.p, (size_t)n_q * 8, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    for (uint32_t q = 0; q < n_q; ++q) {
        min_dist[q] = (uint32_t)(best[q] >> 32);
        argmin_row[q] = (uint32_t)(best[q] & 0xffffffffu);
    }
    return MMLST_OK;
}

extern "C" int mmlst_hamming_min(mmlst_ctx* c, const uint32_t* q_hi, const uint32_t* q_lo, const uint16_t* q_len, uint32_t n_q,
                                 const uint32_t* blocks, uint32_t n_blocks, uint32_t* min_dist, uint32_t* argmin_row) {
    return mmlst_hamming_min_x(c, q_hi, q_lo, q_len, n_q, nullptr, nullptr, nullptr, 0, blocks, n_blocks, min_dist, argmin_row);
}

// ---------------------------------------------------------------------------------------------------------------
// Rows a10 / a11 (csrc/st_match.cu): exact-sequence lookup against the resident DB, ST assignment against the resident profiles.
extern "C" int mmlst_exact_match_dev(const uint32_t*, const uint32_t*, const uint16_t*, uint32_t, uint32_t, const uint32_t*, const uint32_t*,
                                     const uint16_t*, uint32_t, const uint32_t*, uint32_t, uint32_t, uint32_t, const uint32_t*, const uint32_t*,
                                     const uint8_t*, uint32_t, const uint32_t*, const uint8_t*, uint32_t, uint32_t*, void*);
extern "C" int mmlst_st_match_dev(const uint32_t*, const uint32_t*, uint32_t, const uint32_t*, const uint32_t*, uint32_t, uint32_t, uint32_t*,
                                  uint32_t*, uint32_t*, uint32_t*, uint32_t, void*);

extern "C" int mmlst_exact_match(mmlst_ctx* c, const uint32_t* q_hi, const uint32_t* q_lo, const uint16_t* q_len, uint32_t n_q,
                                 const uint32_t* xq_ids, const uint8_t* xq_bytes, uint32_t n_xq,
                                 const uint32_t* blocks, uint32_t n_blocks, uint32_t* first_row) {
    CTX_ENTER(c);
    if (!c->db_rows) { mmlst_set_error("mmlst_exact_match: no DB uploaded"); return MMLST_E_ARG; }
    if (n_q == 0) return MMLST_OK;
    if (!q_hi || !q_lo || !q_len || !blocks || !first_row || (n_xq && (!xq_ids || !xq_bytes))) { mmlst_set_error("mmlst_exact_match: null pointer"); return MMLST_E_ARG; }
    uint32_t max_rows = 0;
    for (uint32_t b = 0; b < n_blocks; ++b) {
        if (blocks[4 * b + 1] < blocks[4 * b] || blocks[4 * b + 3] < blocks[4 * b + 2] || blocks[4 * b + 1] > n_q || blocks[4 * b + 3] > c->db_rows) {
            mmlst_set_error("mmlst_exact_match: block %u out of range", b);
            return MMLST_E_ARG;
        }
        max_rows = std::max(max_rows, blocks[4 * b + 3] - blocks[4 * b + 2]);
    }
    cudaStream_t s = c->stream;
    const uint32_t W = c->db_W;
    TRY(h2d(c->q_hi, q_hi, (size_t)n_q * W, s));
    TRY(h2d(c->q_lo, q_lo, (size_t)n_q * W, s));
    TRY(h2d(c->q_len, q_len, n_q, s));
    TRY(h2d(c->blocks, blocks, (size_t)n_blocks * 4, s));
    TRY(h2d(c->xq_ids, xq_ids, n_xq, s));
    TRY(h2d(c->xq_bytes, xq_bytes, (size_t)n_xq * W * 32, s));
    TRY(c->first_row.reserve((size_t)n_q * 4));
    CUDA_TRY(cudaMemsetAsync(c->first_row.p, 0xff, (size_t)n_q * 4, s));
    for (uint32_t b0 = 0; b0 < n_blocks; b0 += 65535) {
        const uint32_t nb = std::min(65535u, n_blocks - b0);
        TRY(mmlst_exact_match_dev(c->db_hi.as<uint32_t>(), c->db_lo.as<uint32_t>(), c->db_len.as<uint16_t>(), c->db_rows, W,
                                  c->q_hi.as<uint32_t>(), c->q_lo.as<uint32_t>(), c->q_len.as<uint16_t>(), n_q,
                                  c->blocks.as<uint32_t>() + 4 * (size_t)b0, nb, max_rows, 0, c->has_row_key ? c->row_key.as<uint32_t>() : nullptr,
                                  c->xr_ids.as<uint32_t>(), c->xr_bytes.as<uint8_t>(), c->db_n_xr,
                                  c->xq_ids.as<uint32_t>(), c->xq_bytes.as<uint8_t>(), n_xq, c->first_row.as<uint32_t>(), s));
    }
    CUDA_TRY(cudaMemcpyAsync(first_row, c->first_row.p, (size_t)n_q * 4, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return MMLST_OK;
}

extern "C" int mmlst_db_row_keys(mmlst_ctx* c, const uint32_t* row_key, uint32_t n_rows) {
    CTX_ENTER(c);
    if (!row_key) { c->has_row_key = false; return MMLST_OK; }
    if (n_rows != c->db_rows) { mmlst_set_error("mmlst_db_row_keys: %u keys for %u resident rows", n_rows, c->db_rows); return MMLST_E_ARG; }
    TRY(h2d(c->row_key, row_key, n_rows, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    c->has_row_key = true;
    return MMLST_OK;
}

extern "C" int mmlst_profiles_upload(mmlst_ctx* c, const uint32_t* prof_start, const uint32_t* prof_allele, uint32_t n_st) {
    CTX_ENTER(c);
    if (!prof_start || (n_st && prof_start[n_st] && !prof_allele)) { mmlst_set_error("mmlst_profiles_upload: null pointer"); return MMLST_E_ARG; }
    for (uint32_t p = 0; p < n_st; ++p)
        if (prof_start[p + 1] < prof_start[p]) { mmlst_set_error("mmlst_profiles_upload: prof_start must be non-decreasing"); return MMLST_E_ARG; }
    TRY(h2d(c->prof_start, prof_start, (size_t)n_st + 1, c->stream));
    TRY(h2d(c->prof_allele, prof_allele, (size_t)prof_start[n_st], c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    c->n_st = n_st;
    return MMLST_OK;
}

extern "C" int mmlst_st_match(mmlst_ctx* c, const uint32_t* q_alleles, const uint32_t* q_n, uint32_t l_max, uint32_t n_q,
                              uint32_t* best, uint32_t* n_best, uint32_t* out_idx, uint32_t max_out) {
    CTX_ENTER(c);
    if (n_q == 0) return MMLST_OK;
    if (!q_alleles || !q_n || !best || !n_best || !out_idx || max_out == 0) { mmlst_set_error("mmlst_st_match: null pointer"); return MMLST_E_ARG; }
    if (!c->prof_start.p) { mmlst_set_error("mmlst_st_match: no profile table uploaded (mmlst_profiles_upload)"); return MMLST_E_ARG; }
    cudaStream_t s = c->stream;
    for (uint32_t q0 = 0; q0 < n_q; q0 += 32768) {
        const uint32_t nq = std::min(32768u, n_q - q0);
        TRY(h2d(c->st_q, q_alleles + (size_t)q0 * l_max, (size_t)nq * l_max, s));
        TRY(h2d(c->st_qn, q_n + q0, nq, s));
        TRY(c->st_count.reserve((size_t)nq * std::max(c->n_st, 1u) * 4));
        TRY(c->st_best.reserve((size_t)nq * 4));
        TRY(c->st_nbest.reserve((size_t)nq * 4));
        TRY(c->st_out.reserve((size_t)nq * max_out * 4));
        TRY(mmlst_st_match_dev(c->prof_start.as<uint32_t>(), c->prof_allele.as<uint32_t>(), c->n_st, c->st_q.as<uint32_t>(), c->st_qn.as<uint32_t>(),
                               l_max, nq, c->st_count.as<uint32_t>(), c->st_best.as<uint32_t>(), c->st_nbest.as<uint32_t>(), c->st_out.as<uint32_t>(),
                               max_out, s));
        CUDA_TRY(cudaMemcpyAsync(best + q0, c->st_best.p, (size_t)nq * 4, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaMemcpyAsync(n_best + q0, c->st_nbest.p, (size_t)nq * 4, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaMemcpyAsync(out_idx + (size_t)q0 * max_out, c->st_out.p, (size_t)nq * max_out * 4, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaStreamSynchronize(s));
    }
    return MMLST_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Host-side (sequential) htslib depth-cap admission, H1.  See include/mmlst.h.
extern "C" int mmlst_depth_cap(const uint32_t* tid, const int32_t* pos, const uint32_t* reflen, uint64_t n, uint32_t maxcnt,
                               uint32_t sentinel_nodes, uint8_t* admitted) {
    if (n == 0) return MMLST_OK;
    if (!tid || !pos || !reflen || !admitted) { mmlst_set_error("mmlst_depth_cap: null pointer"); return MMLST_E_ARG; }
    std::vector<uint32_t> endhist;
    uint64_t i = 0;
    while (i < n) {
        uint64_t j = i;
        int64_t maxend = 0;
        while (j < n && tid[j] == tid[i]) {
            if (j > i && pos[j] < pos[j - 1]) { mmlst_set_error("mmlst_depth_cap: records not coordinate-sorted at %llu", (unsigned long long)j); return MMLST_E_UNSORTED; }
            maxend = std::max<int64_t>(maxend, (int64_t)pos[j] + reflen[j]);
            ++j;
        }
        if (j < n && tid[j] < tid[i]) { mmlst_set_error("mmlst_depth_cap: contigs out of order at %llu", (unsigned long long)j); return MMLST_E_UNSORTED; }
        if ((j - i) + sentinel_nodes <= (uint64_t)maxcnt) {  // the mempool can never exceed the cap
            memset(admitted + i, 1, j - i);
            i = j;
            continue;
        }
        endhist.assign((size_t)maxend + 2, 0);
        uint64_t live = 0;
        int64_t cursor = 0;  // ends < cursor already removed
        uint64_t k = i;
        while (k < j) {
            const int32_t B = pos[k];
            for (; cursor <= (int64_t)B - 1; ++cursor) live -= endhist[(size_t)cursor];  // freed while emitting columns < B
            bool first = true;
            for (; k < j && pos[k] == B; ++k) {
                if (!first && (uint64_t)sentinel_nodes + live > (uint64_t)maxcnt) { admitted[k] = 0; continue; }
                admitted[k] = 1;
                const int64_t end = (int64_t)B + reflen[k];
                if (first || end > B) { ++live; ++endhist[(size_t)end]; }  // linked into the buffer (mp_alloc)
                first = false;
            }
        }
        i = j;
    }
    return MMLST_OK;
}
