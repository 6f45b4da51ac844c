// BAM ingest ON THE DEVICE (SURVEY.md 8f rank 1): compressed BGZF bytes cross PCIe (2.4x fewer than the inflated records),
// everything else happens in HBM and the sample never comes back to the host -- the output IS the packed record streams of
// include/mmlst.h, resident, ready for the score / pileup kernels.  Replaces `samtools view -h -` (metamlst.py:96-110), pysam's
// record access (cmseq/cmseq.py:54,527-545) and `samtools sort` / `index` (metaMLST_functions.py:237-247) like the host unpacker
// (csrc/bam_unpack.cpp, same per-record text: csrc/ingest_core.cuh), at device bandwidth instead of 10^6 records/s.
//
//   host   scan the BGZF block headers (18 + 8 bytes per <= 64 KB block): payload offset / size, ISIZE           sequential, tiny
//   H2D    the file's bytes, one copy
//   DE     raw DEFLATE of every block by Blackwell's hardware decompression engine: cuMemBatchDecompressAsync,
//          CU_MEM_DECOMPRESS_ALGORITHM_DEFLATE (measured 132 GB/s of output on B200, byte-identical to zlib:
//          profiles/r2a_de_probe.json) -- BGZF blocks are independent raw-deflate streams, exactly its batch shape
//   CRC    opts.check_crc: CRC-32 of every inflated block against its trailer, a CTA per block at a time (bgzf_crc.cuh)
//   K1     record chain: a BAM record only says where the NEXT one starts.  One thread per BGZF block guesses the first record
//          boundary at or after its block start (htslib never splits a record across blocks, so the guess is offset 0 there;
//          otherwise the first offset passing a strict plausibility test) and walks the chain to the block end; the guesses are
//          then VERIFIED -- the chain of block k must land exactly on the guess of block k+1 -- and re-walked from the
//          predecessor's exit where they do not, until nothing changes.  By induction from the first record (known from the
//          header) every accepted boundary is a true one.
//   K2     per record (thread): core fields, aux by POSITION and by NAME, reference span, QNAME hash, refusals (ingest_core.cuh)
//   sort   `samtools sort` order (stable by tid, pos, strand) by LSD radix sort of (key, file index) unless already so (CUB)
//   K3     score stream in sorted order + run-length arrays + len(SEQ) per 256-record chunk
//   K4     htslib depth cap (H1): one warp per contig that can exceed the cap, groups of equal start position in order, the
//          closed form of csrc/api.cu mmlst_depth_cap (first min(n_B, max(1, maxcnt - live(B) - sentinel + 1)) records per start)
//   K5     compaction of the admitted records, row offsets, plane rows (thread per record: CIGAR walk over 4-bit bases + qualities)
#include <cuda.h>
#include <cub/cub.cuh>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "bgzf_crc.cuh"
#include "common.cuh"
#include "de.h"
#include "ingest_core.cuh"

namespace {

using namespace ingest;

thread_local cudaStream_t g_cur_stream = nullptr;   // stream of the mmlst_bam_ingest call running on this thread (DBuf picks it up)

constexpr uint64_t kNoErr = ~0ull;
constexpr int kT = 256;

// Device workspace cache: an ingest makes ~60 allocations of up to several GB; cudaMalloc / cudaFree cost a fraction of a millisecond to
// milliseconds each and cudaFree synchronises the device, which was a third of the wall time of a call.  Blocks are cudaMalloc'ed once
// (plain cudaMalloc: memory the decompression engine accepts), handed out best-fit, and taken back with an event recorded on the stream
// that used them; a block is reused by ANOTHER stream only after that event.  mmlst_ingest_trim() gives the idle blocks back.
struct WsBlock { void* p; size_t bytes; bool used; cudaStream_t last; cudaEvent_t ev; bool has_ev; };
struct Workspace { std::mutex m; std::vector<WsBlock> blocks; };
Workspace g_ws[MMLST_MAX_DEVICES];

int ws_get(int dev, size_t need, cudaStream_t st, void** out, size_t* got) {
    Workspace& w = g_ws[dev % MMLST_MAX_DEVICES];
    need = (need + 511) & ~size_t(511);
    {
        std::lock_guard<std::mutex> g(w.m);
        int best = -1;
        for (size_t i = 0; i < w.blocks.size(); ++i) {
            const WsBlock& b = w.blocks[i];
            if (b.used || b.bytes < need || b.bytes > 2 * need + (1u << 20)) continue;
            if (best < 0 || b.bytes < w.blocks[best].bytes) best = static_cast<int>(i);
        }
        if (best >= 0) {
            WsBlock& b = w.blocks[best];
            b.used = true;
            if (b.has_ev && b.last != st) cudaEventSynchronize(b.ev);
            *out = b.p; *got = b.bytes;
            return MMLST_OK;
        }
    }
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, need);
    if (e != cudaSuccess) {  // give the idle blocks back and try once more
        cudaGetLastError();
        {
            std::lock_guard<std::mutex> g(w.m);
            for (size_t i = 0; i < w.blocks.size();) {
                if (!w.blocks[i].used) { if (w.blocks[i].has_ev) cudaEventDestroy(w.blocks[i].ev); cudaFree(w.blocks[i].p); w.blocks.erase(w.blocks.begin() + i); } else ++i;
            }
        }
        e = cudaMalloc(&p, need);
    }
    if (e != cudaSuccess) { cudaGetLastError(); mmlst_set_error("mmlst_bam_ingest: cudaMalloc(%zu) failed: %s", need, cudaGetErrorString(e)); return MMLST_E_NOMEM; }
    std::lock_guard<std::mutex> g(w.m);
    w.blocks.push_back(WsBlock{p, need, true, st, nullptr, false});
    *out = p; *got = need;
    return MMLST_OK;
}

void ws_put(int dev, void* p, cudaStream_t st, bool record) {
    Workspace& w = g_ws[dev % MMLST_MAX_DEVICES];
    std::lock_guard<std::mutex> g(w.m);
    for (WsBlock& b : w.blocks) {
        if (b.p != p) continue;
        if (record) {
            if (!b.has_ev) b.has_ev = cudaEventCreateWithFlags(&b.ev, cudaEventDisableTiming) == cudaSuccess;
            if (b.has_ev) cudaEventRecord(b.ev, st);
            b.last = st;
        } else if (b.has_ev) { cudaEventDestroy(b.ev); b.has_ev = false; }
        b.used = false;
        return;
    }
}

// page-locked staging buffer, one per device, grown on demand; held (mutex) for the duration of one header fetch
struct PinnedCache { std::mutex m; uint8_t* p = nullptr; size_t bytes = 0; };
PinnedCache g_pinned[MMLST_MAX_DEVICES];
struct PinnedStage {
    PinnedCache& c;
    std::unique_lock<std::mutex> lock;
    explicit PinnedStage(int dev) : c(g_pinned[dev % MMLST_MAX_DEVICES]), lock(c.m) {}
    uint8_t* get(size_t n) {
        if (n <= c.bytes) return c.p;
        if (c.p) cudaFreeHost(c.p);
        c.p = nullptr; c.bytes = 0;
        const size_t want = n + n / 2 + (1u << 16);
        if (cudaHostAlloc(reinterpret_cast<void**>(&c.p), want, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); c.p = nullptr; return nullptr; }
        c.bytes = want;
        return c.p;
    }
};

struct DBuf {
    void* p = nullptr;
    size_t bytes = 0;
    int dev = 0;
    cudaStream_t st = nullptr;
    int alloc(size_t n) {
        release();
        if (n == 0) n = 16;
        return ws_get(dev, n, st, &p, &bytes);
    }
    void release() { if (p) ws_put(dev, p, st, true); p = nullptr; bytes = 0; }
    template <class T> T* as() const { return static_cast<T*>(p); }
    DBuf() { cudaGetDevice(&dev); st = g_cur_stream; }
    ~DBuf() { release(); }
};

__device__ __forceinline__ void report(unsigned long long* err, uint64_t index, uint32_t code) {
    atomicMin(err, (static_cast<unsigned long long>(index) << 8) | code);
}

// ---- K1: record chain -------------------------------------------------------------------------------------------------------
// first_record == kNoEntry: no record boundary is known inside the buffer (a shard that starts past the header): every block guesses.
// uend: where the last block's records stop STARTING (usize, or the end of a shard's own blocks when a halo of the next shard's
// bytes follows them so that its last record can end there).  need (optional) [b]: after a walk that met a record running past usize,
// the buffer size that record needs (0 when the walk ended normally or the record is malformed).
constexpr uint64_t kNoEntry = ~0ull;
struct ChainArgs {
    const uint8_t* u; uint64_t usize; const uint64_t* uoff; uint32_t n_blocks; uint64_t first_record;
    int32_t n_ref; const uint32_t* ref_len;
    uint64_t* start; uint64_t* exit_; uint32_t* count; uint32_t* bad_walk;   // bad_walk[b] = 1: the walk from start[b] met a malformed record
    uint64_t uend; uint64_t* need;
};

__device__ __forceinline__ uint64_t block_end(const ChainArgs& a, uint32_t b) { return (b + 1 < a.n_blocks) ? a.uoff[b + 1] : a.uend; }

__device__ __forceinline__ void walk_block(const ChainArgs& a, uint32_t b, uint64_t s) {
    const uint64_t bend = block_end(a, b);
    uint64_t off = s, need = 0;
    uint32_t cnt = 0, bad = 0;
    while (off < bend) {
        const uint64_t nx = next_record(a.u, off, a.usize);
        if (nx == 0) {
            bad = 1;
            if (off + 4 > a.usize) need = off + 4;
            else { const int32_t bs = rdi32(a.u + off); need = bs >= 32 ? off + 4 + static_cast<uint64_t>(bs) : 0; }
            off = a.usize;
            break;
        }
        ++cnt;
        off = nx;
    }
    a.start[b] = s; a.exit_[b] = off; a.count[b] = cnt; a.bad_walk[b] = bad;
    if (a.need) a.need[b] = need;
}

__global__ void __launch_bounds__(kT) chain_guess_kernel(const ChainArgs a) {
    const uint32_t b = blockIdx.x * kT + threadIdx.x;
    if (b >= a.n_blocks) return;
    uint64_t s;
    if (a.first_record != kNoEntry && a.uoff[b] <= a.first_record) {
        const uint64_t bend = block_end(a, b);
        s = a.first_record < bend ? a.first_record : bend;   // header blocks hold no record start before first_record
        if (a.first_record >= bend) {
            a.start[b] = bend; a.exit_[b] = bend; a.count[b] = 0; a.bad_walk[b] = 0;
            if (a.need) a.need[b] = 0;
            return;
        }
    } else {
        s = a.uoff[b];
        const uint64_t lim = (s + (1ull << 20) < a.usize) ? s + (1ull << 20) : a.usize;
        while (s < lim && !plausible_record(a.u, s, a.usize, a.n_ref, a.ref_len)) ++s;
        if (s >= lim) s = a.usize;
    }
    walk_block(a, b, s);
}

// one verification / repair sweep: a block whose start is not its predecessor's exit is re-walked from there
__global__ void __launch_bounds__(kT) chain_repair_kernel(const ChainArgs a, uint32_t* changed) {
    const uint32_t b = blockIdx.x * kT + threadIdx.x;
    if (b == 0 || b >= a.n_blocks) return;
    if (a.first_record != kNoEntry && a.uoff[b] <= a.first_record) return;
    const uint64_t want = a.exit_[b - 1];
    if (a.start[b] == want) return;
    atomicAdd(changed, 1u);
    walk_block(a, b, want);
}

__global__ void __launch_bounds__(kT) chain_offsets_kernel(const ChainArgs a, const uint32_t* base, uint64_t* roff, unsigned long long* err) {
    const uint32_t b = blockIdx.x * kT + threadIdx.x;
    if (b >= a.n_blocks) return;
    const uint64_t bend = block_end(a, b);
    uint64_t off = a.start[b];
    uint64_t i = base[b];
    while (off < bend) {
        const uint64_t nx = next_record(a.u, off, a.usize);
        if (nx == 0) { report(err, i, E_TRUNC); return; }
        roff[i++] = off;
        off = nx;
    }
}

__global__ void __launch_bounds__(kT) check_isize_kernel(const uint32_t* act, const uint32_t* isize, uint32_t n_blocks, unsigned long long* err) {
    const uint32_t b = blockIdx.x * kT + threadIdx.x;
    if (b < n_blocks && act[b] != isize[b]) report(err, b, E_CHAIN);
}

// ---- BGZF CRC-32 (opts.check_crc) ------------------------------------------------------------------------------------------
// A CTA per block, looping over blocks so that the tables are built once per CTA: 8 KB of slice-by-8 tables and the byte tables of
// the kCrcLevels combine operators (32 KB) in shared memory.  Thread t takes segment t of the block's frame (bgzf_crc.cuh); the
// segments are combined by five shuffle levels inside a warp and three across the warps.
struct CrcArgs {
    const uint8_t* u; const uint64_t* uoff; const uint32_t* isize;
    const uint32_t* want;                             // [b] trailer CRC ^ crc32(0^isize): the block's raw CRC
    uint32_t n_blocks;
    uint32_t ops[bgzf_crc::kCrcLevels][32];           // bgzf_crc::make_ops
};

__global__ void __launch_bounds__(bgzf_crc::kCrcThreads, 4) crc_kernel(const CrcArgs a, unsigned long long* err) {
    namespace bc = bgzf_crc;
    constexpr uint32_t kWarps = bc::kCrcThreads / 32;
    static_assert(kWarps <= 32 && (1u << bc::kCrcLevels) == bc::kCrcThreads && bc::kCrcThreads == 256, "one table entry per thread");
    __shared__ uint32_t T[8][256];
    __shared__ uint32_t O[bc::kCrcLevels][4][256];
    __shared__ uint32_t warp_r[kWarps];
    const uint32_t t = threadIdx.x, lane = t & 31u, warp = t >> 5;
    T[0][t] = bc::t0_entry(t);
#pragma unroll 1
    for (uint32_t k = 0; k < bc::kCrcLevels; ++k)
#pragma unroll 1
        for (uint32_t j = 0; j < 4; ++j) O[k][j][t] = bc::op_entry(a.ops[k], j, t);
    __syncthreads();
    uint32_t c = T[0][t];
    for (int k = 1; k < 8; ++k) { c = bc::zero_byte(c, T[0]); T[k][t] = c; }
    __syncthreads();
    for (uint32_t b = blockIdx.x; b < a.n_blocks; b += gridDim.x) {
        const uint8_t* blk = a.u + a.uoff[b];
        const uint32_t n = a.isize[b];
        uint32_t r = bc::segment(blk, n, t, T);
#pragma unroll
        for (uint32_t k = 0; k < 5; ++k) r = bc::shift(r, O[k]) ^ __shfl_down_sync(0xffffffffu, r, 1u << k);
        if (lane == 0) warp_r[warp] = r;
        __syncthreads();
        if (warp == 0) {
            r = lane < kWarps ? warp_r[lane] : 0u;
#pragma unroll
            for (uint32_t k = 5; k < bc::kCrcLevels; ++k) r = bc::shift(r, O[k]) ^ __shfl_down_sync(0xffffffffu, r, 1u << (k - 5));
            if (lane == 0 && !bc::matches(r, a.want[b], blk, n, T[0])) report(err, b, E_CRC);
        }
        __syncthreads();   // warp_r is rewritten by the next block
    }
}

// ---- shard front half: routing + partition of the raw records by destination rank ------------------------------------------
// A shard's records go to the rank that owns their contig; a record whose refID is outside the dictionary goes to rank 0, where
// its refusal is raised exactly as on the whole file.  ord_key is the sort key without its strand bit: what --presorted compares.
constexpr int kMaxShardRanks = 256;

__device__ __forceinline__ uint64_t ord_key(int32_t tid, int32_t pos) {
    const uint64_t key = (static_cast<uint64_t>(static_cast<uint32_t>(tid)) << 33) | ((static_cast<uint64_t>(static_cast<uint32_t>(pos)) + 1ull) << 1);
    return key >> 1;
}

// dest[i], rlen[i] = 4 + block_size, dcount[d] += records for d; flags[0] = 1 when two neighbours are out of coordinate order;
// keys[0] / keys[1] = ord_key of the first / last record
__global__ void __launch_bounds__(kT) route_kernel(const uint8_t* u, const uint64_t* roff, uint64_t n, int32_t n_ref, const int32_t* owner, int world,
                                                   uint32_t* dest, uint32_t* rlen, unsigned long long* dcount, uint32_t* flags, uint64_t* keys) {
    __shared__ unsigned long long h[kMaxShardRanks];
    for (int d = threadIdx.x; d < world; d += kT) h[d] = 0;
    __syncthreads();
    const uint64_t i = static_cast<uint64_t>(blockIdx.x) * kT + threadIdx.x;
    if (i < n) {
        const uint8_t* r = u + roff[i];
        const int32_t tid = rdi32(r + 4), pos = rdi32(r + 8);
        const uint32_t d = (tid >= 0 && tid < n_ref) ? static_cast<uint32_t>(owner[tid]) : 0u;
        dest[i] = d;
        rlen[i] = 4u + rd32(r);
        atomicAdd(&h[d], 1ull);
        const uint64_t k = ord_key(tid, pos);
        if (i > 0) {
            const uint8_t* q = u + roff[i - 1];
            if (k < ord_key(rdi32(q + 4), rdi32(q + 8))) atomicOr(flags, 1u);
        }
        if (i == 0) keys[0] = k;
        if (i == n - 1) keys[1] = k;
    }
    __syncthreads();
    for (int d = threadIdx.x; d < world; d += kT) if (h[d]) atomicAdd(&dcount[d], h[d]);
}

__global__ void __launch_bounds__(kT) part_len_kernel(const uint32_t* order, const uint32_t* rlen, uint64_t n, uint64_t* plen) {
    const uint64_t j = static_cast<uint64_t>(blockIdx.x) * kT + threadIdx.x;
    if (j < n) plen[j] = rlen[order[j]];
    if (j == n) plen[j] = 0;
}

// one warp per record j of the partitioned order: its raw bytes to out + boff[j], its length and its index in the shard to the sidecars
__global__ void __launch_bounds__(kT) partition_kernel(const uint8_t* u, const uint64_t* roff, const uint32_t* order, const uint32_t* rlen,
                                                       const uint64_t* boff, uint64_t n, uint8_t* out, uint32_t* out_len, uint32_t* out_idx) {
    const uint64_t j = (static_cast<uint64_t>(blockIdx.x) * kT + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31u;
    if (j >= n) return;
    const uint32_t i = order[j], len = rlen[i];
    const uint8_t* src = u + roff[i];
    uint8_t* dst = out + boff[j];
    for (uint32_t b = lane; b < len; b += 32) dst[b] = src[b];
    if (lane == 0) { out_len[j] = len; out_idx[j] = i; }
}

__global__ void __launch_bounds__(kT) widen_kernel(const uint32_t* x, uint64_t n, uint64_t* y) {
    const uint64_t i = static_cast<uint64_t>(blockIdx.x) * kT + threadIdx.x;
    if (i < n) y[i] = x[i];
    if (i == n) y[i] = 0;
}

// ---- K2: per record ---------------------------------------------------------------------------------------------------------
struct ParseOut {
    uint64_t* key; uint16_t* reflen; int16_t* as0; int16_t* asn; uint16_t* qlen; uint8_t* xm3; uint8_t* xmn; uint8_t* bits; uint64_t* qh;
};

// gidx (shards): file index of record i, for the refusal text; nullptr = i
__global__ void __launch_bounds__(kT) parse_kernel(const uint8_t* u, const uint64_t* roff, const uint32_t* gidx, uint64_t n, int32_t n_ref, ParseOut o,
                                                   bool lenient, unsigned long long* err) {
    const uint64_t i = static_cast<uint64_t>(blockIdx.x) * kT + threadIdx.x;
    if (i >= n) return;
    Core c;
    uint64_t qh[2];
    const uint32_t e = parse_record(u, roff[i], n_ref, &c, o.qh ? qh : nullptr, lenient);
    if (e != E_NONE) { report(err, gidx ? gidx[i] : i, e); o.key[i] = ~0ull; return; }
    o.key[i] = c.key; o.reflen[i] = static_cast<uint16_t>(c.reflen); o.as0[i] = c.as0; o.asn[i] = c.asn; o.qlen[i] = c.qlen;
    o.xm3[i] = c.xm3; o.xmn[i] = c.xmn; o.bits[i] = c.bits;
    if (o.qh) { o.qh[2 * i] = qh[0]; o.qh[2 * i + 1] = qh[1]; }
}

// flags[0] |= 1: not in `samtools sort` order; flags[0] |= 2: not even coordinate order
__global__ void __launch_bounds__(kT) check_sorted_kernel(const uint64_t* key, uint64_t n, uint32_t* flags) {
    const uint64_t i = static_cast<uint64_t>(blockIdx.x) * kT + threadIdx.x + 1;
    if (i >= n) return;
    const uint64_t a = key[i - 1], b = key[i];
    uint32_t f = 0;
    if (b < a) f |= 1u;
    if ((b >> 1) < (a >> 1)) f |= 3u;
    if (f) atomicOr(flags, f);
}

__global__ void __launch_bounds__(kT) iota_kernel(uint32_t* x, uint64_t n) {
    const uint64_t i = static_cast<uint64_t>(blockIdx.x) * kT + threadIdx.x;
    if (i < n) x[i] = static_cast<uint32_t>(i);
}

// ---- K3: score stream in sorted order ---------------------------------------------------------------------------------------
struct GatherArgs {
    const uint64_t* key_sorted; const uint32_t* order;   // order == nullptr: identity
    ParseOut in; const uint64_t* roff; const uint32_t* gidx;   // gidx: file index of record i (shards); nullptr = i
    uint32_t* tid; int16_t* as0; uint8_t* xm3; uint16_t* qlen; uint32_t* orig_idx; uint64_t* qhash;
    int32_t* s_pos; uint16_t* s_reflen; uint8_t* s_bits; int16_t* s_asn; uint8_t* s_xmn; uint64_t* s_roff;
    uint32_t* run_flag; uint32_t* n_unmapped;
    uint64_t n;
};

__global__ void __launch_bounds__(kT) gather_kernel(const GatherArgs a) {
    const uint64_t k = static_cast<uint64_t>(blockIdx.x) * kT + threadIdx.x;
    if (k >= a.n) return;
    const uint64_t i = a.order ? a.order[k] : k;
    const uint64_t key = a.key_sorted[k];
    const uint32_t tid = static_cast<uint32_t>(key >> 33);
    a.tid[k] = tid; a.as0[k] = a.in.as0[i]; a.xm3[k] = a.in.xm3[i]; a.qlen[k] = a.in.qlen[i];
    if (a.orig_idx) a.orig_idx[k] = a.gidx ? a.gidx[i] : static_cast<uint32_t>(i);
    if (a.qhash) { a.qhash[2 * k] = a.in.qh[2 * i]; a.qhash[2 * k + 1] = a.in.qh[2 * i + 1]; }
    a.s_pos[k] = static_cast<int32_t>(((key >> 1) & 0xffffffffull) - 1ull);
    a.s_reflen[k] = a.in.reflen[i]; a.s_bits[k] = a.in.bits[i]; a.s_asn[k] = a.in.asn[i]; a.s_xmn[k] = a.in.xmn[i]; a.s_roff[k] = a.roff[i];
    const uint32_t prev = k ? static_cast<uint32_t>(a.key_sorted[k - 1] >> 33) : 0xffffffffu;
    a.run_flag[k] = (k == 0 || prev != tid) ? 1u : 0u;
    if (!(a.in.bits[i] & 1u)) atomicAdd(a.n_unmapped, 1u);
}

__global__ void __launch_bounds__(kT) runs_kernel(const uint32_t* run_flag, const uint32_t* run_incl, const uint32_t* tid, uint64_t n,
                                                  uint32_t* run_tid, uint32_t* run_start, uint32_t* chunk_run) {
    const uint64_t k = static_cast<uint64_t>(blockIdx.x) * kT + threadIdx.x;
    if (k >= n) return;
    const uint32_t r = run_incl[k] - 1u;
    if (run_flag[k]) { run_tid[r] = tid[k]; run_start[r] = static_cast<uint32_t>(k); }
    if ((k & 255u) == 0) chunk_run[k >> 8] = r;
    if (k == n - 1) run_start[r + 1] = static_cast<uint32_t>(n);
}

// one warp per 256-record chunk: chunk_qlen[c] = len(SEQ) of its first record; *uniform cleared when a chunk is mixed
__global__ void __launch_bounds__(kT) chunk_qlen_kernel(const uint16_t* qlen, uint64_t n, uint16_t* chunk_qlen, uint32_t* uniform) {
    const uint64_t c = (static_cast<uint64_t>(blockIdx.x) * kT + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31u;
    if (c * 256 >= n) return;
    const uint16_t q0 = qlen[c * 256];
    bool same = true;
    for (uint32_t j = lane; j < 256; j += 32) { const uint64_t k = c * 256 + j; if (k < n && qlen[k] != q0) same = false; }
    same = __all_sync(0xffffffffu, same);
    if (lane == 0) { chunk_qlen[c] = q0; if (!same) atomicAnd(uniform, 0u); }
}

// ---- K4: htslib depth cap ---------------------------------------------------------------------------------------------------
struct CapArgs {
    const uint32_t* run_tid; const uint32_t* run_start; uint32_t n_runs;
    const int32_t* s_pos; const uint16_t* s_reflen; const uint8_t* s_bits; const uint32_t* ref_len;
    uint32_t maxcnt, sentinel;
    const uint64_t* hist_off;    // [n_runs+1] offsets into hist (0-sized for runs that cannot exceed the cap)
    uint32_t* hist;              // zeroed scratch
    uint32_t* adm;               // [n] out: 1 admitted, 0 not
};

__global__ void __launch_bounds__(kT) cap_sizes_kernel(const CapArgs a, uint64_t* hist_size) {
    const uint32_t r = blockIdx.x * kT + threadIdx.x;
    if (r >= a.n_runs) return;
    const uint64_t len = a.run_start[r + 1] - a.run_start[r];
    hist_size[r] = (a.maxcnt && len + a.sentinel > a.maxcnt) ? static_cast<uint64_t>(a.ref_len[a.run_tid[r]]) + 3ull : 0ull;
}

__global__ void __launch_bounds__(kT) cap_kernel(const CapArgs a) {
    const uint32_t r = (blockIdx.x * kT + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31u;
    if (r >= a.n_runs) return;
    const uint64_t i0 = a.run_start[r], i1 = a.run_start[r + 1];
    const uint64_t hsz = a.hist_off[r + 1] - a.hist_off[r];
    if (hsz == 0) {  // the mempool can never exceed the cap: every candidate is admitted
        for (uint64_t k = i0 + lane; k < i1; k += 32) a.adm[k] = a.s_bits[k] & 1u;
        return;
    }
    uint32_t* hist = a.hist + a.hist_off[r];
    const uint32_t hmax = static_cast<uint32_t>(hsz - 1);   // ends beyond the contig are clamped here: never expired before the contig ends
    int64_t live = 0;
    uint32_t cursor = 0;
    uint64_t k = i0;
    while (k < i1) {
        const int32_t B = a.s_pos[k];
        // end of the group of equal start position (positions ascend inside a contig): upper bound by bisection, all lanes alike
        uint64_t lo = k + 1, hi = i1;
        while (lo < hi) { const uint64_t mid = (lo + hi) >> 1; if (a.s_pos[mid] <= B) lo = mid + 1; else hi = mid; }
        const uint64_t ge = lo;
        // expire the records whose end was passed while the iterator emitted the columns before B
        const uint32_t upto = static_cast<uint32_t>(B) < hmax ? static_cast<uint32_t>(B) : hmax;   // cursor runs to B - 1
        uint32_t freed = 0;
        for (uint32_t c = cursor + lane; c < upto; c += 32) freed += hist[c];
        freed = __reduce_add_sync(0xffffffffu, freed);
        if (upto > cursor) cursor = upto;
        live -= freed;
        uint32_t links = 0;
        bool seen = false, dropping = false;
        for (uint64_t c0 = k; c0 < ge && !dropping; c0 += 32) {
            const uint64_t m = c0 + lane;
            const bool in = m < ge;
            const bool cand = in && (a.s_bits[m] & 1u);
            const uint32_t rl = in ? a.s_reflen[m] : 0u;
            const uint32_t cmask = __ballot_sync(0xffffffffu, cand);
            const bool first = cand && !seen && (cmask & ((1u << lane) - 1u)) == 0u;
            const bool link = cand && (first || rl > 0);
            const uint32_t lmask = __ballot_sync(0xffffffffu, link);
            const uint32_t before = links + __popc(lmask & ((1u << lane) - 1u));
            const bool admit = cand && (first || static_cast<int64_t>(a.sentinel) + live + before <= static_cast<int64_t>(a.maxcnt));
            if (in) a.adm[m] = admit ? 1u : 0u;
            if (admit && link) {
                const uint64_t end = static_cast<uint64_t>(B) + rl;
                atomicAdd(&hist[end < hmax ? end : hmax], 1u);
            }
            const uint32_t amask = __ballot_sync(0xffffffffu, admit && link);
            links += __popc(amask);
            seen = seen || cmask != 0u;
            dropping = __any_sync(0xffffffffu, cand && !admit);
        }
        // (records of the group after the first refusal keep adm == 0: the array is zeroed before the launch)
        __syncwarp();
        live += links;
        k = ge;
    }
}

// ---- K5: compaction + plane rows --------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kT) scatter_adm_kernel(const uint32_t* adm, const uint32_t* adm_excl, uint64_t n, uint32_t* list) {
    const uint64_t k = static_cast<uint64_t>(blockIdx.x) * kT + threadIdx.x;
    if (k < n && adm[k]) list[adm_excl[k]] = static_cast<uint32_t>(k);
}

__global__ void __launch_bounds__(kT) row_sizes_kernel(const uint32_t* list, uint64_t P, const int32_t* s_pos, const uint16_t* s_reflen, uint64_t* rw, uint32_t* maxrw) {
    const uint64_t j = static_cast<uint64_t>(blockIdx.x) * kT + threadIdx.x;
    uint32_t w = 0;
    if (j < P) { const uint32_t k = list[j]; w = row_words(touched_words(static_cast<uint32_t>(s_pos[k]), s_reflen[k])); rw[j] = w; }
    w = __reduce_max_sync(0xffffffffu, w);
    if ((threadIdx.x & 31u) == 0 && w) atomicMax(maxrw, w);
}

__global__ void __launch_bounds__(kT) contig_start_kernel(const uint32_t* run_tid, const uint32_t* run_start, uint32_t n_runs, const uint32_t* adm_excl,
                                                          uint64_t P, uint32_t n_ref, uint64_t* contig_start) {
    const uint32_t t = blockIdx.x * kT + threadIdx.x;
    if (t > n_ref) return;
    uint32_t lo = 0, hi = n_runs;   // first run with run_tid >= t
    while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (run_tid[mid] < t) lo = mid + 1; else hi = mid; }
    contig_start[t] = lo < n_runs ? adm_excl[run_start[lo]] : P;
}

struct PackArgs {
    const uint8_t* u; const uint32_t* list; uint64_t P; const uint64_t* rowoff;
    const int32_t* s_pos; const uint16_t* s_reflen; const uint8_t* s_bits; const int16_t* s_asn; const uint8_t* s_xmn; const uint64_t* s_roff;
    const uint32_t* orig_idx; int minqual; mmlst_prec* recs; uint32_t* planes;
    int lenient; uint32_t* n_untagged;   // opts.lenient_tags: records without integer AS:i / XM:i are packed and counted here
};

// one WARP per admitted record: lane = contig column inside the 32-column word being built; every lane finds the query base aligned to
// its column by walking the (short) CIGAR, three ballots assemble the word's planes -- no atomics, no serial walk over the read
__global__ void __launch_bounds__(kT) pack_kernel(const PackArgs a, unsigned long long* err) {
    const uint64_t j = (static_cast<uint64_t>(blockIdx.x) * kT + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31u;
    if (j >= a.P) return;
    const uint32_t k = a.list[j];
    const uint32_t pos = static_cast<uint32_t>(a.s_pos[k]), rl = a.s_reflen[k];
    const uint32_t nw = touched_words(pos, rl), rw = row_words(nw);
    uint32_t* row = a.planes + a.rowoff[j];
    if (lane == 0) {
        mmlst_prec m;
        m.pos = static_cast<int32_t>(pos); m.row_off = static_cast<uint32_t>(a.rowoff[j]); m.reflen = static_cast<uint16_t>(rl);
        m.as_named = a.s_asn[k]; m.xm_named = a.s_xmn[k]; m.pad = 0; m.nw = static_cast<uint16_t>(nw);
        a.recs[j] = m;
    }
    if (rl == 0) return;
    const uint8_t* r = a.u + a.s_roff[k];
    const uint32_t l_name = r[12], n_cig = rd16(r + 16), l_seq = rd32(r + 20);
    const uint8_t* cig = r + 36 + l_name;
    const uint8_t* seq = cig + 4ull * n_cig;
    const uint8_t* qual = seq + (static_cast<uint64_t>(l_seq) + 1) / 2;
    uint32_t e = E_NONE;
    if (!(a.s_bits[k] & 2u) && !a.lenient) e = E_NAMED;
    else if (l_seq && qual[0] == 0xff) e = E_NOQUAL;
    else if (!(a.s_bits[k] & 2u) && lane == 0) atomicAdd(a.n_untagged, 1u);
    if (e != E_NONE) {
        for (uint32_t w = lane; w < rw; w += 32) row[w] = 0;
        if (lane == 0) report(err, a.orig_idx ? a.orig_idx[k] : k, e);
        return;
    }
    for (uint32_t w = 0; w < nw; ++w) {
        const uint32_t col = ((pos >> 5) + w) * 32u + lane;
        const uint32_t cls = column_class(cig, n_cig, seq, qual, l_seq, pos, rl, col, a.minqual);
        const uint32_t pv = __ballot_sync(0xffffffffu, cls >= 1u && cls <= 4u);
        const uint32_t p1 = __ballot_sync(0xffffffffu, cls == 3u || cls == 4u);
        const uint32_t p0 = __ballot_sync(0xffffffffu, cls == 2u || cls == 4u || cls == 5u);
        if (lane == 0) { row[3 * w] = pv; row[3 * w + 1] = p1; row[3 * w + 2] = p0; }
    }
    if (lane == 0 && rw > 3 * nw) row[3 * nw] = 0;
}

const char* err_text(uint32_t code) {
    switch (code) {
        case E_TRUNC: return "truncated / malformed record";
        case E_OVERRUN: return "record overruns its block_size";
        case E_NOREF: return "record has no reference (RNAME '*'): the reference crashes at metamlst.py:107";
        case E_PAIRED: return "record is a proper-pair mate: htslib overlap handling (H2) is not implemented -- refusing";
        case E_NEGPOS: return "record has POS 0 on a reference";
        case E_REFSPAN: return "record spans more than 65535 reference bases";
        case E_CIGQ: return "CIGAR query length != l_seq";
        case E_AUX: return "malformed aux field";
        case E_AUXPOS: return "1st / 4th aux field missing or not an integer: the reference crashes at metamlst.py:109-110";
        case E_AS0: return "1st aux field outside int16";
        case E_XM3: return "negative 4th aux field";
        case E_NAMED: return "record enters the pileup without integer AS:i / XM:i tags (pysam get_tag KeyError, cmseq/cmseq.py:545)";
        case E_NOQUAL: return "record has no base qualities: query_qualities is None (TypeError at cmseq/cmseq.py:538)";
        case E_QLEN: return "read longer than 65535 bases (len(SEQ) is carried as 16 bits)";
        case E_CRC: return "CRC mismatch in BGZF block";
        default: return "hardware decompression produced a block of the wrong size / record chain broken";
    }
}
int err_class(uint32_t code) {
    switch (code) {
        case E_PAIRED: return MMLST_E_PAIRED;
        case E_REFSPAN: case E_AS0: case E_XM3: case E_QLEN: return MMLST_E_RANGE;
        default: return MMLST_E_BAM;
    }
}

inline uint32_t h_rd16(const uint8_t* p) { return p[0] | (p[1] << 8); }
inline uint32_t h_rd32(const uint8_t* p) { return p[0] | (p[1] << 8) | (p[2] << 16) | (static_cast<uint32_t>(p[3]) << 24); }

}  // namespace

struct mmlst_dev_bam {
    int device = 0;
    DBuf tid, as0, xm3, qlen, orig_idx, qhash, run_tid, run_start, chunk_run, chunk_qlen, p_recs, planes;
    std::vector<uint64_t> contig_start;
    std::vector<uint32_t> ref_len;
    std::string names_blob, header_text;
    uint64_t n_rec = 0, n_prec = 0, n_plane_words = 0, n_dropped = 0, n_unmapped = 0, n_blocks = 0, comp_bytes = 0, infl_bytes = 0, n_untagged = 0;
    uint32_t n_runs = 0, max_row_words = 0, n_ref = 0, max_depth = 0, repairs = 0;
    int presorted = 0, minqual = 20, qc = 0, explicit_idx = 0;   // explicit_idx: a shard's streams carry orig_idx even in file order
    double seconds[8] = {0, 0, 0, 0, 0, 0, 0, 0};
};

extern "C" void mmlst_dev_bam_free(mmlst_dev_bam* b) {
    if (!b) return;
    cudaSetDevice(b->device);
    cudaDeviceSynchronize();   // whatever stream still reads the streams: the blocks go back to the cache for any stream to take
    for (DBuf* d : {&b->tid, &b->as0, &b->xm3, &b->qlen, &b->orig_idx, &b->qhash, &b->run_tid, &b->run_start, &b->chunk_run, &b->chunk_qlen, &b->p_recs, &b->planes}) {
        if (d->p) ws_put(d->dev, d->p, d->st, false);
        d->p = nullptr;
    }
    delete b;
}

extern "C" int mmlst_ingest_trim(int device) {
    CUDA_TRY(cudaSetDevice(device));
    CUDA_TRY(cudaDeviceSynchronize());
    Workspace& w = g_ws[device % MMLST_MAX_DEVICES];
    std::lock_guard<std::mutex> g(w.m);
    for (size_t i = 0; i < w.blocks.size();) {
        if (!w.blocks[i].used) { if (w.blocks[i].has_ev) cudaEventDestroy(w.blocks[i].ev); cudaFree(w.blocks[i].p); w.blocks.erase(w.blocks.begin() + i); } else ++i;
    }
    return MMLST_OK;
}

extern "C" int mmlst_dev_bam_info(const mmlst_dev_bam* b, mmlst_dev_bam_info_t* o) {
    if (!b || !o) { mmlst_set_error("mmlst_dev_bam_info: null argument"); return MMLST_E_ARG; }
    memset(o, 0, sizeof(*o));
    o->tid = b->tid.as<uint32_t>(); o->as0 = b->as0.as<int16_t>(); o->xm3 = b->xm3.as<uint8_t>(); o->qlen = b->qlen.as<uint16_t>();
    o->orig_idx = (b->presorted && !b->explicit_idx) ? nullptr : b->orig_idx.as<uint32_t>();
    o->qhash = b->qhash.as<uint64_t>();
    o->run_tid = b->run_tid.as<uint32_t>(); o->run_start = b->run_start.as<uint32_t>(); o->chunk_run = b->chunk_run.as<uint32_t>();
    o->chunk_qlen = b->qc ? b->chunk_qlen.as<uint16_t>() : nullptr;
    o->n_runs = b->n_runs;
    o->p_recs = b->p_recs.as<mmlst_prec>(); o->planes = b->planes.as<uint32_t>();
    o->n_rec = b->n_rec; o->n_prec = b->n_prec; o->n_plane_words = b->n_plane_words; o->max_row_words = b->max_row_words;
    o->contig_start = b->contig_start.data(); o->ref_len = b->ref_len.data(); o->ref_names = b->names_blob.c_str();
    o->header_text = b->header_text.c_str(); o->n_ref = b->n_ref;
    o->n_dropped_by_cap = b->n_dropped; o->n_unmapped_flag = b->n_unmapped; o->n_bgzf_blocks = b->n_blocks;
    o->compressed_bytes = b->comp_bytes; o->inflated_bytes = b->infl_bytes;
    o->presorted = b->presorted; o->minqual = b->minqual; o->max_depth = b->max_depth; o->boundary_repairs = static_cast<int>(b->repairs);
    for (int i = 0; i < 8; ++i) o->seconds[i] = b->seconds[i];
    o->n_untagged = b->n_untagged;
    return MMLST_OK;
}

#define ING_TRY(expr) do { int _r = (expr); if (_r != MMLST_OK) return _r; } while (0)

static int fetch_error(unsigned long long* d_err, cudaStream_t st, const char* what, unsigned long long* got = nullptr) {
    unsigned long long e = kNoErr;
    CUDA_TRY(cudaMemcpyAsync(&e, d_err, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (got) *got = e;
    if (e == kNoErr) return MMLST_OK;
    const uint32_t code = static_cast<uint32_t>(e & 0xff);
    mmlst_set_error("%s: record %llu: %s", what, static_cast<unsigned long long>(e >> 8), err_text(code));
    return err_class(code);
}


namespace {

struct Blk { uint64_t coff; uint32_t clen, isize, crc; uint64_t uoff; };

// BGZF block table of bam[0, n_bytes): payload offset / size, CRC, ISIZE and inflated offset of every non-empty block
int scan_blocks(const uint8_t* bam, size_t n_bytes, std::vector<Blk>& blocks, uint64_t& usize) {
    usize = 0;
    for (size_t p = 0; p < n_bytes;) {
        if (n_bytes - p < 18 || bam[p] != 0x1f || bam[p + 1] != 0x8b || bam[p + 2] != 8 || !(bam[p + 3] & 4)) {
            mmlst_set_error("mmlst_bam_ingest: not a BGZF block at byte %zu (plain gzip / truncated file?)", p);
            return MMLST_E_BAM;
        }
        const uint32_t xlen = h_rd16(&bam[p + 10]);
        if (n_bytes - p < 12 + static_cast<size_t>(xlen) + 8) { mmlst_set_error("mmlst_bam_ingest: truncated BGZF header at %zu", p); return MMLST_E_BAM; }
        int64_t bsize = -1;
        for (size_t q = p + 12; q + 4 <= p + 12 + xlen;) {
            const uint32_t slen = h_rd16(&bam[q + 2]);
            if (bam[q] == 66 && bam[q + 1] == 67 && slen == 2) bsize = h_rd16(&bam[q + 4]);
            q += 4 + slen;
        }
        if (bsize < 0) { mmlst_set_error("mmlst_bam_ingest: BGZF block without BC subfield at %zu", p); return MMLST_E_BAM; }
        const size_t total = static_cast<size_t>(bsize) + 1;
        if (total < 12 + static_cast<size_t>(xlen) + 8 || n_bytes - p < total) { mmlst_set_error("mmlst_bam_ingest: truncated BGZF block at %zu", p); return MMLST_E_BAM; }
        Blk b;
        b.coff = p + 12 + xlen;
        b.clen = static_cast<uint32_t>(total - 12 - xlen - 8);
        b.crc = h_rd32(&bam[p + total - 8]);
        b.isize = h_rd32(&bam[p + total - 4]);
        b.uoff = usize;
        if (b.isize > 65536) { mmlst_set_error("mmlst_bam_ingest: BGZF block with ISIZE %u > 64 KiB at %zu", b.isize, p); return MMLST_E_BAM; }
        usize += b.isize;
        if (b.isize) blocks.push_back(b);
        p += total;
    }
    return MMLST_OK;
}

// Device buffers of the inflated stream and its block table
struct Inflated {
    DBuf d_comp, d_u, d_act, d_isize, d_uoff, d_crc;
};

// H2D + hardware inflate of every block, ISIZE check of every block, CRC-32 of the first n_crc blocks (opts.check_crc); failures go to
// err as (block << 8 | code).  mark() is called after the block table is uploaded (the H2D / inflate split of the phase timer).
template <class Mark>
int inflate_blocks(int device, cudaStream_t st, const uint8_t* bam, size_t n_bytes, const std::vector<Blk>& blocks, uint64_t usize, bool check_crc,
                   uint32_t n_crc, Inflated& I, unsigned long long* err, Mark&& mark) {
    const uint32_t nb = static_cast<uint32_t>(blocks.size());
    ING_TRY(I.d_comp.alloc(n_bytes + 64));
    ING_TRY(I.d_u.alloc(usize + 64));
    ING_TRY(I.d_act.alloc(static_cast<size_t>(nb) * 4));
    ING_TRY(I.d_isize.alloc(static_cast<size_t>(nb) * 4));
    ING_TRY(I.d_uoff.alloc((static_cast<size_t>(nb) + 1) * 8));
    if (check_crc) ING_TRY(I.d_crc.alloc(static_cast<size_t>(nb) * 4));
    std::vector<uint32_t> h_isize(nb);
    std::vector<uint64_t> h_uoff(nb + 1);
    for (uint32_t b = 0; b < nb; ++b) { h_isize[b] = blocks[b].isize; h_uoff[b] = blocks[b].uoff; }
    h_uoff[nb] = usize;
    CUDA_TRY(cudaMemcpyAsync(I.d_isize.p, h_isize.data(), static_cast<size_t>(nb) * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(I.d_uoff.p, h_uoff.data(), (static_cast<size_t>(nb) + 1) * 8, cudaMemcpyHostToDevice, st));
    std::vector<uint32_t> h_want;
    if (check_crc) {   // the raw CRC each block must have: trailer ^ crc32(0^isize)
        static const std::vector<uint32_t> zeros = [] { std::vector<uint32_t> z(65537); bgzf_crc::make_zeros(z.data(), 65536); return z; }();
        h_want.resize(nb);
        for (uint32_t b = 0; b < nb; ++b) h_want[b] = blocks[b].crc ^ zeros[blocks[b].isize];
        CUDA_TRY(cudaMemcpyAsync(I.d_crc.p, h_want.data(), static_cast<size_t>(nb) * 4, cudaMemcpyHostToDevice, st));
    }
    mark();
    if (nb == 0) return MMLST_OK;
    std::vector<CUmemDecompressParams> prm(nb);
    memset(prm.data(), 0, sizeof(CUmemDecompressParams) * nb);
    for (uint32_t b = 0; b < nb; ++b) {
        prm[b].srcNumBytes = blocks[b].clen;
        prm[b].dstNumBytes = blocks[b].isize;
        prm[b].dstActBytes = I.d_act.as<cuuint32_t>() + b;
        prm[b].src = I.d_comp.as<uint8_t>() + blocks[b].coff;
        prm[b].dst = I.d_u.as<uint8_t>() + blocks[b].uoff;
        prm[b].algo = CU_MEM_DECOMPRESS_ALGORITHM_DEFLATE;
    }
    // the file goes over in slices on a copy stream while the decompression engine works on the slices that have landed: the copy
    // engine and the decompression engine are different units, so PCIe time hides behind the inflate (or the other way round)
    {
        std::vector<uint64_t> src_off(nb);
        for (uint32_t b = 0; b < nb; ++b) src_off[b] = blocks[b].coff;
        ING_TRY(mmlst_h2d_inflate(device, st, I.d_comp.as<uint8_t>(), bam, n_bytes, prm, src_off));
    }
    check_isize_kernel<<<(nb + kT - 1) / kT, kT, 0, st>>>(I.d_act.as<uint32_t>(), I.d_isize.as<uint32_t>(), nb, err);
    CUDA_TRY(cudaGetLastError());
    if (check_crc && n_crc) {
        static const CrcArgs proto = [] { CrcArgs c{}; bgzf_crc::make_ops(c.ops); return c; }();
        CrcArgs ca = proto;
        ca.u = I.d_u.as<uint8_t>(); ca.uoff = I.d_uoff.as<uint64_t>(); ca.isize = I.d_isize.as<uint32_t>(); ca.want = I.d_crc.as<uint32_t>(); ca.n_blocks = n_crc;
        int sms = 0, per_sm = 0;
        CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, crc_kernel, bgzf_crc::kCrcThreads, 0));
        const uint32_t grid = std::min<uint32_t>(n_crc, static_cast<uint32_t>(std::max(sms, 1) * std::max(per_sm, 1)));
        crc_kernel<<<grid, bgzf_crc::kCrcThreads, 0, st>>>(ca, err);
        CUDA_TRY(cudaGetLastError());
    }
    return MMLST_OK;
}

// K1: guess every block's first record boundary, then verify / repair until nothing changes
int run_chain(const ChainArgs& ca, uint32_t* d_changed, cudaStream_t st, uint32_t* repairs) {
    const uint32_t nb = ca.n_blocks;
    chain_guess_kernel<<<(nb + kT - 1) / kT, kT, 0, st>>>(ca);
    CUDA_TRY(cudaGetLastError());
    for (uint32_t sweep = 0;; ++sweep) {
        CUDA_TRY(cudaMemsetAsync(d_changed, 0, 4, st));
        chain_repair_kernel<<<(nb + kT - 1) / kT, kT, 0, st>>>(ca, d_changed);
        CUDA_TRY(cudaGetLastError());
        uint32_t changed = 0;
        CUDA_TRY(cudaMemcpyAsync(&changed, d_changed, 4, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        if (!changed) break;
        *repairs += changed;
        if (sweep > nb) { mmlst_set_error("mmlst_bam_ingest: record chain did not converge"); return MMLST_E_BAM; }
    }
    return MMLST_OK;
}

// Where the back half stopped: 1 = a record refusal (K2), 2 = --presorted on records out of coordinate order, 3 = plane array too
// large, 4 = a refusal of a record entering the pileup (K5).  A shard's ranks agree on the least (phase, error word) before raising.
enum BackPhase { kPhaseRecord = 1, kPhaseUnsorted = 2, kPhasePlanes = 3, kPhasePileup = 4 };

struct BackIn {
    const uint8_t* u; const uint64_t* roff; const uint32_t* gidx; uint64_t n;   // gidx: file index of record i (shards); nullptr = i
    int32_t n_ref; const uint32_t* d_reflen;
    unsigned long long* err; uint32_t* d_flags;
    int unsorted;   // -1: decide from these records (the whole file); 0 / 1: decided across the shards of the file
};

const char* kUnsortedText = "mmlst_bam_ingest: --presorted given but records are not coordinate-sorted (htslib: 'The input is not sorted')";

// The records known, everything after: K2 parse -> sort (stable by key, then file index) -> K3 score stream -> K4 depth cap -> K5 plane
// rows.  The one back half of the whole-file ingest and of a shard's owner.  mark() after K2, the sort, K3, K4 and K5.
template <class Mark>
int back_half(const BackIn& in, const mmlst_unpack_opts& o, cudaStream_t st, mmlst_dev_bam* B, Mark&& mark, int* phase, unsigned long long* err_word) {
    const uint64_t n = in.n;
    const int32_t n_ref = in.n_ref;
    unsigned long long* err = in.err;
    uint32_t* d_flags = in.d_flags;
    B->explicit_idx = in.gidx ? 1 : 0;
    // ---- K2: per record
    DBuf k_key, k_reflen, k_as0, k_asn, k_qlen, k_xm3, k_xmn, k_bits, k_qh;
    ING_TRY(k_key.alloc(n * 8)); ING_TRY(k_reflen.alloc(n * 2)); ING_TRY(k_as0.alloc(n * 2)); ING_TRY(k_asn.alloc(n * 2)); ING_TRY(k_qlen.alloc(n * 2));
    ING_TRY(k_xm3.alloc(n)); ING_TRY(k_xmn.alloc(n)); ING_TRY(k_bits.alloc(n));
    if (o.want_qhash) ING_TRY(k_qh.alloc(n * 16));
    const ParseOut po{k_key.as<uint64_t>(), k_reflen.as<uint16_t>(), k_as0.as<int16_t>(), k_asn.as<int16_t>(), k_qlen.as<uint16_t>(), k_xm3.as<uint8_t>(),
                      k_xmn.as<uint8_t>(), k_bits.as<uint8_t>(), o.want_qhash ? k_qh.as<uint64_t>() : nullptr};
    const unsigned gn = static_cast<unsigned>((n + kT - 1) / kT);
    if (n) {
        parse_kernel<<<gn, kT, 0, st>>>(in.u, in.roff, in.gidx, n, n_ref, po, o.lenient_tags != 0, err);
        CUDA_TRY(cudaGetLastError());
        check_sorted_kernel<<<gn, kT, 0, st>>>(k_key.as<uint64_t>(), n, d_flags);
        CUDA_TRY(cudaGetLastError());
    }
    uint32_t sflags = 0;
    CUDA_TRY(cudaMemcpyAsync(&sflags, d_flags, 4, cudaMemcpyDeviceToHost, st));
    {
        const int rc = fetch_error(err, st, "mmlst_bam_ingest", err_word);
        if (rc != MMLST_OK) { *phase = kPhaseRecord; return rc; }
    }
    mark();  // 4
    bool sorted = !(sflags & 1u);
    if (o.assume_sorted) {
        if (in.unsorted < 0 ? (sflags & 2u) != 0 : in.unsorted != 0) { mmlst_set_error("%s", kUnsortedText); *phase = kPhaseUnsorted; *err_word = 0; return MMLST_E_UNSORTED; }
        sorted = true;
    }
    B->presorted = sorted ? 1 : 0;
    const bool keep_idx = !sorted || in.gidx;

    // ---- sort
    DBuf d_key2, d_ord, d_ord2;
    const uint64_t* key_sorted = k_key.as<uint64_t>();
    const uint32_t* order = nullptr;
    if (!sorted && n) {
        ING_TRY(d_key2.alloc(n * 8)); ING_TRY(d_ord.alloc(n * 4)); ING_TRY(d_ord2.alloc(n * 4));
        iota_kernel<<<gn, kT, 0, st>>>(d_ord.as<uint32_t>(), n);
        CUDA_TRY(cudaGetLastError());
        int end_bit = 34;
        while (end_bit < 64 && (static_cast<uint64_t>(n_ref) >> (end_bit - 33)) != 0) ++end_bit;
        size_t sb = 0;
        CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, sb, k_key.as<uint64_t>(), d_key2.as<uint64_t>(), d_ord.as<uint32_t>(), d_ord2.as<uint32_t>(),
                                                 static_cast<int>(n), 0, end_bit, st));
        DBuf d_sorttmp;
        ING_TRY(d_sorttmp.alloc(sb));
        CUDA_TRY(cub::DeviceRadixSort::SortPairs(d_sorttmp.p, sb, k_key.as<uint64_t>(), d_key2.as<uint64_t>(), d_ord.as<uint32_t>(), d_ord2.as<uint32_t>(),
                                                 static_cast<int>(n), 0, end_bit, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        key_sorted = d_key2.as<uint64_t>();
        order = d_ord2.as<uint32_t>();
    }
    mark();  // 5

    // ---- K3: score stream
    B->n_rec = n;
    ING_TRY(B->tid.alloc(n * 4)); ING_TRY(B->as0.alloc(n * 2)); ING_TRY(B->xm3.alloc(n)); ING_TRY(B->qlen.alloc(n * 2));
    if (keep_idx) ING_TRY(B->orig_idx.alloc(n * 4));
    if (o.want_qhash) ING_TRY(B->qhash.alloc(n * 16));
    DBuf s_pos, s_reflen, s_bits, s_asn, s_xmn, s_roff, d_runflag, d_runincl;
    ING_TRY(s_pos.alloc(n * 4)); ING_TRY(s_reflen.alloc(n * 2)); ING_TRY(s_bits.alloc(n)); ING_TRY(s_asn.alloc(n * 2)); ING_TRY(s_xmn.alloc(n)); ING_TRY(s_roff.alloc(n * 8));
    ING_TRY(d_runflag.alloc(n * 4 + 4)); ING_TRY(d_runincl.alloc(n * 4 + 4));
    uint32_t n_runs = 0;
    const uint64_t n_chunks = (n + 255) / 256;
    ING_TRY(B->chunk_run.alloc(n_chunks * 4)); ING_TRY(B->chunk_qlen.alloc(n_chunks * 2));
    if (n) {
        const GatherArgs ga{key_sorted, order, po, in.roff, in.gidx, B->tid.as<uint32_t>(), B->as0.as<int16_t>(), B->xm3.as<uint8_t>(), B->qlen.as<uint16_t>(),
                            keep_idx ? B->orig_idx.as<uint32_t>() : nullptr, o.want_qhash ? B->qhash.as<uint64_t>() : nullptr,
                            s_pos.as<int32_t>(), s_reflen.as<uint16_t>(), s_bits.as<uint8_t>(), s_asn.as<int16_t>(), s_xmn.as<uint8_t>(), s_roff.as<uint64_t>(),
                            d_runflag.as<uint32_t>(), d_flags + 4, n};
        gather_kernel<<<gn, kT, 0, st>>>(ga);
        CUDA_TRY(cudaGetLastError());
        size_t sb = 0;
        CUDA_TRY(cub::DeviceScan::InclusiveSum(nullptr, sb, d_runflag.as<uint32_t>(), d_runincl.as<uint32_t>(), static_cast<int>(n), st));
        DBuf d_scantmp;
        ING_TRY(d_scantmp.alloc(sb));
        CUDA_TRY(cub::DeviceScan::InclusiveSum(d_scantmp.p, sb, d_runflag.as<uint32_t>(), d_runincl.as<uint32_t>(), static_cast<int>(n), st));
        CUDA_TRY(cudaMemcpyAsync(&n_runs, d_runincl.as<uint32_t>() + (n - 1), 4, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        ING_TRY(B->run_tid.alloc(static_cast<size_t>(n_runs) * 4)); ING_TRY(B->run_start.alloc((static_cast<size_t>(n_runs) + 1) * 4));
        runs_kernel<<<gn, kT, 0, st>>>(d_runflag.as<uint32_t>(), d_runincl.as<uint32_t>(), B->tid.as<uint32_t>(), n, B->run_tid.as<uint32_t>(),
                                       B->run_start.as<uint32_t>(), B->chunk_run.as<uint32_t>());
        CUDA_TRY(cudaGetLastError());
        const uint32_t one = 1;
        CUDA_TRY(cudaMemcpyAsync(d_flags + 2, &one, 4, cudaMemcpyHostToDevice, st));
        chunk_qlen_kernel<<<static_cast<unsigned>((n_chunks * 32 + kT - 1) / kT), kT, 0, st>>>(B->qlen.as<uint16_t>(), n, B->chunk_qlen.as<uint16_t>(), d_flags + 2);
        CUDA_TRY(cudaGetLastError());
    }
    B->n_runs = n_runs;
    mark();  // 6

    // ---- K4: depth cap
    DBuf d_adm, d_admx, d_hsz, d_hoff, d_hist, d_list, d_rw, d_rowoff, d_cs;
    ING_TRY(d_adm.alloc(n * 4 + 4)); ING_TRY(d_admx.alloc(n * 4 + 4));
    ING_TRY(d_cs.alloc((static_cast<size_t>(n_ref) + 1) * 8));
    uint64_t P = 0, total_words = 0;
    uint32_t fl[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    B->contig_start.assign(static_cast<size_t>(n_ref) + 1, 0);
    if (n) {
        CUDA_TRY(cudaMemsetAsync(d_adm.p, 0, n * 4 + 4, st));
        ING_TRY(d_hsz.alloc((static_cast<size_t>(n_runs) + 1) * 8)); ING_TRY(d_hoff.alloc((static_cast<size_t>(n_runs) + 1) * 8));
        CapArgs cap{B->run_tid.as<uint32_t>(), B->run_start.as<uint32_t>(), n_runs, s_pos.as<int32_t>(), s_reflen.as<uint16_t>(), s_bits.as<uint8_t>(),
                    in.d_reflen, o.max_depth, o.sentinel_nodes, nullptr, nullptr, d_adm.as<uint32_t>()};
        CUDA_TRY(cudaMemsetAsync(d_hsz.p, 0, (static_cast<size_t>(n_runs) + 1) * 8, st));
        cap_sizes_kernel<<<(n_runs + kT - 1) / kT, kT, 0, st>>>(cap, d_hsz.as<uint64_t>());
        CUDA_TRY(cudaGetLastError());
        size_t sb = 0;
        CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, sb, d_hsz.as<uint64_t>(), d_hoff.as<uint64_t>(), static_cast<int>(n_runs + 1), st));
        DBuf t1;
        ING_TRY(t1.alloc(sb));
        CUDA_TRY(cub::DeviceScan::ExclusiveSum(t1.p, sb, d_hsz.as<uint64_t>(), d_hoff.as<uint64_t>(), static_cast<int>(n_runs + 1), st));
        uint64_t hist_words = 0;
        CUDA_TRY(cudaMemcpyAsync(&hist_words, d_hoff.as<uint64_t>() + n_runs, 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        ING_TRY(d_hist.alloc(hist_words * 4 + 16));
        CUDA_TRY(cudaMemsetAsync(d_hist.p, 0, hist_words * 4 + 16, st));
        cap.hist_off = d_hoff.as<uint64_t>(); cap.hist = d_hist.as<uint32_t>();
        cap_kernel<<<static_cast<unsigned>((static_cast<uint64_t>(n_runs) * 32 + kT - 1) / kT), kT, 0, st>>>(cap);
        CUDA_TRY(cudaGetLastError());
        // ---- K5: compaction
        CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, sb, d_adm.as<uint32_t>(), d_admx.as<uint32_t>(), static_cast<int>(n + 1), st));
        DBuf t2;
        ING_TRY(t2.alloc(sb));
        CUDA_TRY(cub::DeviceScan::ExclusiveSum(t2.p, sb, d_adm.as<uint32_t>(), d_admx.as<uint32_t>(), static_cast<int>(n + 1), st));
        uint32_t P32 = 0;
        CUDA_TRY(cudaMemcpyAsync(&P32, d_admx.as<uint32_t>() + n, 4, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        P = P32;
        ING_TRY(d_list.alloc(P * 4)); ING_TRY(d_rw.alloc((P + 1) * 8)); ING_TRY(d_rowoff.alloc((P + 1) * 8));
        scatter_adm_kernel<<<gn, kT, 0, st>>>(d_adm.as<uint32_t>(), d_admx.as<uint32_t>(), n, d_list.as<uint32_t>());
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaMemsetAsync(d_rw.p, 0, (P + 1) * 8, st));
        if (P) {
            row_sizes_kernel<<<static_cast<unsigned>((P + kT - 1) / kT), kT, 0, st>>>(d_list.as<uint32_t>(), P, s_pos.as<int32_t>(), s_reflen.as<uint16_t>(),
                                                                                     d_rw.as<uint64_t>(), d_flags + 3);
            CUDA_TRY(cudaGetLastError());
        }
        CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, sb, d_rw.as<uint64_t>(), d_rowoff.as<uint64_t>(), static_cast<int>(P + 1), st));
        DBuf t3;
        ING_TRY(t3.alloc(sb));
        CUDA_TRY(cub::DeviceScan::ExclusiveSum(t3.p, sb, d_rw.as<uint64_t>(), d_rowoff.as<uint64_t>(), static_cast<int>(P + 1), st));
        contig_start_kernel<<<(static_cast<unsigned>(n_ref) + 1 + kT - 1) / kT, kT, 0, st>>>(B->run_tid.as<uint32_t>(), B->run_start.as<uint32_t>(), n_runs,
                                                                                             d_admx.as<uint32_t>(), P, static_cast<uint32_t>(n_ref), d_cs.as<uint64_t>());
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaMemcpyAsync(&total_words, d_rowoff.as<uint64_t>() + P, 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaMemcpyAsync(fl, d_flags, 32, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaMemcpyAsync(B->contig_start.data(), d_cs.p, (static_cast<size_t>(n_ref) + 1) * 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
    }
    mark();  // 7
    const uint64_t kSlack = 8;
    if (total_words + kSlack >= (1ull << 32)) { mmlst_set_error("mmlst_bam_ingest: plane array exceeds 2^32 words"); *phase = kPhasePlanes; *err_word = 0; return MMLST_E_RANGE; }
    B->n_prec = P; B->n_plane_words = total_words + kSlack; B->max_row_words = fl[3]; B->qc = (n && fl[2]) ? 1 : 0;
    ING_TRY(B->p_recs.alloc(P * sizeof(mmlst_prec))); ING_TRY(B->planes.alloc((total_words + kSlack) * 4));
    CUDA_TRY(cudaMemsetAsync(B->planes.as<uint32_t>() + total_words, 0, kSlack * 4, st));
    if (P) {
        const PackArgs pa{in.u, d_list.as<uint32_t>(), P, d_rowoff.as<uint64_t>(), s_pos.as<int32_t>(), s_reflen.as<uint16_t>(), s_bits.as<uint8_t>(),
                          s_asn.as<int16_t>(), s_xmn.as<uint8_t>(), s_roff.as<uint64_t>(), keep_idx ? B->orig_idx.as<uint32_t>() : nullptr, o.minqual,
                          B->p_recs.as<mmlst_prec>(), B->planes.as<uint32_t>(), o.lenient_tags != 0, d_flags + 5};
        pack_kernel<<<static_cast<unsigned>((P * 32 + kT - 1) / kT), kT, 0, st>>>(pa, err);
        CUDA_TRY(cudaGetLastError());
    }
    mark();  // 8
    uint32_t n_untagged = 0;
    CUDA_TRY(cudaMemcpyAsync(&n_untagged, d_flags + 5, 4, cudaMemcpyDeviceToHost, st));
    {
        const int rc = fetch_error(err, st, "mmlst_bam_ingest (pileup stream)", err_word);
        if (rc != MMLST_OK) { *phase = kPhasePileup; return rc; }
    }
    B->n_untagged = n_untagged;
    B->n_unmapped = fl[4];
    B->n_dropped = n - fl[4] - P;
    B->minqual = o.minqual; B->max_depth = o.max_depth;
    CUDA_TRY(cudaStreamSynchronize(st));
    return MMLST_OK;
}

mmlst_unpack_opts ingest_opts(const mmlst_unpack_opts* opts_in) {
    mmlst_unpack_opts o;
    o.minqual = 20; o.max_depth = 8000; o.sentinel_nodes = 1; o.n_threads = 0; o.pinned = 1; o.assume_sorted = 0; o.want_qhash = 1; o.check_crc = 0; o.lenient_tags = 0;
    if (opts_in) o = *opts_in;
    return o;
}

}  // namespace

extern "C" int mmlst_bam_ingest(int device, const uint8_t* bam, size_t n_bytes, const mmlst_unpack_opts* opts_in, void* stream_in, mmlst_dev_bam** out) {
    if (!bam || !out) { mmlst_set_error("mmlst_bam_ingest: null argument"); return MMLST_E_ARG; }
    const mmlst_unpack_opts o = ingest_opts(opts_in);
    CUDA_TRY(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream_in);
    g_cur_stream = st;
    {
        const int rc = mmlst_de_available(device);
        if (rc != MMLST_OK) { mmlst_set_error("mmlst_bam_ingest: %s; use mmlst_bam_unpack", mmlst_last_error()); return rc; }
    }
    // ---- host: BGZF block table
    std::vector<Blk> blocks;
    uint64_t usize = 0;
    ING_TRY(scan_blocks(bam, n_bytes, blocks, usize));
    const uint32_t nb = static_cast<uint32_t>(blocks.size());
    if (usize < 12 || nb == 0) { mmlst_set_error("mmlst_bam_ingest: not a BAM file (empty)"); return MMLST_E_BAM; }

    cudaEvent_t ev[10];
    for (auto& e : ev) CUDA_TRY(cudaEventCreate(&e));
    struct EvGuard { cudaEvent_t* e; ~EvGuard() { for (int i = 0; i < 10; ++i) cudaEventDestroy(e[i]); } } evg{ev};
    int evn = 0;
    auto mark = [&]() { cudaEventRecord(ev[evn++], st); };

    // ---- H2D + hardware inflate
    DBuf d_err;
    ING_TRY(d_err.alloc(8 + 32));
    unsigned long long* err = d_err.as<unsigned long long>();
    uint32_t* d_flags = reinterpret_cast<uint32_t*>(err + 1);   // [0] sortedness, [1] repair counter, [2] uniform qlen, [3] max row words, [4] records with the unmapped flag,
                                                                //  [5] untagged pileup records (lenient_tags)
    CUDA_TRY(cudaMemsetAsync(err, 0xff, 8, st));
    CUDA_TRY(cudaMemsetAsync(d_flags, 0, 32, st));
    mark();  // 0
    Inflated I;
    ING_TRY(inflate_blocks(device, st, bam, n_bytes, blocks, usize, o.check_crc != 0, nb, I, err, mark));   // mark 1 inside
    mark();  // 2
    // ---- header (first bytes of the inflated stream come back to the host)
    std::unique_ptr<mmlst_dev_bam> B(new mmlst_dev_bam());
    B->device = device;
    PinnedStage stage_guard(device);   // page-locked staging for the header, cached per device (a pageable D2H of a megabyte costs a millisecond)
    const uint8_t* head = nullptr;
    uint64_t first_record = 0;
    {
        // l_text first (16 bytes), then ONE right-sized fetch: the reference dictionary is never longer than the @SQ lines that describe it
        size_t want = std::min<uint64_t>(usize, 16);
        for (int round = 0;; ++round) {
            uint8_t* hb = stage_guard.get(want);
            if (!hb) { mmlst_set_error("mmlst_bam_ingest: cudaHostAlloc(%zu) failed", want); return MMLST_E_NOMEM; }
            head = hb;
            CUDA_TRY(cudaMemcpyAsync(hb, I.d_u.p, want, cudaMemcpyDeviceToHost, st));
            {
                unsigned long long e = kNoErr;
                const int rc = fetch_error(err, st, "mmlst_bam_ingest (inflate)", &e);
                if (rc != MMLST_OK) {
                    // block k counts the non-empty blocks, as the host unpacker's message does
                    if (e != kNoErr && (e & 0xff) == E_CRC) mmlst_set_error("mmlst_bam_ingest: CRC mismatch in BGZF block %llu", e >> 8);
                    else mmlst_set_error("mmlst_bam_ingest: a BGZF block did not inflate to its ISIZE (corrupt file?)");
                    return MMLST_E_BAM;
                }
            }
            if (round == 0 && want >= 12 && want < usize && memcmp(head, "BAM\1", 4) == 0) {
                const int32_t lt = static_cast<int32_t>(h_rd32(&head[4]));
                if (lt >= 0) { want = std::min<uint64_t>(usize, 2ull * static_cast<uint64_t>(lt) + (64u << 10)); continue; }
            }
            if (want < 12 || memcmp(head, "BAM\1", 4) != 0) { mmlst_set_error("mmlst_bam_ingest: not a BAM file (magic)"); return MMLST_E_BAM; }
            size_t p = 4;
            bool more = false;
            const int32_t l_text = static_cast<int32_t>(h_rd32(&head[p])); p += 4;
            if (l_text < 0 || p + static_cast<uint64_t>(l_text) + 4 > usize) { mmlst_set_error("mmlst_bam_ingest: bad l_text"); return MMLST_E_BAM; }
            if (p + static_cast<size_t>(l_text) + 4 > want) more = true;
            int32_t n_ref = 0;
            if (!more) {
                B->header_text.assign(reinterpret_cast<const char*>(&head[p]), strnlen(reinterpret_cast<const char*>(&head[p]), static_cast<size_t>(l_text)));
                p += static_cast<size_t>(l_text);
                n_ref = static_cast<int32_t>(h_rd32(&head[p])); p += 4;
                if (n_ref < 0) { mmlst_set_error("mmlst_bam_ingest: bad n_ref"); return MMLST_E_BAM; }
                B->ref_len.clear(); B->names_blob.clear();
                B->ref_len.reserve(n_ref);
                for (int32_t i = 0; i < n_ref && !more; ++i) {
                    if (p + 4 > want) { more = true; break; }
                    const int32_t ln = static_cast<int32_t>(h_rd32(&head[p])); p += 4;
                    if (ln < 1 || p + static_cast<uint64_t>(ln) + 4 > usize) { mmlst_set_error("mmlst_bam_ingest: truncated reference dictionary"); return MMLST_E_BAM; }
                    if (p + static_cast<size_t>(ln) + 4 > want) { more = true; break; }
                    if (i) B->names_blob.push_back('\n');
                    B->names_blob.append(reinterpret_cast<const char*>(&head[p]), strnlen(reinterpret_cast<const char*>(&head[p]), static_cast<size_t>(ln)));
                    p += static_cast<size_t>(ln);
                    B->ref_len.push_back(h_rd32(&head[p])); p += 4;
                }
            }
            if (!more) { B->n_ref = static_cast<uint32_t>(n_ref); first_record = p; break; }
            if (want >= usize) { mmlst_set_error("mmlst_bam_ingest: truncated BAM header"); return MMLST_E_BAM; }
            want = std::min<uint64_t>(usize, want * 4);
        }
    }
    const int32_t n_ref = static_cast<int32_t>(B->n_ref);
    DBuf d_reflen;
    ING_TRY(d_reflen.alloc(static_cast<size_t>(n_ref) * 4 + 16));
    if (n_ref) CUDA_TRY(cudaMemcpyAsync(d_reflen.p, B->ref_len.data(), static_cast<size_t>(n_ref) * 4, cudaMemcpyHostToDevice, st));

    // ---- K1: record chain
    DBuf d_start, d_exit, d_count, d_badw, d_base, d_tmp;
    ING_TRY(d_start.alloc(static_cast<size_t>(nb) * 8)); ING_TRY(d_exit.alloc(static_cast<size_t>(nb) * 8));
    ING_TRY(d_count.alloc(static_cast<size_t>(nb) * 4 + 4)); ING_TRY(d_badw.alloc(static_cast<size_t>(nb) * 4)); ING_TRY(d_base.alloc(static_cast<size_t>(nb) * 4 + 4));
    const ChainArgs ca{I.d_u.as<uint8_t>(), usize, I.d_uoff.as<uint64_t>(), nb, first_record, n_ref, d_reflen.as<uint32_t>(),
                       d_start.as<uint64_t>(), d_exit.as<uint64_t>(), d_count.as<uint32_t>(), d_badw.as<uint32_t>(), usize, nullptr};
    ING_TRY(run_chain(ca, d_flags + 1, st, &B->repairs));
    size_t tmp_bytes = 0;
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_count.as<uint32_t>(), d_base.as<uint32_t>(), nb + 1, st));
    ING_TRY(d_tmp.alloc(tmp_bytes));
    CUDA_TRY(cudaMemsetAsync(d_count.as<uint32_t>() + nb, 0, 4, st));
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(d_tmp.p, tmp_bytes, d_count.as<uint32_t>(), d_base.as<uint32_t>(), nb + 1, st));
    uint32_t n32 = 0;
    CUDA_TRY(cudaMemcpyAsync(&n32, d_base.as<uint32_t>() + nb, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    const uint64_t n = n32;
    if (n >= 0x7fffff00ull) { mmlst_set_error("mmlst_bam_ingest: more than 2^31-257 records in one call"); return MMLST_E_RANGE; }
    DBuf d_roff;
    ING_TRY(d_roff.alloc(n * 8));
    chain_offsets_kernel<<<(nb + kT - 1) / kT, kT, 0, st>>>(ca, d_base.as<uint32_t>(), d_roff.as<uint64_t>(), err);
    CUDA_TRY(cudaGetLastError());
    mark();  // 3

    const BackIn in{I.d_u.as<uint8_t>(), d_roff.as<uint64_t>(), nullptr, n, n_ref, d_reflen.as<uint32_t>(), err, d_flags, -1};
    int phase = 0;
    unsigned long long ew = kNoErr;
    ING_TRY(back_half(in, o, st, B.get(), mark, &phase, &ew));
    B->n_blocks = nb; B->comp_bytes = n_bytes; B->infl_bytes = usize;
    // phase seconds from the device events: h2d, inflate, chain, parse, sort, score stream, cap + compaction, pack
    for (int i = 0; i + 1 < evn && i < 8; ++i) { float ms = 0; cudaEventElapsedTime(&ms, ev[i], ev[i + 1]); B->seconds[i] = ms * 1e-3; }
    *out = B.release();
    return MMLST_OK;
}

// ================================================================================================================================
// One BAM over several ranks.  Front half (per rank): the rank's own BGZF blocks (+ a halo of the next blocks, so that its last
// record can end there) are inflated, the record chain is walked from an agreed entry, and the records that START in its own blocks
// are partitioned by owner rank.  The ranks exchange the partitions; the back half (per owner) is back_half() above.
// ================================================================================================================================
struct mmlst_ingest_front {
    int device = 0;
    cudaStream_t st = nullptr;
    std::vector<Blk> blocks;
    uint32_t nb = 0, n_own = 0;
    uint64_t usize = 0, uend = 0, n_comp = 0;
    int32_t n_ref = 0;
    Inflated I;
    DBuf d_err, d_reflen, d_start, d_exit, d_count, d_badw, d_need, d_base, d_owner, d_roff, d_dest, d_rlen, d_order, d_boff, d_dcount, d_keys;
    DBuf send, send_len, send_idx;
    unsigned long long block_err = kNoErr, chain_err = kNoErr;
    uint64_t entry = kNoEntry, exit = kNoEntry, need = 0, n_rec = 0;
    uint32_t repairs = 0;
    int world = 0, unsorted = 0, walked = 0;
    uint64_t keys[2] = {0, 0};
    std::vector<uint64_t> dest_records, dest_bytes;
    double seconds[4] = {0, 0, 0, 0};
};

namespace {
double since(std::chrono::steady_clock::time_point t0) { return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count(); }
}

extern "C" int mmlst_ingest_front_open(int device, const uint8_t* comp, size_t n_comp, size_t n_own_bytes, const uint32_t* ref_len, int32_t n_ref,
                                       int check_crc, void* stream_in, mmlst_ingest_front** out) {
    if ((!comp && n_comp) || !out || n_own_bytes > n_comp || n_ref < 0 || (n_ref && !ref_len)) { mmlst_set_error("mmlst_ingest_front_open: bad argument"); return MMLST_E_ARG; }
    CUDA_TRY(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream_in);
    g_cur_stream = st;
    {
        const int rc = mmlst_de_available(device);
        if (rc != MMLST_OK) { mmlst_set_error("mmlst_ingest_front_open: %s; use mmlst_bam_unpack", mmlst_last_error()); return rc; }
    }
    const auto t0 = std::chrono::steady_clock::now();
    std::unique_ptr<mmlst_ingest_front> F(new mmlst_ingest_front());
    F->device = device; F->st = st; F->n_ref = n_ref; F->n_comp = n_comp;
    ING_TRY(scan_blocks(comp, n_comp, F->blocks, F->usize));
    F->nb = static_cast<uint32_t>(F->blocks.size());
    F->uend = F->usize;
    for (uint32_t b = 0; b < F->nb; ++b) {
        const uint64_t hdr = F->blocks[b].coff;   // payload offset; the block's header starts before it, inside the same range
        if (hdr >= n_own_bytes) { F->uend = F->blocks[b].uoff; break; }
        F->n_own = b + 1;
    }
    ING_TRY(F->d_err.alloc(16 + 32));
    unsigned long long* err = F->d_err.as<unsigned long long>();
    CUDA_TRY(cudaMemsetAsync(err, 0xff, 16, st));
    CUDA_TRY(cudaMemsetAsync(err + 2, 0, 32, st));
    ING_TRY(inflate_blocks(device, st, comp, n_comp, F->blocks, F->usize, check_crc != 0, F->n_own, F->I, err, [] {}));
    ING_TRY(F->d_reflen.alloc(static_cast<size_t>(n_ref) * 4 + 16));
    if (n_ref) CUDA_TRY(cudaMemcpyAsync(F->d_reflen.p, ref_len, static_cast<size_t>(n_ref) * 4, cudaMemcpyHostToDevice, st));
    const size_t nb = F->nb;
    ING_TRY(F->d_start.alloc(nb * 8)); ING_TRY(F->d_exit.alloc(nb * 8)); ING_TRY(F->d_count.alloc(nb * 4 + 4)); ING_TRY(F->d_badw.alloc(nb * 4));
    ING_TRY(F->d_need.alloc(nb * 8)); ING_TRY(F->d_base.alloc(nb * 4 + 4));
    CUDA_TRY(cudaMemcpyAsync(&F->block_err, err, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    F->seconds[0] = since(t0);
    *out = F.release();
    return MMLST_OK;
}

extern "C" int mmlst_ingest_front_walk(mmlst_ingest_front* F, uint64_t entry) {
    if (!F) { mmlst_set_error("mmlst_ingest_front_walk: null argument"); return MMLST_E_ARG; }
    CUDA_TRY(cudaSetDevice(F->device));
    g_cur_stream = F->st;
    cudaStream_t st = F->st;
    const auto t0 = std::chrono::steady_clock::now();
    F->walked = 1; F->need = 0; F->n_rec = 0; F->chain_err = kNoErr;
    if (F->n_own == 0 || (entry != kNoEntry && entry >= F->uend)) {   // no record starts here: the chain passes through
        F->entry = entry; F->exit = entry;
        CUDA_TRY(cudaMemsetAsync(F->d_count.p, 0, 4, st));
        return MMLST_OK;
    }
    const uint32_t n_own = F->n_own;
    const ChainArgs ca{F->I.d_u.as<uint8_t>(), F->usize, F->I.d_uoff.as<uint64_t>(), n_own, entry, F->n_ref, F->d_reflen.as<uint32_t>(),
                       F->d_start.as<uint64_t>(), F->d_exit.as<uint64_t>(), F->d_count.as<uint32_t>(), F->d_badw.as<uint32_t>(), F->uend,
                       F->d_need.as<uint64_t>()};
    uint32_t* d_changed = reinterpret_cast<uint32_t*>(F->d_err.as<unsigned long long>() + 2);
    ING_TRY(run_chain(ca, d_changed, st, &F->repairs));
    std::vector<uint32_t> badw(n_own);
    std::vector<uint64_t> need(n_own);
    uint64_t first_start = 0, last_exit = 0;
    CUDA_TRY(cudaMemcpyAsync(badw.data(), F->d_badw.p, n_own * 4ull, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(need.data(), F->d_need.p, n_own * 8ull, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(&first_start, F->d_start.p, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(&last_exit, F->d_exit.as<uint64_t>() + (n_own - 1), 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    F->entry = entry == kNoEntry ? first_start : entry;
    F->exit = last_exit;
    for (uint32_t b = 0; b < n_own; ++b) {
        if (!badw[b]) continue;
        F->exit = kNoEntry;            // the chain is broken here (a malformed record), unless the halo is only too short
        if (need[b] > F->usize) F->need = need[b];
        break;
    }
    F->seconds[1] += since(t0);
    return MMLST_OK;
}

extern "C" int mmlst_ingest_front_partition(mmlst_ingest_front* F, const int32_t* owner, int world) {
    if (!F || world < 1 || world > kMaxShardRanks || (F->n_ref && !owner)) { mmlst_set_error("mmlst_ingest_front_partition: bad argument (world <= %d)", kMaxShardRanks); return MMLST_E_ARG; }
    if (!F->walked || F->need) { mmlst_set_error("mmlst_ingest_front_partition: the record chain has not been walked to its end"); return MMLST_E_ARG; }
    for (int32_t t = 0; t < F->n_ref; ++t)
        if (owner[t] < 0 || owner[t] >= world) { mmlst_set_error("mmlst_ingest_front_partition: owner[%d] = %d outside [0, %d)", t, owner[t], world); return MMLST_E_ARG; }
    CUDA_TRY(cudaSetDevice(F->device));
    g_cur_stream = F->st;
    cudaStream_t st = F->st;
    const auto t0 = std::chrono::steady_clock::now();
    F->world = world;
    F->dest_records.assign(world, 0); F->dest_bytes.assign(world, 0);
    F->unsorted = 0; F->keys[0] = F->keys[1] = 0; F->n_rec = 0; F->chain_err = kNoErr;
    unsigned long long* err = F->d_err.as<unsigned long long>();
    uint32_t* d_flags = reinterpret_cast<uint32_t*>(err + 2);
    ING_TRY(F->send.alloc(16)); ING_TRY(F->send_len.alloc(16)); ING_TRY(F->send_idx.alloc(16));
    const bool walks = F->n_own && !(F->entry != kNoEntry && F->entry >= F->uend);
    if (!walks) { F->seconds[2] = since(t0); return MMLST_OK; }
    const uint32_t nb = F->n_own;
    const ChainArgs ca{F->I.d_u.as<uint8_t>(), F->usize, F->I.d_uoff.as<uint64_t>(), nb, F->entry, F->n_ref, F->d_reflen.as<uint32_t>(),
                       F->d_start.as<uint64_t>(), F->d_exit.as<uint64_t>(), F->d_count.as<uint32_t>(), F->d_badw.as<uint32_t>(), F->uend, nullptr};
    size_t tb = 0;
    DBuf d_tmp;
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, tb, F->d_count.as<uint32_t>(), F->d_base.as<uint32_t>(), nb + 1, st));
    ING_TRY(d_tmp.alloc(tb));
    CUDA_TRY(cudaMemsetAsync(F->d_count.as<uint32_t>() + nb, 0, 4, st));
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(d_tmp.p, tb, F->d_count.as<uint32_t>(), F->d_base.as<uint32_t>(), nb + 1, st));
    uint32_t n32 = 0;
    CUDA_TRY(cudaMemcpyAsync(&n32, F->d_base.as<uint32_t>() + nb, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemsetAsync(err + 1, 0xff, 8, st));
    CUDA_TRY(cudaMemsetAsync(d_flags, 0, 4, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    const uint64_t n = n32;
    F->n_rec = n;
    ING_TRY(F->d_roff.alloc(n * 8 + 8));
    chain_offsets_kernel<<<(nb + kT - 1) / kT, kT, 0, st>>>(ca, F->d_base.as<uint32_t>(), F->d_roff.as<uint64_t>(), err + 1);
    CUDA_TRY(cudaGetLastError());
    if (n) {
        const unsigned gn = static_cast<unsigned>((n + kT - 1) / kT);
        ING_TRY(F->d_owner.alloc(static_cast<size_t>(F->n_ref) * 4 + 16));
        if (F->n_ref) CUDA_TRY(cudaMemcpyAsync(F->d_owner.p, owner, static_cast<size_t>(F->n_ref) * 4, cudaMemcpyHostToDevice, st));
        ING_TRY(F->d_dest.alloc(n * 4)); ING_TRY(F->d_rlen.alloc(n * 4)); ING_TRY(F->d_dcount.alloc(static_cast<size_t>(world) * 8)); ING_TRY(F->d_keys.alloc(16));
        CUDA_TRY(cudaMemsetAsync(F->d_dcount.p, 0, static_cast<size_t>(world) * 8, st));
        route_kernel<<<gn, kT, 0, st>>>(F->I.d_u.as<uint8_t>(), F->d_roff.as<uint64_t>(), n, F->n_ref, F->d_owner.as<int32_t>(), world, F->d_dest.as<uint32_t>(),
                                        F->d_rlen.as<uint32_t>(), F->d_dcount.as<unsigned long long>(), d_flags, F->d_keys.as<uint64_t>());
        CUDA_TRY(cudaGetLastError());
        // stable partition by destination: LSD radix sort of (dest, shard index) over the bits a rank number needs
        DBuf d_iota, d_dest2;
        ING_TRY(d_iota.alloc(n * 4)); ING_TRY(F->d_order.alloc(n * 4)); ING_TRY(d_dest2.alloc(n * 4));
        iota_kernel<<<gn, kT, 0, st>>>(d_iota.as<uint32_t>(), n);
        CUDA_TRY(cudaGetLastError());
        int end_bit = 1;
        while ((1 << end_bit) < world) ++end_bit;
        size_t sb = 0;
        CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, sb, F->d_dest.as<uint32_t>(), d_dest2.as<uint32_t>(), d_iota.as<uint32_t>(), F->d_order.as<uint32_t>(),
                                                 static_cast<int>(n), 0, end_bit, st));
        DBuf d_stmp;
        ING_TRY(d_stmp.alloc(sb));
        CUDA_TRY(cub::DeviceRadixSort::SortPairs(d_stmp.p, sb, F->d_dest.as<uint32_t>(), d_dest2.as<uint32_t>(), d_iota.as<uint32_t>(), F->d_order.as<uint32_t>(),
                                                 static_cast<int>(n), 0, end_bit, st));
        DBuf d_plen;
        ING_TRY(d_plen.alloc((n + 1) * 8)); ING_TRY(F->d_boff.alloc((n + 1) * 8));
        part_len_kernel<<<static_cast<unsigned>((n + 1 + kT - 1) / kT), kT, 0, st>>>(F->d_order.as<uint32_t>(), F->d_rlen.as<uint32_t>(), n, d_plen.as<uint64_t>());
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, sb, d_plen.as<uint64_t>(), F->d_boff.as<uint64_t>(), static_cast<int>(n + 1), st));
        ING_TRY(d_stmp.alloc(sb));
        CUDA_TRY(cub::DeviceScan::ExclusiveSum(d_stmp.p, sb, d_plen.as<uint64_t>(), F->d_boff.as<uint64_t>(), static_cast<int>(n + 1), st));
        uint64_t total = 0;
        CUDA_TRY(cudaMemcpyAsync(&total, F->d_boff.as<uint64_t>() + n, 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaMemcpyAsync(F->dest_records.data(), F->d_dcount.p, static_cast<size_t>(world) * 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        ING_TRY(F->send.alloc(total + 16)); ING_TRY(F->send_len.alloc(n * 4)); ING_TRY(F->send_idx.alloc(n * 4));
        partition_kernel<<<static_cast<unsigned>((n * 32 + kT - 1) / kT), kT, 0, st>>>(F->I.d_u.as<uint8_t>(), F->d_roff.as<uint64_t>(), F->d_order.as<uint32_t>(),
                                                                                      F->d_rlen.as<uint32_t>(), F->d_boff.as<uint64_t>(), n, F->send.as<uint8_t>(),
                                                                                      F->send_len.as<uint32_t>(), F->send_idx.as<uint32_t>());
        CUDA_TRY(cudaGetLastError());
        // bytes per destination: boff at the first record of every destination
        std::vector<uint64_t> first(world + 1, 0);
        for (int d = 0; d < world; ++d) first[d + 1] = first[d] + F->dest_records[d];
        std::vector<uint64_t> at(world + 1, 0);
        for (int d = 0; d <= world; ++d) CUDA_TRY(cudaMemcpyAsync(&at[d], F->d_boff.as<uint64_t>() + first[d], 8, cudaMemcpyDeviceToHost, st));
        uint32_t fl = 0;
        CUDA_TRY(cudaMemcpyAsync(&fl, d_flags, 4, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaMemcpyAsync(F->keys, F->d_keys.p, 16, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        for (int d = 0; d < world; ++d) F->dest_bytes[d] = at[d + 1] - at[d];
        F->unsorted = fl & 1u;
    }
    CUDA_TRY(cudaMemcpyAsync(&F->chain_err, err + 1, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    F->seconds[2] = since(t0);
    return MMLST_OK;
}

extern "C" int mmlst_ingest_front_info(const mmlst_ingest_front* F, mmlst_ingest_front_info_t* o) {
    if (!F || !o) { mmlst_set_error("mmlst_ingest_front_info: null argument"); return MMLST_E_ARG; }
    memset(o, 0, sizeof(*o));
    o->n_blocks = F->nb; o->n_own_blocks = F->n_own; o->own_inflated = F->uend; o->inflated = F->usize; o->compressed = F->n_comp;
    o->block_error = F->block_err; o->entry = F->entry; o->exit = F->exit; o->need = F->need; o->n_rec = F->n_rec; o->chain_error = F->chain_err;
    o->repairs = F->repairs; o->world = F->world;
    o->send = F->send.as<uint8_t>(); o->send_len = F->send_len.as<uint32_t>(); o->send_idx = F->send_idx.as<uint32_t>();
    o->dest_records = F->dest_records.empty() ? nullptr : F->dest_records.data();
    o->dest_bytes = F->dest_bytes.empty() ? nullptr : F->dest_bytes.data();
    o->unsorted = F->unsorted; o->first_key = F->keys[0]; o->last_key = F->keys[1];
    for (int i = 0; i < 3; ++i) o->seconds[i] = F->seconds[i];
    return MMLST_OK;
}

extern "C" void mmlst_ingest_front_free(mmlst_ingest_front* F) {
    if (!F) return;
    cudaSetDevice(F->device);
    cudaStreamSynchronize(F->st);
    delete F;
}

extern "C" int mmlst_bam_ingest_back(int device, const uint8_t* recs, const uint32_t* rec_len, const uint32_t* file_idx, uint64_t n,
                                     const mmlst_ingest_back_args* a, const mmlst_unpack_opts* opts_in, void* stream_in, mmlst_dev_bam** out,
                                     uint64_t* error_out) {
    if (error_out) *error_out = kNoErr;
    if (!a || !out || (n && (!recs || !rec_len || !file_idx)) || a->n_ref < 0 || (a->n_ref && !a->ref_len)) {
        mmlst_set_error("mmlst_bam_ingest_back: bad argument");
        return MMLST_E_ARG;
    }
    const mmlst_unpack_opts o = ingest_opts(opts_in);
    if (n >= 0x7fffff00ull) { mmlst_set_error("mmlst_bam_ingest_back: more than 2^31-257 records in one call"); return MMLST_E_RANGE; }
    CUDA_TRY(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream_in);
    g_cur_stream = st;
    cudaEvent_t ev[6];
    for (auto& e : ev) CUDA_TRY(cudaEventCreate(&e));
    struct EvGuard { cudaEvent_t* e; ~EvGuard() { for (int i = 0; i < 6; ++i) cudaEventDestroy(e[i]); } } evg{ev};
    int evn = 0;
    auto mark = [&]() { cudaEventRecord(ev[evn++], st); };
    std::unique_ptr<mmlst_dev_bam> B(new mmlst_dev_bam());
    B->device = device;
    B->n_ref = static_cast<uint32_t>(a->n_ref);
    B->ref_len.assign(a->ref_len, a->ref_len + a->n_ref);
    B->names_blob = a->ref_names ? a->ref_names : "";
    B->header_text = a->header_text ? a->header_text : "";
    DBuf d_err, d_reflen, d_roff, d_w;
    ING_TRY(d_err.alloc(8 + 32));
    unsigned long long* err = d_err.as<unsigned long long>();
    uint32_t* d_flags = reinterpret_cast<uint32_t*>(err + 1);
    CUDA_TRY(cudaMemsetAsync(err, 0xff, 8, st));
    CUDA_TRY(cudaMemsetAsync(d_flags, 0, 32, st));
    mark();  // 0
    ING_TRY(d_reflen.alloc(static_cast<size_t>(a->n_ref) * 4 + 16));
    if (a->n_ref) CUDA_TRY(cudaMemcpyAsync(d_reflen.p, a->ref_len, static_cast<size_t>(a->n_ref) * 4, cudaMemcpyHostToDevice, st));
    // record offsets in the received bytes: exclusive prefix of the lengths
    ING_TRY(d_roff.alloc((n + 1) * 8)); ING_TRY(d_w.alloc((n + 1) * 8));
    widen_kernel<<<static_cast<unsigned>((n + 1 + kT - 1) / kT), kT, 0, st>>>(rec_len, n, d_w.as<uint64_t>());
    CUDA_TRY(cudaGetLastError());
    {
        size_t sb = 0;
        CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, sb, d_w.as<uint64_t>(), d_roff.as<uint64_t>(), static_cast<int>(n + 1), st));
        DBuf t;
        ING_TRY(t.alloc(sb));
        CUDA_TRY(cub::DeviceScan::ExclusiveSum(t.p, sb, d_w.as<uint64_t>(), d_roff.as<uint64_t>(), static_cast<int>(n + 1), st));
    }
    const BackIn in{recs, d_roff.as<uint64_t>(), file_idx, n, a->n_ref, d_reflen.as<uint32_t>(), err, d_flags, a->unsorted ? 1 : 0};
    int phase = 0;
    unsigned long long ew = kNoErr;
    const int rc = back_half(in, o, st, B.get(), mark, &phase, &ew);
    if (rc != MMLST_OK) {
        if (error_out && phase) *error_out = (static_cast<uint64_t>(phase) << 56) | (ew == kNoErr ? 0ull : ew);
        return rc;
    }
    B->explicit_idx = 1;   // also for an owner that received no record
    if (!B->orig_idx.p) ING_TRY(B->orig_idx.alloc(4));
    // phase seconds: parse, sort, score stream, cap + compaction, pack (slots 3..7 of the whole-file ingest)
    for (int i = 0; i + 1 < evn && i < 5; ++i) { float ms = 0; cudaEventElapsedTime(&ms, ev[i], ev[i + 1]); B->seconds[3 + i] = ms * 1e-3; }
    *out = B.release();
    return MMLST_OK;
}

// The refusal a shard's ranks agreed on: (phase << 56 | record-or-block << 8 | code), phase 0 = a BGZF block, 1..4 = BackPhase.  Sets
// the text the whole-file ingest gives for it and returns its code.
extern "C" int mmlst_ingest_refusal(uint64_t e) {
    const uint32_t phase = static_cast<uint32_t>(e >> 56), code = static_cast<uint32_t>(e & 0xff);
    const unsigned long long at = (e & ((1ull << 56) - 1)) >> 8;
    switch (phase) {
        case 0:
            if (code == E_CRC) mmlst_set_error("mmlst_bam_ingest: CRC mismatch in BGZF block %llu", at);
            else mmlst_set_error("mmlst_bam_ingest: a BGZF block did not inflate to its ISIZE (corrupt file?)");
            return MMLST_E_BAM;
        case kPhaseRecord: mmlst_set_error("mmlst_bam_ingest: record %llu: %s", at, err_text(code)); return err_class(code);
        case kPhaseUnsorted: mmlst_set_error("%s", kUnsortedText); return MMLST_E_UNSORTED;
        case kPhasePlanes: mmlst_set_error("mmlst_bam_ingest: plane array exceeds 2^32 words"); return MMLST_E_RANGE;
        case kPhasePileup: mmlst_set_error("mmlst_bam_ingest (pileup stream): record %llu: %s", at, err_text(code)); return err_class(code);
        default: mmlst_set_error("mmlst_ingest_refusal: unknown phase %u", phase); return MMLST_E_ARG;
    }
}
