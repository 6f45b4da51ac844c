// Shared helpers for libmmlst (sm_100a only).
#pragma once
#ifdef MMLST_HOST_EMUL
#include "simt_host_emul.h"  // tests/simt: CUDA vocabulary for a host build, one std::thread per lane
#else
#include <cuda_runtime.h>
#endif
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/mmlst.h"

#define MMLST_NUM_SMS_DEFAULT 148
#define MMLST_CHUNKS_PER_SM 2u  // resident CTAs per SM of the bit-sliced pileup kernel ("slots" = SMs x this)

// Tiles (512 records) per pileup chunk for a launch over n_rec records on `slots` resident CTAs.  Every (chunk, column
// word) pair costs one cross-lane flush, so chunks should be long; the static round-robin over slots wants the chunk
// count to be a whole number of waves.  Pick the number of waves k (fewest first) whose chunk length
// ceil(tiles / (k slots)) <= 8 tiles wastes the least of the last wave; short inputs get exactly one wave.
__host__ __device__ inline uint32_t mmlst_chunk_tiles(unsigned long long n_rec, uint32_t slots) {
    const unsigned long long tiles64 = (n_rec + 511ull) / 512ull;
    if (tiles64 == 0 || slots == 0) return 1u;
    if (tiles64 > 0x7fffffffull / 64ull) return 63u;
    const uint32_t tiles = static_cast<uint32_t>(tiles64);  // 32-bit from here on: 64-bit division is a subroutine on the GPU
    uint32_t kmin = (tiles + 8u * slots - 1u) / (8u * slots);  // fewest waves with chunks of <= 8 tiles
    if (kmin == 0) kmin = 1;
    uint32_t best_cr = (tiles + kmin * slots - 1u) / (kmin * slots), best_cost = kmin * best_cr;
    for (uint32_t k = kmin + 1; k < kmin + 12; ++k) {
        const uint32_t cr = (tiles + k * slots - 1u) / (k * slots);
        if (cr < 2u) break;
        if (k * cr < best_cost) { best_cost = k * cr; best_cr = cr; }  // makespan in tiles
    }
    return best_cr > 63u ? 63u : best_cr;
}

#ifndef MMLST_HOST_EMUL
void mmlst_set_error(const char* fmt, ...);
int mmlst_cuda_fail(cudaError_t e, const char* what);

#define CUDA_TRY(expr)                                          \
    do {                                                        \
        cudaError_t _e = (expr);                                \
        if (_e != cudaSuccess) return mmlst_cuda_fail(_e, #expr); \
    } while (0)

int mmlst_num_sms();

// MMLST_OK when the selection launch of mmlst_select_dev for n_loci / n_species fits the current device's shared memory per block (the opt-in
// maximum less the kernel's static part), else MMLST_E_RANGE with a message that names both sizes (`who` = the refusing call)
int mmlst_select_fits(uint32_t n_loci, uint32_t n_species, const char* who);

// MMLST_TRACE=1: host wall-clock marks inside the host-buffer calls, printed to stderr when the call returns (profiles/tools/e2e_trace.py)
void mmlst_trace_mark(const char* label);
void mmlst_trace_flush(const char* call);

// Function attributes (dynamic shared-memory limit, carve-out) and occupancy answers belong to ONE device: caches of "already
// configured" are indexed by the current device, so that a process driving several GPUs (sample.type_cohort) configures each.
constexpr int MMLST_MAX_DEVICES = 64;
inline int mmlst_current_device() {
    int d = 0;
    if (cudaGetDevice(&d) != cudaSuccess || d < 0) d = 0;
    return d % MMLST_MAX_DEVICES;
}

// Every kernel of a pass asks for the SAME L1 / shared-memory split (all of it shared memory): the score and pileup kernels need it, and an SM whose
// split differs from what the next kernel wants has to drain and reconfigure before that kernel's CTAs can start -- between the links of a pass and,
// with several passes in flight on different streams, between kernels that could otherwise share an SM.  MMLST_UNIFORM_CARVEOUT=0 leaves the small
// kernels on the driver's default (profiling aid).  Once per (kernel, device).
int mmlst_uniform_carveout();
template <class K>
inline void mmlst_prefer_max_shared(K kernel, bool (&done)[MMLST_MAX_DEVICES]) {
    bool& d = done[mmlst_current_device()];
    if (d) return;
    d = true;
    if (mmlst_uniform_carveout()) { cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared); cudaGetLastError(); }
}

// Profiling aid (mmlst_debug_timeline): when a device buffer is registered, thread 0 of every CTA of the tail kernels stores %globaltimer (ns) and the
// SM's clock64() at a few marks -- tl[(base + blockIdx.x) * 8 + slot] and the same index + MMLST_TL_WORDS for the cycle counter.  `dep` makes the read
// wait for a value (a load whose arrival the mark is meant to time).  nullptr (the normal state) costs one predicated branch per mark.
constexpr uint32_t MMLST_TL_WORDS = 8192;   // u64 words per half: 1024 CTA rows of 8 marks
constexpr uint32_t MMLST_TL_SELECT = 0, MMLST_TL_PILEUP = 128, MMLST_TL_CONSENSUS = 896;   // first row of each kernel
unsigned long long* mmlst_timeline_buffer();
__device__ __forceinline__ void tl_mark(unsigned long long* tl, uint32_t base, uint32_t slot, uint32_t dep = 0) {
    if (tl && threadIdx.x == 0 && base + blockIdx.x < MMLST_TL_WORDS / 8) {
        unsigned long long t, c;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t) : "r"(dep) : "memory");
        asm volatile("mov.u64 %0, %%clock64;" : "=l"(c) : "r"(dep) : "memory");
        tl[(base + blockIdx.x) * 8 + slot] = t;
        tl[MMLST_TL_WORDS + (base + blockIdx.x) * 8 + slot] = c;
    }
}

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }

// cmseq's majority call of a recorded column (cmseq/cmseq.py:202-209): max(sorted(freq), key=freq.get) is the first maximum in the
// order A, C, G, N, T, and N competes with the bases (H8).  The consensus kernels and the contig statistics share it.
__device__ __forceinline__ uint8_t mmlst_majority_call(uint32_t A, uint32_t C, uint32_t G, uint32_t T, uint32_t N) {
    uint32_t best = A; uint8_t call = 'A';
    if (C > best) { best = C; call = 'C'; }
    if (G > best) { best = G; call = 'G'; }
    if (N > best) { best = N; call = 'N'; }
    if (T > best) { best = T; call = 'T'; }
    return call;
}

// streaming 128-bit load: read once, do not pollute L1
__device__ __forceinline__ uint4 ld_stream_u4(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ uint2 ld_stream_u2(const void* p) {
    uint2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ uint32_t ld_stream_u1(const void* p) {
    uint32_t r;
    asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}

// ---- L2 residency hints (createpolicy + .L2::cache_hint): a stream read once should not push the small tables read by
// every warp (run arrays, allow[]) out of the L2 between launches
__device__ __forceinline__ uint64_t l2_policy(int kind) {  // 0 normal, 1 evict first (streams), 2 evict last (tables)
    uint64_t p;
    if (kind == 1) asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    else if (kind == 2) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    else asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint4 ld_stream_u4_hint(const void* p, uint64_t pol) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ uint2 ld_stream_u2_hint(const void* p, uint64_t pol) {
    uint2 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v2.u32 {%0,%1}, [%2], %3;" : "=r"(r.x), "=r"(r.y) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ uint32_t ld_table_u32(const uint32_t* p, uint64_t pol) {
    uint32_t r;
    asm volatile("ld.global.nc.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ uint32_t ld_table_u16(const uint16_t* p, uint64_t pol) {
    uint16_t r;
    asm volatile("ld.global.nc.L2::cache_hint.u16 %0, [%1], %2;" : "=h"(r) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ uint32_t ld_table_u8(const uint8_t* p, uint64_t pol) {
    uint32_t r;
    asm volatile("ld.global.nc.L2::cache_hint.u8 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(pol));
    return r;
}

// ---- mbarrier + 1-D TMA bulk copy (cp.async.bulk, SASS UBLKCP) into shared memory
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void bulk_g2s_hint(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint64_t pol) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t phase) {
    const uint32_t addr = smem_u32(bar);
    uint32_t done;
    do {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(done)
                     : "r"(addr), "r"(phase)
                     : "memory");
    } while (!done);
}
// ---- programmatic dependent launch (PDL): the kernels of one pass form a chain (score -> select -> pileup -> consensus) whose links are short;
// a dependent kernel launched with the programmatic-serialization attribute becomes resident as soon as every CTA of its predecessor has
// called pdl_launch_dependents() and then blocks in pdl_wait() until the predecessor has COMPLETED (memory visible): the launch latency and
// the ramp of each link run under the previous kernel.  Both are no-ops for a kernel launched the ordinary way.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

int mmlst_pdl_enabled();

template <class... KArgs, class... Args>
inline cudaError_t mmlst_launch_dependent(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = mmlst_pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
#else
inline void pdl_wait() {}
inline void pdl_launch_dependents() {}
#endif  // MMLST_HOST_EMUL
