// Host build of form 7 of the run-length score kernel and of the pack kernel that defines its compact stream
// (metamlst_b200/csrc/score_runs_kernels.cuh) on the emulation of simt_host_emul.h.  TEST INFRASTRUCTURE ONLY.
#include "simt_score.cpp"

// code[] / head[] of the compact stream from (as0, xm3, chunk_qlen); `grid` CTAs of 256 threads, one warp per chunk (grid-stride)
extern "C" int simt_pack16(unsigned grid, const int16_t* as0, const uint8_t* xm3, const uint16_t* chunk_qlen, uint64_t n_rec, uint16_t* code,
                           uint32_t* head) {
    RunArgs a{};
    launch([&](const RunArgs&) { score_pack16_kernel(as0, xm3, chunk_qlen, n_rec, code, head); }, grid, 256, a);
    return 0;
}

// what mmlst_score_runs16_dev launches under form 7: the compact kernel, or form 6 when max_xm does not fit the 4-bit XM field
extern "C" int simt_score16(unsigned grid, const uint32_t* run_tid, const uint32_t* run_start, uint32_t n_runs, const uint32_t* chunk_run,
                            const uint16_t* chunk_qlen, const int16_t* as0, const uint8_t* xm3, const uint16_t* code, const uint32_t* head,
                            uint64_t n_rec, uint64_t idx_base, const uint8_t* allow, uint32_t n_ref, int minscore, int max_xm, int min_read_len,
                            int64_t* sum_as, uint32_t* n_hit, uint32_t* first_idx, uint64_t* counters) {
    RunArgs a{run_tid, run_start, chunk_run, n_runs, as0, xm3, nullptr, nullptr, chunk_qlen, n_rec, idx_base, allow, n_ref, minscore, max_xm,
              min_read_len, reinterpret_cast<long long*>(sum_as), n_hit, first_idx, reinterpret_cast<unsigned long long*>(counters), 1, code, head};
    launch(max_xm >= 15 ? score_runs_ring_pair_kernel : score_runs_ring_pair16_kernel, grid, kThreads, a);
    return 0;
}
