"""ctypes binding of libmmlst.so (include/mmlst.h).  No fallback: a missing library or device raises."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmmlst.so")


class MmlstError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("libmmlst error %d: %s" % (code, msg))
        self.code = code


E_ARG, E_CUDA, E_IO, E_BAM, E_UNSORTED, E_PAIRED, E_RANGE, E_NOMEM = -1, -2, -3, -4, -5, -6, -7, -8   # include/mmlst.h


class Chunk(C.Structure):
    _fields_ = [("rec_begin", C.c_uint32), ("rec_end", C.c_uint32), ("col_base", C.c_uint32), ("contig_len", C.c_uint32),
                ("plane_delta", C.c_uint32), ("reserved", C.c_uint32 * 3)]


class Soa(C.Structure):
    _fields_ = [("tid", C.c_void_p), ("as0", C.c_void_p), ("xm3", C.c_void_p), ("qlen", C.c_void_p), ("orig_idx", C.c_void_p),
                ("n_rec", C.c_uint64),
                ("p_recs", C.c_void_p),
                ("planes", C.c_void_p), ("n_prec", C.c_uint64), ("n_plane_words", C.c_uint64), ("max_row_words", C.c_uint32),
                ("contig_start", C.c_void_p), ("n_ref", C.c_uint32),
                ("n_runs", C.c_uint32), ("run_tid", C.c_void_p), ("run_start", C.c_void_p), ("chunk_run", C.c_void_p),
                ("chunk_qlen", C.c_void_p), ("z", C.c_void_p), ("zp", C.c_void_p)]


class ZStream(C.Structure):
    _fields_ = [("bytes", C.c_void_p), ("n_bytes", C.c_uint64), ("table", C.c_void_p), ("n_blocks", C.c_uint32), ("as_xm_coeff", C.c_int32)]


class ZPileup(C.Structure):   # mmlst_zpileup
    _fields_ = [("bytes", C.c_void_p), ("n_bytes", C.c_uint64), ("table", C.c_void_p), ("n_blocks", C.c_uint32), ("contig_block", C.c_void_p)]


class ScoreParams(C.Structure):
    _fields_ = [("minscore", C.c_int), ("max_xm", C.c_int), ("min_read_len", C.c_int)]


class Index(C.Structure):   # mmlst_index
    _fields_ = [("locus_of", C.c_void_p), ("allele_num", C.c_void_p), ("n_ref", C.c_uint32),
                ("species_of_locus", C.c_void_p), ("n_loci", C.c_uint32),
                ("genes_in_db", C.c_void_p), ("n_species", C.c_uint32),
                ("db_ascii", C.c_void_p), ("db_off", C.c_void_p), ("bam_ln", C.c_void_p)]


class SampleParams(C.Structure):   # mmlst_sample_params
    _fields_ = [("minscore", C.c_int), ("max_xm", C.c_int), ("min_read_len", C.c_int), ("penalty", C.c_int), ("nloci_pct", C.c_int),
                ("mincov", C.c_uint32), ("pileup_impl", C.c_int)]


class SampleResult(C.Structure):   # mmlst_sample_result
    _fields_ = [("n_chosen", C.c_uint32), ("error_bits", C.c_uint32), ("bad_len_tid", C.c_uint32), ("reserved", C.c_uint32),
                ("total_reads", C.c_uint64), ("ignored_reads", C.c_uint64),
                ("chosen_tid", C.c_void_p), ("chosen_species", C.c_void_p), ("col_off", C.c_void_p),
                ("cons", C.c_void_p), ("cons_capacity", C.c_uint64),
                ("holes", C.c_void_p), ("snps", C.c_void_p),
                ("sum_as", C.c_void_p), ("n_hit", C.c_void_p), ("first_idx", C.c_void_p)]


class ContigStatsParams(C.Structure):   # mmlst_contig_stats_params
    _fields_ = [("mode", C.c_uint32), ("mincov", C.c_uint32), ("trunc", C.c_uint32), ("none_char", C.c_uint32), ("dominant_frq_thrsh", C.c_double)]


class ContigStatsOut(C.Structure):   # mmlst_contig_stats_out
    _fields_ = [("sel_off", C.c_void_p), ("low_off", C.c_void_p), ("depth_off", C.c_void_p), ("out_col", C.c_void_p), ("out_val", C.c_void_p),
                ("cons", C.c_void_p), ("capacity", C.c_uint64), ("n_out", C.c_uint64)]


STATS_COLUMNS, STATS_DEPTH, STATS_LOWDOM = 0, 1, 2   # include/mmlst.h MMLST_STATS_*
CONTIG_STATS_MAX_COLS = 858993459                     # MMLST_CONTIG_STATS_MAX_COLS


_COVERAGE_ARGS = [C.c_void_p] * 6 + [C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                      C.c_uint64, C.c_void_p, C.c_void_p]   # mmlst_coverage_dev and its two passes

EXPORTS = {
    # name: (restype, argtypes)
    "mmlst_last_error": (C.c_char_p, []),
    "mmlst_version": (C.c_int, []),
    "mmlst_device_count": (C.c_int, []),
    "mmlst_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "mmlst_destroy": (None, [C.c_void_p]),
    "mmlst_stream": (C.c_void_p, [C.c_void_p]),
    "mmlst_sync": (C.c_int, [C.c_void_p]),
    "mmlst_pinned_alloc": (C.c_void_p, [C.c_size_t]),
    "mmlst_pinned_free": (None, [C.c_void_p]),
    "mmlst_score_dev": (C.c_int, [C.c_void_p] * 5 + [C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint32,
                                  C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mmlst_build_runs": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint32)]),
    "mmlst_score_runs_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32] + [C.c_void_p] * 5 + [C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint32,
                                       C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mmlst_chunk_qlen": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.POINTER(C.c_int)]),
    "mmlst_score_runs_qc_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32] + [C.c_void_p] * 5 + [C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint32,
                                          C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mmlst_score_pack16_dev": (C.c_int, [C.c_void_p] * 3 + [C.c_uint64] + [C.c_void_p] * 3),
    "mmlst_score_runs16_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32] + [C.c_void_p] * 6 + [C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint32,
                                         C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mmlst_expand_chunk_qlen_dev": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "mmlst_inflate_raw": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]),
    "mmlst_set_score_variant": (C.c_int, [C.c_int]),
    "mmlst_set_score_l2_hints": (C.c_int, [C.c_int]),
    "mmlst_set_score_grid_scale": (C.c_int, [C.c_int]),
    "mmlst_debug_timeline": (C.c_int, [C.c_void_p]),
    "mmlst_set_select_warp_finalize": (C.c_int, [C.c_int]),
    "mmlst_as_untransform_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p]),
    "mmlst_set_pdl": (C.c_int, [C.c_int]),
    "mmlst_expand_runs_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "mmlst_coverage_table_slots": (C.c_uint64, [C.c_uint64]),
    "mmlst_coverage_dev": (C.c_int, _COVERAGE_ARGS),
    "mmlst_coverage_insert_dev": (C.c_int, _COVERAGE_ARGS),
    "mmlst_coverage_sum_dev": (C.c_int, _COVERAGE_ARGS),
    "mmlst_coverage_merge_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p]),
    "mmlst_coverage": (C.c_int, [C.c_void_p, C.POINTER(Soa), C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(ScoreParams),
                                 C.c_uint32, C.c_void_p]),
    "mmlst_pileup_dev": (C.c_int, [C.c_void_p] * 3 + [C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.c_void_p, C.c_uint32,
                                   C.c_int, C.c_void_p]),
    "mmlst_consensus_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p]),
    "mmlst_hamming_min_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]),
    "mmlst_hamming_min_dev2": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                         C.c_void_p, C.c_void_p]),
    "mmlst_select_dev": (C.c_int, [C.c_void_p] * 6 + [C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.c_int,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_size_t] + [C.c_void_p] * 6 +
                         [C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mmlst_pileup_indirect_dev": (C.c_int, [C.c_void_p] * 4 + [C.c_uint32, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "mmlst_consensus_indirect_dev": (C.c_int, [C.c_void_p] * 4 + [C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                                C.c_uint32, C.c_void_p]),
    "mmlst_pileup_consensus_indirect_dev": (C.c_int, [C.c_void_p] * 4 + [C.c_uint32, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                                      C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "mmlst_chunk_records": (C.c_uint32, [C.c_uint64]),
    "mmlst_contig_stats_scratch_bytes": (C.c_size_t, [C.c_uint32]),
    "mmlst_contig_stats_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(ContigStatsParams), C.c_void_p, C.c_size_t]
                               + [C.c_void_p] * 6 + [C.c_uint32, C.c_void_p]),
    "mmlst_contig_stats": (C.c_int, [C.c_void_p, C.POINTER(Soa), C.c_void_p, C.c_uint32, C.c_void_p, C.c_int, C.c_int,
                                     C.POINTER(ContigStatsParams), C.POINTER(ContigStatsOut)]),
    "mmlst_contig_stats_resident": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32,
                                              C.c_void_p, C.c_int, C.c_int, C.POINTER(ContigStatsParams), C.POINTER(ContigStatsOut)]),
    "mmlst_xchg_publish_dev": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint64, C.c_uint64,
                                         C.c_void_p, C.c_void_p]),
    "mmlst_xchg_await_dev": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p]),
    "mmlst_depth_cap": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p]),
    "mmlst_score": (C.c_int, [C.c_void_p, C.POINTER(Soa), C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(ScoreParams),
                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mmlst_pileup_consensus": (C.c_int, [C.c_void_p, C.POINTER(Soa), C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_int,
                                         C.c_int, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mmlst_db_upload": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32]),
    "mmlst_db_upload_x": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_uint32]),
    "mmlst_hamming_min_x": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "mmlst_hamming_exact_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "mmlst_exact_match_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                        C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p,
                                        C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "mmlst_db_row_keys": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32]),
    "mmlst_exact_match": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p,
                                    C.c_uint32, C.c_void_p]),
    "mmlst_st_match_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]),
    "mmlst_profiles_upload": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32]),
    "mmlst_st_match": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32]),
    "mmlst_bam_unpack": (C.c_int, [C.c_char_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "mmlst_bam_info": (C.c_int, [C.c_void_p, C.c_void_p]),
    "mmlst_bam_free": (None, [C.c_void_p]),
    "mmlst_hamming_min": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32,
                                    C.c_void_p, C.c_void_p]),
    "mmlst_hamming_tc_image_bytes": (C.c_size_t, [C.c_uint32, C.c_uint32, C.c_uint32]),
    "mmlst_hamming_tc_expand_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mmlst_hamming_tc_search_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32,
                                              C.c_uint32, C.c_void_p, C.c_void_p]),
    "mmlst_ingest_trim": (C.c_int, [C.c_int]),
    "mmlst_comm_unique_id": (C.c_int, [C.c_void_p]),
    "mmlst_comm_create": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "mmlst_comm_destroy": (None, [C.c_void_p]),
    "mmlst_allreduce": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]),
    "mmlst_bam_ingest": (C.c_int, [C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "mmlst_dev_bam_info": (C.c_int, [C.c_void_p, C.c_void_p]),
    "mmlst_dev_bam_free": (None, [C.c_void_p]),
    "mmlst_ingest_front_open": (C.c_int, [C.c_int, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_int32, C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]),
    "mmlst_ingest_front_walk": (C.c_int, [C.c_void_p, C.c_uint64]),
    "mmlst_ingest_front_partition": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "mmlst_ingest_front_info": (C.c_int, [C.c_void_p, C.c_void_p]),
    "mmlst_ingest_front_free": (None, [C.c_void_p]),
    "mmlst_bam_ingest_back": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]),
    "mmlst_ingest_refusal": (C.c_int, [C.c_uint64]),
    "mmlst_index_upload": (C.c_int, [C.c_void_p, C.c_void_p]),
    "mmlst_sample": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
}

_lib = None
SELECT_CONSUME, SELECT_SCRATCH_CLEAN, SELECT_LOCAL, CONSENSUS_CONSUME, COVERAGE_STREAM_RESIDENT = 1, 2, 4, 1, 1  # include/mmlst.h flags


def lib() -> C.CDLL:
    """Load libmmlst.so (built in-tree by metamlst_b200/csrc/build.sh or __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(metamlst_b200 has no CPU fallback)" % LIB_PATH)
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in EXPORTS.items():
            f = getattr(l, name)  # AttributeError if the symbol is not exported
            f.restype = res
            f.argtypes = args
        _lib = l
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        raise MmlstError(rc, lib().mmlst_last_error().decode(errors="replace"))


def ptr(x) -> int:
    """Address of a numpy array / torch tensor / None."""
    if x is None:
        return 0
    if hasattr(x, "data_ptr"):
        return x.data_ptr()
    return x.ctypes.data


class Context:
    """mmlst_ctx: one per GPU; owns a stream and the staging device memory of the host-buffer entry points."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        check(lib().mmlst_create(device, C.byref(self._h)))
        self.device = device

    @property
    def handle(self):
        return self._h

    def close(self):
        if self._h:
            lib().mmlst_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
