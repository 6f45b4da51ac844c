/*
 * libmmlst -- B200-native (sm_100a) kernels for MetaMLST's post-alignment allele-calling hot path.
 *
 * C ABI: plain pointers and sizes only.  The reference (SegataLab/metamlst, pure Python) has no FFI of its own;
 * each entry point below names the reference lines it replaces (paths relative to the reference root) and
 * INTEGRATION.md shows the ctypes binding a maintainer adds at the four Python seams (SURVEY.md 8b).
 *
 * Conventions
 *   - every call returns 0 on success or a negative MMLST_E_* code; mmlst_last_error() gives the thread-local text;
 *   - "*_dev" entry points take DEVICE pointers and a cudaStream_t (as void*), launch asynchronously and own nothing;
 *   - the other entry points take HOST pointers (pinned memory from mmlst_pinned_alloc gives async copies), stage
 *     through device memory owned by the mmlst_ctx and return after the results are back on the host;
 *   - there is no CPU fallback: without a CUDA device every compute call fails with MMLST_E_CUDA.
 *
 * Record streams (structure-of-arrays, produced once per BAM by mmlst_bam_unpack or metamlst_b200.packing)
 *   score stream   : every BAM record, any order (coordinate-sorted gives run-length aggregation):
 *                      tid u32 (BAM reference index == allele row), as0 i16 (1st aux field by POSITION),
 *                      xm3 u8 (4th aux field by POSITION, saturated at 255), qlen u16 (len(SEQ) as SAM prints it),
 *                      optional orig_idx u32 (index in file order; NULL = identity + idx_base).        9 B / record
 *                    run-length form (coordinate-sorted streams): tid per RUN of equal tid instead of per record
 *                      (run_tid, run_start, chunk_run -- see mmlst_score_runs_dev).                      5 B / record
 *   pileup stream  : records ADMITTED by the htslib depth cap, coordinate-sorted, CIGAR already projected on the
 *                    reference: one 16-byte mmlst_prec per record {pos i32, row_off u32 (word offset into planes),
 *                    reflen u16, as_named i16, xm_named u8 (AS, XM by NAME), nw u16} -- array-of-16-byte-structs so
 *                    that the metadata of a 512-record tile is ONE contiguous 8 KB bulk copy -- and per record a row
 *                    of 3 bit-planes x nw words, ALIGNED TO THE CONTIG'S 32-COLUMN WORDS: nw = number of words the
 *                    record touches = ((pos & 31) + reflen + 31) >> 5 (0 when reflen == 0); word-interleaved
 *                    [V_j, B1_j, B0_j], bit i of word j = contig column 32 ((pos >> 5) + j) + i:
 *                    V=1 -> ACGT base with quality >= minqual and code B1B0 (A=0,C=1,G=2,T=3);
 *                    V=0,B0=1 -> counted non-ACGT base (bin N); V=0,B0=0 -> not in the column (deletion, refskip,
 *                    quality < minqual, outside the read).  Rows are padded to an odd number of words (bank-conflict-
 *                    free stride in shared memory).  Aligning at unpack time removes every shift from the kernel.
 *   count tensor   : u32 [total_columns][5], bins A,C,G,T,N.
 */
#ifndef MMLST_H
#define MMLST_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MMLST_VERSION 200

enum {
    MMLST_OK = 0,
    MMLST_E_ARG = -1,        /* bad argument */
    MMLST_E_CUDA = -2,       /* CUDA runtime error / no device */
    MMLST_E_IO = -3,         /* file cannot be read */
    MMLST_E_BAM = -4,        /* malformed BAM / aux fields the reference would crash on (metamlst.py:107-110) */
    MMLST_E_UNSORTED = -5,   /* pileup needs coordinate order (htslib "The input is not sorted") */
    MMLST_E_PAIRED = -6,     /* BAM_FPROPER_PAIR record: htslib overlap handling (H2) refused, never silently differs */
    MMLST_E_RANGE = -7,      /* value does not fit the packed field (AS outside int16, reflen > 65535, ...) */
    MMLST_E_NOMEM = -8
};

typedef struct mmlst_ctx mmlst_ctx;

const char* mmlst_last_error(void);
int mmlst_version(void);
int mmlst_device_count(void);

int mmlst_create(int device, mmlst_ctx** out);
void mmlst_destroy(mmlst_ctx* ctx);
/* stream owned by the context (cudaStream_t) */
void* mmlst_stream(mmlst_ctx* ctx);
int mmlst_sync(mmlst_ctx* ctx);

void* mmlst_pinned_alloc(size_t bytes);
void mmlst_pinned_free(void* p);

/* ---------------------------------------------------------------------------------------------------------------
 * Stage 1 -- per-allele scoring.  Replaces metamlst.py:101-130 (filter + append) and the integer half of :133-151
 * (sum, hit count).  Per-locus max hit count, penalty, division and round(.,1) stay on the host (H6).
 *   allow[tid]    : 1 if the record's species passes --filter (metamlst.py:114), else the record is not counted at all
 *   locus_of[tid] : global locus index of the allele row
 *   sum_as[tid] += as0, n_hit[tid] += 1 for records with as0 >= minscore && qlen >= min_read_len && xm3 <= max_xm
 *   first_idx[tid] = min(orig index) over the allele's passing records (H5: dict insertion order of species, loci
 *                    and alleles all follow from it); caller presets 0xFFFFFFFF
 *   counters[0] += allowed records (totalReads), counters[1] += allowed but failing (ignoredReads)
 * Outputs are ACCUMULATED (caller zeroes them), so shards / GPUs can be summed (SURVEY.md 8e).
 * --------------------------------------------------------------------------------------------------------------- */
int mmlst_score_dev(const uint32_t* tid, const int16_t* as0, const uint8_t* xm3, const uint16_t* qlen,
                    const uint32_t* orig_idx, uint64_t n_rec, uint64_t idx_base,
                    const uint8_t* allow, const uint32_t* locus_of, uint32_t n_ref,
                    int minscore, int max_xm, int min_read_len,
                    int64_t* sum_as, uint32_t* n_hit, uint32_t* first_idx, uint64_t* counters, void* stream);

/* The same stage over the RUN-LENGTH form of the score stream (what a coordinate-sorted BAM is shipped in: 5 B / record).
 * The allele id is stored per RUN of equal tid, not per record:
 *   run_tid[n_runs], run_start[n_runs+1] (run r = records run_start[r] .. run_start[r+1]; run_start[0] = 0,
 *   run_start[n_runs] = n_rec; no empty runs), chunk_run[ceil(n_rec/256)] = run holding record 256*c.
 * Any record order is legal (a run is just a maximal stretch of equal tid); it pays off when n_runs << n_rec.
 * n_rec < 2^32 - 256.  Same filter, outputs and accumulation rules as mmlst_score_dev (locus_of is not needed).
 * mmlst_build_runs (HOST) derives the three arrays from tid[]: pass run_tid = NULL to get the counts only
 * (*n_runs = runs, return value OK); capacity of run_tid / run_start is *n_runs on entry. */
int mmlst_build_runs(const uint32_t* tid, uint64_t n_rec, uint32_t* run_tid, uint32_t* run_start, uint32_t* chunk_run,
                     uint32_t* n_runs);
int mmlst_score_runs_dev(const uint32_t* run_tid, const uint32_t* run_start, uint32_t n_runs, const uint32_t* chunk_run,
                         const int16_t* as0, const uint8_t* xm3, const uint16_t* qlen, const uint32_t* orig_idx,
                         uint64_t n_rec, uint64_t idx_base, const uint8_t* allow, uint32_t n_ref,
                         int minscore, int max_xm, int min_read_len,
                         int64_t* sum_as, uint32_t* n_hit, uint32_t* first_idx, uint64_t* counters, void* stream);
/* Run-length form with len(SEQ) stored once per 256-record chunk ("QC": 3 B / record): chunk_qlen[ceil(n_rec/256)] =
 * len(SEQ) shared by every record of the chunk.  Legal only when every chunk is uniform (untrimmed reads of one
 * sequencing run); mmlst_chunk_qlen (HOST) builds the array and returns MMLST_OK with *uniform = 0 when it is not.
 * Same filter, outputs and accumulation rules as mmlst_score_dev. */
int mmlst_chunk_qlen(const uint16_t* qlen, uint64_t n_rec, uint16_t* chunk_qlen, int* uniform);
int mmlst_score_runs_qc_dev(const uint32_t* run_tid, const uint32_t* run_start, uint32_t n_runs, const uint32_t* chunk_run,
                            const uint16_t* chunk_qlen, const int16_t* as0, const uint8_t* xm3, const uint32_t* orig_idx,
                            uint64_t n_rec, uint64_t idx_base, const uint8_t* allow, uint32_t n_ref,
                            int minscore, int max_xm, int min_read_len,
                            int64_t* sum_as, uint32_t* n_hit, uint32_t* first_idx, uint64_t* counters, void* stream);
/* Kernel form used by mmlst_score_runs_dev / mmlst_score_runs_qc_dev (identical results): 0 = register-staged, 1 = register-
 * staged and software-pipelined, 2 = per-warp shared-memory ring filled by TMA bulk copies (records without orig_idx only;
 * other inputs take form 0), 3..5 = the ring with other stage sizes / depths (4 chunks x 3 stages, 8 x 2, 4 x 2),
 * 6 = form 5 with pairs of chunks reduced together (per-chunk len(SEQ) streams; others take form 5): the default since
 * round 2 (B200, configs[1]: 26.7 us against 28.8 us for form 5, profiles/r2a_bench_auto.json).  Returns the previous value; a value outside 0..6 only queries.  The environment variable
 * MMLST_SCORE_VARIANT presets it. */
#define MMLST_SCORE_VARIANT_DEFAULT 6
int mmlst_set_score_variant(int variant);
/* Ring forms only: L2 residency hints (score stream evict-first; forms 2..5 also read run arrays, allow[] and chunk_qlen[] evict-last).  The stream
 * is read once per pass, so marking it evict-first leaves the L2 to what the REST of the pass reads -- the selection tables, the chosen contigs'
 * pileup records, the kernels' code.  The score kernel itself runs as fast either way (27.1 against 27.6 us); serial passes alternating between two
 * samples go from 73.9 to 64.6 us because each sample's tail inputs survive the other sample's 121 MB stream (B200, profiles/r3j_hints{0,1}_l1.json);
 * on since then.  1 = on, 0 = off, other = query; returns the previous value.  MMLST_SCORE_L2_HINTS presets it.  Results do not depend on it. */
#define MMLST_SCORE_L2_HINTS_DEFAULT 1
int mmlst_set_score_l2_hints(int on);
/* Form 6 only: grid size in eighths of one resident wave (8 = exactly one wave; above 8 the surplus CTAs go to whichever SM frees a slot
 * first, i.e. the hardware balances the tail of the launch).  1..64 sets, other = query; returns the previous value.  MMLST_SCORE_GRID presets
 * it.  Results do not depend on it. */
/* Profiling aid: register a DEVICE buffer of 2 x 8192 u64 (or NULL to switch it off, the normal state).  While registered, thread 0 of every CTA of the
 * selection, bit-sliced pileup and consensus kernels stores the global timer (ns; first half) and its SM's cycle counter (second half) at a few marks:
 * word (row * 8 + mark), rows 0.. = selection CTAs, 128.. = pileup CTAs, 896.. = consensus CTAs (profiles/tools/tail_timeline.py reads it).  Applies to
 * launches made after the call (a captured CUDA graph keeps what was set at capture).  Results do not depend on it. */
int mmlst_debug_timeline(uint64_t* dev_buf);
#define MMLST_SCORE_GRID_DEFAULT 8
int mmlst_set_score_grid_scale(int eighths);
/* as0[i] -= coeff * xm3[i] for i < n (device, in place): undoes the decorrelation of a compressed score stream (mmlst_zstream.as_xm_coeff) */
int mmlst_as_untransform_dev(int16_t* as0, const uint8_t* xm3, uint64_t n, int coeff, void* stream);
/* qlen[i] of every record back from the per-chunk form (device; the coverage kernel takes it per record) */
int mmlst_expand_chunk_qlen_dev(const uint16_t* chunk_qlen, uint64_t n_rec, uint16_t* qlen, void* stream);
/* tid[i] of every record back from the run arrays (device; the coverage kernel takes the explicit form) */
int mmlst_expand_runs_dev(const uint32_t* run_tid, const uint32_t* run_start, uint32_t n_runs, const uint32_t* chunk_run,
                          uint64_t n_rec, uint32_t* tid, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Stage 1, coverage column (H7).  Replaces `sequenceBank[species_gene][readCode] = len(sequence)` (metamlst.py:127) and
 * `sum(sequenceBank[key].values())` (metamlst.py:228): per locus the sum over UNIQUE read names of len(SEQ) of the LAST
 * passing record (file order) carrying the name.
 *   qhash[n_rec][2] : 128-bit QNAME hash per score-stream record (two independent 64-bit hashes, mmlst_bam_unpack);
 *                     two names are merged only if both halves collide: P(any false merge) < n^2 / 2^129
 *   table           : device scratch of 24 * table_slots bytes, 16-byte aligned, ZEROED by the caller;
 *                     table_slots = mmlst_coverage_table_slots(upper bound on passing records), a power of two
 *   cov[n_loci]     : ACCUMULATED (caller zeroes); shards that hold whole loci (contig-aligned, SURVEY.md 8e) add up
 * Same filter as mmlst_score_dev (allow, minscore, max_xm, min_read_len).
 * --------------------------------------------------------------------------------------------------------------- */
uint64_t mmlst_coverage_table_slots(uint64_t n_names_upper_bound);
int mmlst_coverage_dev(const uint32_t* tid, const int16_t* as0, const uint8_t* xm3, const uint16_t* qlen,
                       const uint32_t* orig_idx, const uint64_t* qhash, uint64_t n_rec, uint64_t idx_base,
                       const uint8_t* allow, const uint32_t* locus_of, uint32_t n_ref, int minscore, int max_xm,
                       int min_read_len, void* table, uint64_t table_slots, uint64_t* cov, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Stage 2 -- pileup base counts.  Replaces cmseq/cmseq.py:527-548 (+ htslib pileup rules H1-H3 applied at unpack).
 *   chunks[c]: a run of consecutive pileup-stream records of ONE chosen contig, of any length (the library's own rule,
 *   mmlst_chunk_records, gives <= 63 tiles of 512 records); its columns live at
 *   counts[col_base .. col_base+contig_len); plane_delta is added (mod 2^32) to row_off of its records so that a
 *   caller may upload only the chosen contigs' plane ranges.  A base counts as its letter when V=1 and the record
 *   passes as_named >= minscore && xm_named <= max_xm (metaMLST_functions.py:259), else as N.
 *   counts are ACCUMULATED (caller zeroes).  impl: 0 = best available, 1 = per-base atomics (v1), 2 = bit-sliced
 *   carry-save counters (v2).  max_row_words = largest row (3*nw, padded odd) in the stream.
 * --------------------------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t pos;        /* 0-based leftmost reference position */
    uint32_t row_off;   /* word offset of the record's plane row */
    uint16_t reflen;    /* reference span */
    int16_t as_named;   /* AS:i by NAME (cmseq tag filter, metaMLST_functions.py:259) */
    uint8_t xm_named;   /* XM:i by NAME, saturated at 255 */
    uint8_t pad;
    uint16_t nw;        /* 32-column contig words touched by the record = plane words per plane in its row */
} mmlst_prec;

typedef struct {
    uint32_t rec_begin, rec_end;   /* pileup-stream record range */
    uint32_t col_base, contig_len; /* column range in the count tensor */
    uint32_t plane_delta;          /* added to row_off[] */
    uint32_t reserved[3];          /* chunk lists of mmlst_select_dev: [0] = chosen locus (output order) of the chunk, [1] = chunks of that locus */
} mmlst_chunk;

/* records per chunk that fills the chip for a launch over n_rec records (multiple of 512, <= 63*512) */
uint32_t mmlst_chunk_records(uint64_t n_rec);

int mmlst_pileup_dev(const mmlst_prec* recs, const uint32_t* planes,
                     const mmlst_chunk* chunks, uint32_t n_chunks, uint32_t max_row_words,
                     int minscore, int max_xm, uint32_t* counts, uint32_t total_cols, int impl, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * H1 -- htslib pileup depth cap (pysam `pileup(max_depth=8000)` default reaches cmseq/cmseq.py:527 unchanged).
 * HOST function, sequential per contig: records coordinate-sorted (tid, pos), unmapped ones already removed.
 * bam_plp_push drops a record when its start equals the iterator's current column and the mempool holds more than
 * maxcnt nodes; the first record of every start position is pushed while the iterator is still behind it and is
 * always kept, so per start position B the first min(n_B, max(1, maxcnt - live(B) - sentinel_nodes + 1)) records are
 * admitted, live(B) = admitted records with start < B and end >= B.  sentinel_nodes = 1 (htslib >= 1.10).
 * --------------------------------------------------------------------------------------------------------------- */
int mmlst_depth_cap(const uint32_t* tid, const int32_t* pos, const uint32_t* reflen, uint64_t n, uint32_t maxcnt,
                    uint32_t sentinel_nodes, uint8_t* admitted);

/* ---------------------------------------------------------------------------------------------------------------
 * Stage 2b -- consensus call + comparison with the chosen DB allele.  Replaces cmseq/cmseq.py:551-554 (column
 * recorded iff A+C+G+T >= mincov), :202-209 (majority, ties A>C>G>N>T, N competes: H8), :234-237 (fill with 'N')
 * and metaMLST_functions.py:260-276 (N -> lower-case DB base + hole; mismatch -> SNP).
 *   col_off[n_loci+1] : column range of each chosen locus in counts / dbseq / cons
 *   dbseq             : ASCII DB sequence of the chosen allele per column (host checks len >= BAM LN, H10)
 * --------------------------------------------------------------------------------------------------------------- */
int mmlst_consensus_dev(const uint32_t* counts, const uint8_t* dbseq, const uint32_t* col_off, uint32_t n_loci,
                        uint32_t mincov, uint8_t* cons, uint32_t* holes, uint32_t* snps, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * cmseq contig statistics over a BATCH of contigs (metamlst_b200/cmseq_api.py, the BamFile *_all methods).  Replaces the column
 * loops of cmseq/cmseq.py:507-569 (get_base_stats: column recorded iff A+C+G+T >= min_read_depth; binomial test only where
 * max/sum < dominant_frq_thrsh), :226-241 (reference_free_consensus), :430-456 (polymorphism_rate) and :459-490
 * (breadth_and_depth_of_coverage: window [trunc, len - trunc) when len > 2 trunc).  The ratios, p-values and distributions stay on
 * the host, computed from what this returns.
 *   counts[total_cols][5], col_off[n+1] (col_off[0] = 0, ascending; contigs of length 0 allowed): the batch's count tensor
 *   selected column    : inside the contig's window and A+C+G+T >= mincov
 *   low-dominance      : selected and (double)max(A,C,G,T) / (double)(A+C+G+T) < dominant_frq_thrsh (IEEE division, strict <)
 *   sel_off / low_off / depth_off [n+1]: prefix over the batch's contigs of the number of selected columns, of low-dominance
 *                        columns and of the sum of A+C+G+T over selected columns (contig i: [i+1] - [i])
 *   compacted columns  : ascending column inside a contig, contigs in batch order (positions from scans, never from atomics);
 *                        out_col = column inside the contig (0-based), out_val = `width` u32 per column:
 *                        MMLST_STATS_COLUMNS every selected column, width 5 (A, C, G, T, N)       -- get_base_stats
 *                        MMLST_STATS_DEPTH   every selected column, width 1 (A+C+G+T)            -- breadth_and_depth_of_coverage
 *                        MMLST_STATS_LOWDOM  low-dominance columns, width 2 (max, A+C+G+T)       -- polymorphism_rate, consensus
 *                        capacity: sel_off[n] (low_off[n] for LOWDOM) <= total_cols entries
 *   cons[total_cols] (or NULL): the majority call (first maximum in the order A, C, G, N, T, H8: the column rule of the consensus
 *                        kernel) of every selected column, none_char elsewhere
 *   scratch            : mmlst_contig_stats_scratch_bytes(total_cols) bytes, 16-byte aligned
 *   flags              : MMLST_CONSENSUS_CONSUME = zero the counts it read (the next batch accumulates from zero, no memset)
 * Range: total_cols <= MMLST_CONTIG_STATS_MAX_COLS (the kernels index counts and out_val with 5 * column in 32 bits), else
 * MMLST_E_RANGE before any launch.  Three launches (tile sums, one-CTA scan, emit); 20 B / column in.
 * --------------------------------------------------------------------------------------------------------------- */
#define MMLST_STATS_COLUMNS 0u
#define MMLST_STATS_DEPTH 1u
#define MMLST_STATS_LOWDOM 2u
#define MMLST_CONTIG_STATS_MAX_COLS 858993459u   /* floor((2^32 - 1) / 5) */
typedef struct {
    uint32_t mode;               /* MMLST_STATS_* */
    uint32_t mincov;             /* >= 1 */
    uint32_t trunc;              /* 0 = whole contig */
    uint32_t none_char;          /* byte of unselected columns in cons, 0..255 */
    double dominant_frq_thrsh;
} mmlst_contig_stats_params;
size_t mmlst_contig_stats_scratch_bytes(uint32_t total_cols);
int mmlst_contig_stats_dev(uint32_t* counts, const uint32_t* col_off, uint32_t n, uint32_t total_cols, const mmlst_contig_stats_params* prm,
                           void* scratch, size_t scratch_bytes, uint32_t* sel_off, uint32_t* low_off, uint64_t* depth_off,
                           uint32_t* out_col, uint32_t* out_val, uint8_t* cons, uint32_t flags, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Best-allele selection on the device: no host round trip between stage 1 and stage 2.  Replaces metamlst.py:133-151
 * (maxLen, penalty, round(avg,1) -- computed exactly as integer tenths from the IEEE double quotient, H6), :184-206
 * (--nloci gate), :213-220 + :244 (alleles whose rounded average equals the locus maximum, lowest int(allele)), and the
 * dict-order bookkeeping of H5 (species by first passing record, loci inside a species by first passing record).
 * ONE launch: CTA = locus (three in-CTA reductions, no global atomics), the last CTA to finish finalizes.
 *   locus_rows[n_ref] = allele rows grouped by locus, locus_start[n_loci+1] = range of each locus in locus_rows; locus_rows may be NULL when the rows
 *   already ARE grouped by locus (locus_rows[i] == i: a DB dumped gene by gene), which saves the kernel one dependent trip to memory
 *   allele_num[tid] = int(alleleVariant); species_of_locus[locus]; genes_in_db[species] = rows of `genes` (metamlst.py:184)
 *   contig_start / ref_len / db_off: pileup-stream record range, BAM LN and DB-sequence offset of every allele row
 *   scratch: >= 12*n_loci + 16 bytes, 8-byte aligned.  flags: MMLST_SELECT_CONSUME = the call resets what it has read
 *   (sum_as / n_hit / first_idx of every hit row, counters) so the next pass needs no memset of the score tables;
 *   MMLST_SELECT_SCRATCH_CLEAN = the caller zeroed the scratch once and every call since ran to completion (the
 *   call leaves its ticket at zero; the per-locus results before it are scratch), so the 4-byte ticket memset is skipped.
 *   Outputs: header[0]=n_chosen [1]=n_chunks [2]=total columns [3]=error bits (1: "Database is broken", 2: chunk list
 *   overflow) [4]=records per chunk [6,7]=counters[0] (totalReads) [8,9]=counters[1] (ignoredReads) when `counters` is
 *   given; chosen_tid / chosen_species / col_off / db_start per chosen locus in output order; chunks for
 *   mmlst_pileup_indirect_dev.  header needs 16 words.
 *   Range: n_loci <= 8192, n_species <= 4096, and the finalizing CTA keeps 4 (11 n_loci + 1 + 4 n_species) + 16 bytes in shared memory, which
 *   must fit the current device's opt-in maximum per block (cudaDevAttrMaxSharedMemoryPerBlockOptin, about 227 KB on sm_100, less the kernel's
 *   static shared memory): about 5000 loci at 7 loci per species, 3800 at 4096 species.  An index past either bound is refused with
 *   MMLST_E_RANGE before any launch, and the message names both sizes; mmlst_index_upload applies the same check.
 * --------------------------------------------------------------------------------------------------------------- */
/* Finalization of the selection (gate, dict order, column layout, chunk list) by ONE warp with shuffles instead of the whole last CTA with barriers, when
 * n_loci <= 32 and n_species <= 32 (larger index sets always take the CTA-wide form).  1 = on, 0 = off, other = query; returns the previous value;
 * MMLST_SELECT_WARP presets it.  Results do not depend on it (tests/test_gpu_parity.py runs the selection tests under both).  B200, configs[1]: selection
 * 9.0 us with it, 9.9 us without (profiles/r4b_tail_timeline_warp.json); off by default. */
#define MMLST_SELECT_WARP_DEFAULT 0
int mmlst_set_select_warp_finalize(int on);
#define MMLST_SELECT_CONSUME 1u
#define MMLST_SELECT_SCRATCH_CLEAN 2u
#define MMLST_SELECT_LOCAL 4u  /* this GPU owns a SUBSET of the loci (contig-aligned shard): no --nloci gate here; the caller
                                  merges the per-GPU results (chosen_first gives the H5 order keys) and applies the gate */
int mmlst_select_dev(int64_t* sum_as, uint32_t* n_hit, uint32_t* first_idx, const uint32_t* locus_rows, const uint32_t* locus_start,
                     const uint32_t* allele_num, uint32_t n_ref, const uint32_t* species_of_locus, const uint32_t* genes_in_db,
                     uint32_t n_loci, uint32_t n_species, int penalty, int nloci_pct, const uint64_t* contig_start,
                     const uint32_t* ref_len, const uint64_t* db_off, uint32_t chunk_records, void* scratch, size_t scratch_bytes,
                     uint32_t* header, uint32_t* chosen_tid, uint32_t* chosen_species, uint32_t* col_off, uint64_t* db_start,
                     mmlst_chunk* chunks, uint32_t max_chunks, uint32_t flags, uint64_t* counters,
                     uint32_t* chosen_first /* [n_loci] first passing record per chosen locus, or NULL */, void* stream);
/* The device-driven kernels of a pass (mmlst_select_dev, mmlst_pileup_indirect_dev, mmlst_consensus_indirect_dev) are launched with programmatic
 * stream serialization: each becomes resident while its predecessor still runs and waits (griddepcontrol.wait) for it to complete before touching
 * its data.  1 = on, 0 = off (default), other = query; returns the previous value; MMLST_PDL=1 presets it.  Results do not depend on it.
 * Measured on B200 (profiles/r2l_bench_pdl{0,1}.json): inside the CUDA-graph replay a pass is timed in, the links already follow each other within
 * about a microsecond and PDL changes nothing (serial pass 75.4 us with, 74.8 us without), so it is off unless asked for (eager launches gain). */
int mmlst_set_pdl(int on);
int mmlst_pileup_indirect_dev(const mmlst_prec* recs, const uint32_t* planes, const mmlst_chunk* chunks, const uint32_t* header,
                              uint32_t max_row_words, int minscore, int max_xm, uint32_t* counts, int impl, void* stream);
/* mmlst_pileup_indirect_dev + mmlst_consensus_indirect_dev as ONE launch: the CTA that finishes the last chunk of a chosen locus (the chunk list of
 * mmlst_select_dev carries, per chunk, its locus and that locus's chunk count; a per-locus ticket counts them) calls the consensus of that locus while
 * its counts are still in L2.  ticket: device u32[max_loci], zeroed once by the caller, left zeroed by every call.  Same results as the two calls.
 * Measured on B200 (configs[1], profiles/r2y_bench_fused{0,1}.json): NOT faster (serial pass 76.9 us against 74.3 us) -- the last chunk of every locus
 * ends with the grid, so the fused consensus is a one-CTA-per-locus tail; the pipeline keeps the two launches unless MMLST_FUSED_TAIL=1. */
int mmlst_pileup_consensus_indirect_dev(const mmlst_prec* recs, const uint32_t* planes, const mmlst_chunk* chunks, const uint32_t* header,
                                        uint32_t max_row_words, int minscore, int max_xm, uint32_t* counts, const uint8_t* db_ascii,
                                        const uint64_t* db_start, const uint32_t* col_off, uint32_t max_loci, uint32_t mincov, uint8_t* cons,
                                        uint32_t* holes, uint32_t* snps, uint32_t flags, uint32_t* ticket, void* stream);
/* flags: MMLST_CONSENSUS_CONSUME = zero every count that was read (the next pass accumulates from zero, no memset) */
#define MMLST_CONSENSUS_CONSUME 1u
int mmlst_consensus_indirect_dev(uint32_t* counts, const uint8_t* db_ascii, const uint64_t* db_start, const uint32_t* col_off,
                                 uint32_t max_loci, const uint32_t* header, uint32_t mincov, uint8_t* cons, uint32_t* holes,
                                 uint32_t* snps, uint32_t flags, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Multi-GPU, owner mode (SURVEY.md 8e): a GPU that holds whole loci (contig-aligned shard) finishes them itself and
 * the pass ends with every GPU holding every GPU's result block.  The reference is single-process (no counterpart);
 * this pair replaces an NCCL all-gather by direct stores into the peers' memory over NVLink.
 *   Symmetric buffer, same layout on every GPU (allocated peer-mapped by the caller, zeroed before first use):
 *     [half 0: world x slot_stride][half 1: world x slot_stride][flag[world] u64 at flag_off]
 *   peer_base[p] = address of GPU p's buffer as mapped into THIS GPU's address space (p == rank: the local one).
 *   epoch = device u64 pass counter (starts at 0), advanced by mmlst_xchg_await_dev; both calls are graph-capturable.
 *   mmlst_xchg_publish_dev: store `block` into slot[rank] of half ((epoch+1)&1) on every GPU, then release
 *                           flag[rank] = epoch+1 there.  Never waits.
 *   mmlst_xchg_await_dev  : wait until every local flag >= epoch+1, copy the world slots of that half into out_all
 *                           (world x bytes, contiguous), epoch += 1.  A wait longer than ~2 s sets bit 2 of *status
 *                           instead of hanging.  ticket = device u32 scratch, zero.
 * --------------------------------------------------------------------------------------------------------------- */
int mmlst_xchg_publish_dev(const void* block, uint32_t bytes, const uint64_t* peer_base, uint32_t rank, uint32_t world,
                           uint64_t half_stride, uint64_t slot_stride, uint64_t flag_off, const uint64_t* epoch, void* stream);
int mmlst_xchg_await_dev(void* local_base, uint32_t bytes, uint32_t world, uint64_t half_stride, uint64_t slot_stride,
                         uint64_t flag_off, void* out_all, uint64_t* epoch, uint32_t* ticket, uint32_t* status, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Multi-GPU, all-reduce form (SURVEY.md 8e; north_star: partial score and pileup-count tensors all-reduced with NCCL over NVLink) for callers that
 * are not torch.distributed processes.  One communicator per GPU: rank 0 makes the 128-byte id (mmlst_comm_unique_id) and hands it to the other ranks
 * by any means, every rank calls mmlst_comm_create (collective).  mmlst_allreduce reduces IN PLACE, on `stream`, any of (NULL / 0 = skip):
 *   score_block[score_words] : int64 words, SUM -- the accumulator block of a pass laid out [sum_as i64 x n_ref | counters u64 x 2 | n_hit u32 x n_ref,
 *                              padded to 8 bytes] (u32 pairs add correctly as 64-bit words below 2^32 hits per allele)
 *   first_idx[n_ref]         : u32, MIN (H5: first passing record of every allele; caller presets 0xFFFFFFFF)
 *   counts[n_counts]         : u32, SUM (count tensor of the chosen contigs, columns x 5)
 * Integer reductions: N ranks give one rank's tables bit for bit.  libnccl.so.2 is resolved at run time; MMLST_E_CUDA when it is missing.
 * --------------------------------------------------------------------------------------------------------------- */
typedef struct mmlst_comm mmlst_comm;
int mmlst_comm_unique_id(uint8_t* id128);
int mmlst_comm_create(const uint8_t* id128, int rank, int world, int device, mmlst_comm** out);
void mmlst_comm_destroy(mmlst_comm* comm);
int mmlst_allreduce(mmlst_comm* comm, int64_t* score_block, size_t score_words, uint32_t* first_idx, size_t n_ref, uint32_t* counts, size_t n_counts,
                    void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Stage 3 -- closest known allele by zip-truncated Hamming distance.  Replaces metaMLST_functions.py:230-234
 * (stringDiff) driven by metamlst-merge.py:174-181 over sequencesGetAll (:224-228).
 *   DB rows   : bit-planes hi/lo of the 2-bit code, tiles of 32 rows, word-major inside a tile:
 *               db_hi[(tile*W + w)*32 + r], same for db_lo; row_len u16; zero padded.  W = words per plane.
 *   queries   : q_hi/q_lo [Q][W] row-major, q_len u16.
 *   blocks[b] = { q_begin, q_end, row_begin, row_end }: every query of the range is compared with every row of the
 *               range (locus-restricted mode = one block per locus; all-pairs = one block).
 *   best[q]   = min over rows of (distance << 32 | row) as u64 -- ties resolve to the lowest row; caller presets
 *               ~0ull; results from row shards / GPUs combine with min (SURVEY.md 8e).
 * H9: stringDiff compares characters.  A sequence holding anything but upper-case A/C/G/T is FLAGGED with bit 15 of its
 * length (lengths are <= 1024); its planes carry the codes of its clean columns (0 elsewhere).  Flagged sequences are
 * skipped by mmlst_hamming_min_dev and compared exactly by mmlst_hamming_exact_dev, which needs, for the flagged rows
 * and the flagged queries each: ids[n] ascending, x[n][W] = bit-plane of the exceptional columns, bytes[n][W*32] = the
 * ASCII characters (zero padded).  Both calls min-merge into the same best[].
 * --------------------------------------------------------------------------------------------------------------- */
int mmlst_hamming_min_dev(const uint32_t* db_hi, const uint32_t* db_lo, const uint16_t* row_len, uint32_t n_rows,
                          uint32_t W, const uint32_t* q_hi, const uint32_t* q_lo, const uint16_t* q_len, uint32_t n_q,
                          const uint32_t* blocks, uint32_t n_blocks, uint32_t row_index_base,
                          unsigned long long* best, void* stream);
int mmlst_hamming_exact_dev(const uint32_t* db_hi, const uint32_t* db_lo, const uint16_t* row_len, uint32_t n_rows, uint32_t W,
                            const uint32_t* q_hi, const uint32_t* q_lo, const uint16_t* q_len, uint32_t n_q,
                            const uint32_t* blocks, uint32_t n_blocks, uint32_t row_index_base,
                            const uint32_t* xr_ids, const uint32_t* xr_x, const uint8_t* xr_bytes, uint32_t n_xr,
                            const uint32_t* xq_ids, const uint32_t* xq_x, const uint8_t* xq_bytes, uint32_t n_xq,
                            unsigned long long* best, void* stream);
/* same, with the grid sized by the caller: max_block_rows / max_block_queries = largest row / query range of any block
 * (the plain form assumes every block may span everything) */
int mmlst_hamming_min_dev2(const uint32_t* db_hi, const uint32_t* db_lo, const uint16_t* row_len, uint32_t n_rows,
                           uint32_t W, const uint32_t* q_hi, const uint32_t* q_lo, const uint16_t* q_len, uint32_t n_q,
                           const uint32_t* blocks, uint32_t n_blocks, uint32_t max_block_rows, uint32_t max_block_queries,
                           uint32_t row_index_base, unsigned long long* best, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Host-buffer entry points (what the Python seams call; host<->device copies inside).
 * --------------------------------------------------------------------------------------------------------------- */
/* Optional DEFLATE-compressed copy of the two per-record arrays of the score stream (as0, xm3).  The host-buffer path is PCIe-bound (3 bytes per
 * record cross the bus, the kernel reads them at 4 TB/s); alignment scores and mismatch counts of one sequencing run take a handful of values, so
 * the arrays deflate 3-4x.  When mmlst_soa.z is set (and the run-length form is used) mmlst_score ships THESE bytes and inflates them on the device
 * with the hardware decompression engine, slice by slice behind the copy.  blocks: independent raw-DEFLATE streams of at most 4 MiB of output each,
 * table[b] = { destination array (0 = as0 bytes, 1 = xm3 bytes), destination byte offset, source byte offset in `bytes`,
 * (compressed size << 32) | inflated size }, ordered by source offset.  The blocks of an array tile a PREFIX of it, in order; what they do not
 * cover is copied plain from as0 / xm3 after the compressed bytes (the bus carries it while the engine, the slower of the two, drains its queue).
 * Made once per sample by metamlst_b200.packing.SoaHost.deflate(). */
typedef struct {
    const uint8_t* bytes; uint64_t n_bytes;
    const uint64_t* table; uint32_t n_blocks;
    /* Decorrelation before DEFLATE: the as0 blocks hold as0[i] + as_xm_coeff * xm3[i] (still int16; 0 = as0 itself).  An aligner's score is its match
     * bonus minus a penalty per mismatch, so with the right coefficient (bowtie2: 6) what is left of as0 takes a handful of values and deflates to a
     * fraction: 0.43 instead of 0.85 bytes per record for the two arrays on configs[1].  The library subtracts it again on the device after the blocks
     * are inflated (mmlst_as_untransform_dev); only the part of as0[] covered by blocks is transformed.  SoaHost.deflate() picks the coefficient per
     * sample by trying 0..8 on a slice of the arrays. */
    int32_t as_xm_coeff;
} mmlst_zstream;

/* Optional DEFLATE-compressed copy of the PILEUP stream, contig by contig, so that mmlst_sample ships only the chosen contigs' blocks and the hardware
 * decompression engine writes their records and plane rows in HBM (stage 2 of the call is PCIe-bound too: ~90 bytes per admitted record; plane rows of
 * reads piled on the same columns repeat each other, records differ in a few fields: they deflate about 2x and 3.5x).  Every contig t with records
 * owns the blocks contig_block[t] .. contig_block[t+1]: independent raw-DEFLATE streams of at most 4 MiB of output, stored back to back in `bytes` in
 * table order; table[2b] = byte offset of block b in `bytes`, table[2b+1] = kind << 63 | compressed size << 32 | inflated size, kind 0 = bytes of the
 * contig's plane rows (planes[row_off of its first record .. row end of its last record)), kind 1 = bytes of its 16-byte records; the blocks of a
 * kind tile the contig's range in order.  `p_recs` / `planes` stay mandatory: entry points other than mmlst_sample, and devices without the engine,
 * read them.  Made once per sample by metamlst_b200.packing.SoaHost.deflate(pileup=True). */
typedef struct {
    const uint8_t* bytes; uint64_t n_bytes;
    const uint64_t* table; uint32_t n_blocks;
    const uint32_t* contig_block;   /* [n_ref + 1] */
} mmlst_zpileup;

typedef struct {
    /* score stream */
    const uint32_t* tid; const int16_t* as0; const uint8_t* xm3; const uint16_t* qlen; const uint32_t* orig_idx;
    uint64_t n_rec;
    /* pileup stream */
    const mmlst_prec* p_recs;
    const uint32_t* planes; uint64_t n_prec; uint64_t n_plane_words; uint32_t max_row_words;
    /* per reference (allele row) */
    const uint64_t* contig_start; /* [n_ref+1] first pileup-stream record of each contig */
    uint32_t n_ref;
    /* run-length form of the score stream (mmlst_score_runs_dev); when run_tid != NULL the host entry points upload
     * 5 B / record + the run arrays and never read `tid` (which may then be NULL) */
    uint32_t n_runs;
    const uint32_t* run_tid; const uint32_t* run_start; const uint32_t* chunk_run;
    /* with the run arrays only: len(SEQ) per 256-record chunk (mmlst_score_runs_qc_dev); when != NULL the host entry
     * points upload 3 B / record and never read `qlen` */
    const uint16_t* chunk_qlen;
    /* with the run arrays only: as0 / xm3 as DEFLATE blocks (see mmlst_zstream); mmlst_score then reads `as0` / `xm3` only past what the blocks cover */
    const mmlst_zstream* z;
    /* the pileup stream as DEFLATE blocks per contig (see mmlst_zpileup); read by mmlst_sample only */
    const mmlst_zpileup* zp;
} mmlst_soa;

typedef struct { int minscore, max_xm, min_read_len; } mmlst_score_params;

/* seam S1 (metamlst.py:96-151): uploads the score stream, runs the kernel, returns the integer tables. */
int mmlst_score(mmlst_ctx* ctx, const mmlst_soa* soa, const uint8_t* allow, const uint32_t* locus_of, uint32_t n_loci,
                const mmlst_score_params* prm, int64_t* sum_as, uint32_t* n_hit, uint32_t* first_idx, uint64_t* counters);

/* ---------------------------------------------------------------------------------------------------------------
 * One call per sample over HOST buffers: what metamlst.py:96-287 does for one BAM between reading it and writing the
 * .nfo -- score every record (seam S1), pick the best allele per locus and order species / loci (metamlst.py:133-220,
 * on the device: mmlst_select_dev), pile up and call the consensus of the chosen contigs (seam S2, buildConsensus).
 * Against mmlst_score + a host selection + mmlst_pileup_consensus it saves the D2H of the score tables, the host
 * selection and two synchronisations; only the chosen contigs' pileup records cross the bus, after the selection.
 *
 * mmlst_index: what selection and consensus need from the allele DB and the BAM header, uploaded once per (DB, aligner index):
 *   locus_of[n_ref] locus of every reference (allele row), allele_num[n_ref] = int(alleleVariant),
 *   species_of_locus[n_loci], genes_in_db[n_species] = rows of `genes` per organism (metamlst.py:184),
 *   db_ascii / db_off[n_ref+1]: the DB sequence of every row (metaMLST_functions.py:260-276 compares against it),
 *   bam_ln[n_ref]: @SQ LN of every reference.
 *   An index the selection cannot serve (see the range of mmlst_select_dev) is refused by mmlst_index_upload with MMLST_E_RANGE.
 * mmlst_sample_result: caller-allocated arrays sized for n_loci entries (col_off: n_loci + 1), cons for cons_capacity bytes;
 *   sum_as / n_hit / first_idx optional (all three or none).  Output order = the reference's dict order (H5).
 *   error_bits & 1: "Database is broken" (metamlst.py:188-190), nothing piled up.  MMLST_E_RANGE + bad_len_tid: a chosen reference
 *   whose BAM LN exceeds its DB sequence (the reference raises IndexError, H10).
 * --------------------------------------------------------------------------------------------------------------- */
typedef struct {
    const uint32_t* locus_of; const uint32_t* allele_num; uint32_t n_ref;
    const uint32_t* species_of_locus; uint32_t n_loci;
    const uint32_t* genes_in_db; uint32_t n_species;
    const uint8_t* db_ascii; const uint64_t* db_off; const uint32_t* bam_ln;
} mmlst_index;
typedef struct { int minscore, max_xm, min_read_len, penalty, nloci_pct; uint32_t mincov; int pileup_impl; } mmlst_sample_params;
typedef struct {
    uint32_t n_chosen, error_bits, bad_len_tid, reserved;
    uint64_t total_reads, ignored_reads;
    uint32_t* chosen_tid; uint32_t* chosen_species; uint32_t* col_off;
    uint8_t* cons; uint64_t cons_capacity;
    uint32_t* holes; uint32_t* snps;
    int64_t* sum_as; uint32_t* n_hit; uint32_t* first_idx;
} mmlst_sample_result;
int mmlst_index_upload(mmlst_ctx* ctx, const mmlst_index* index);
int mmlst_sample(mmlst_ctx* ctx, const mmlst_soa* soa, const uint8_t* allow, const mmlst_sample_params* prm, mmlst_sample_result* res);

/* seam S1, coverage column (metamlst.py:127,228).  MMLST_COVERAGE_STREAM_RESIDENT: the score stream of THIS soa is still
 * in the context from the preceding mmlst_score call (only the 16 B/record hashes are uploaded). */
#define MMLST_COVERAGE_STREAM_RESIDENT 1u
int mmlst_coverage(mmlst_ctx* ctx, const mmlst_soa* soa, const uint64_t* qhash, const uint8_t* allow, const uint32_t* locus_of,
                   uint32_t n_loci, const mmlst_score_params* prm, uint32_t flags, uint64_t* cov);

/* seam S2 (metaMLST_functions.py:249-281): uploads the chosen contigs' pileup records, runs pileup + consensus.
 *   chosen_tid[n_loci], dbseq/col_off as in mmlst_consensus_dev; counts may be NULL. */
int mmlst_pileup_consensus(mmlst_ctx* ctx, const mmlst_soa* soa, const uint32_t* chosen_tid, uint32_t n_loci,
                           const uint8_t* dbseq, const uint32_t* col_off, int minscore, int max_xm, uint32_t mincov,
                           int impl, uint32_t* counts, uint8_t* cons, uint32_t* holes, uint32_t* snps);

/* seam S2' bulk (cmseq_api.BamFile *_all methods): mmlst_contig_stats_dev over a batch of contigs of a pileup stream, host buffers.
 * The records and plane rows of the contigs (consecutive contigs are one contiguous range of the sorted stream and cross the bus as
 * one copy) -> mmlst_pileup_dev (library chunk rule) ->
 * mmlst_contig_stats_dev -> the [n+1] prefixes, then the compacted prefix they size, back to the host.  tid[n] ascending,
 * col_off[n+1] = prefix of the contigs' lengths (host).  Range: col_off[n] <= MMLST_CONTIG_STATS_MAX_COLS, else MMLST_E_RANGE
 * (checked before anything else).  out->capacity = entries of out_col (out_val holds width x as many); out->n_out = entries written. */
typedef struct {
    uint32_t* sel_off;           /* [n+1] */
    uint32_t* low_off;           /* [n+1] */
    uint64_t* depth_off;         /* [n+1] */
    uint32_t* out_col;           /* [capacity] */
    uint32_t* out_val;           /* [capacity * width] */
    uint8_t* cons;               /* [col_off[n]] or NULL */
    uint64_t capacity;
    uint64_t n_out;
} mmlst_contig_stats_out;
int mmlst_contig_stats(mmlst_ctx* ctx, const mmlst_soa* soa, const uint32_t* tid, uint32_t n, const uint32_t* col_off, int minscore,
                       int max_xm, const mmlst_contig_stats_params* prm, mmlst_contig_stats_out* out);

/* seam S3 (metamlst-merge.py:177-181): DB planes stay resident in the context across calls / samples. */
int mmlst_db_upload(mmlst_ctx* ctx, const uint32_t* db_hi, const uint32_t* db_lo, const uint16_t* row_len,
                    uint32_t n_rows, uint32_t W);
int mmlst_hamming_min(mmlst_ctx* ctx, const uint32_t* q_hi, const uint32_t* q_lo, const uint16_t* q_len, uint32_t n_q,
                      const uint32_t* blocks, uint32_t n_blocks, uint32_t* min_dist, uint32_t* argmin_row);
/* the same two calls with the flagged (non-ACGT, H9) rows / queries attached; runs the fast and the exact kernels */
int mmlst_db_upload_x(mmlst_ctx* ctx, const uint32_t* db_hi, const uint32_t* db_lo, const uint16_t* row_len, uint32_t n_rows,
                      uint32_t W, const uint32_t* xr_ids, const uint32_t* xr_x, const uint8_t* xr_bytes, uint32_t n_xr);
int mmlst_hamming_min_x(mmlst_ctx* ctx, const uint32_t* q_hi, const uint32_t* q_lo, const uint16_t* q_len, uint32_t n_q,
                        const uint32_t* xq_ids, const uint32_t* xq_x, const uint8_t* xq_bytes, uint32_t n_xq,
                        const uint32_t* blocks, uint32_t n_blocks, uint32_t* min_dist, uint32_t* argmin_row);

/* ---------------------------------------------------------------------------------------------------------------
 * Stage 3 on the tensor cores (csrc/hamming_tc.cu): the all-pairs closest-allele sweep as a tcgen05 GEMM.  Same semantics, same best[]
 * convention as mmlst_hamming_min_dev for ONE block covering every query and every row (metaMLST_functions.py:230-234 over
 * metamlst-merge.py:174-181): distance = (3 min(len) - <f(q), f(r)>) / 4 with every base written as three signs in e4m3 and zeros
 * beyond the end of a sequence (the zip truncation, H9); exact (integers in an FP32 accumulator).  Flagged sequences are skipped
 * (mmlst_hamming_exact_dev covers them).
 *   mmlst_hamming_tc_expand_dev : bit planes -> e4m3 tile image (device, 16-byte aligned, mmlst_hamming_tc_image_bytes bytes) + the
 *                                 largest clean length of every tile; tile_rows = 128 for queries ([Q][W] row-major planes,
 *                                 db_tiled_layout = 0), 256 for DB rows (the tiled plane layout of mmlst_hamming_min_dev,
 *                                 db_tiled_layout = 1).  W a multiple of 4.  The DB image is made once and stays resident.
 *   mmlst_hamming_tc_search_dev : min-merges into best[q] (caller presets ~0ull); persistent kernel, one CTA per SM.
 * --------------------------------------------------------------------------------------------------------------- */
size_t mmlst_hamming_tc_image_bytes(uint32_t n, uint32_t W, uint32_t tile_rows);
int mmlst_hamming_tc_expand_dev(const uint32_t* hi, const uint32_t* lo, const uint16_t* len, uint32_t n, uint32_t W, int db_tiled_layout,
                                uint32_t tile_rows, uint8_t* image, uint32_t* tile_maxlen, void* stream);
int mmlst_hamming_tc_search_dev(const uint8_t* q_image, const uint32_t* q_tile_maxlen, const uint16_t* q_len, uint32_t n_q,
                                const uint8_t* db_image, const uint32_t* db_tile_maxlen, const uint16_t* row_len, uint32_t n_rows,
                                uint32_t W, uint32_t row_index_base, unsigned long long* best, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Exact-sequence lookup (row a10).  Replaces the un-indexed scans `SELECT .. FROM alleles WHERE sequence = ? AND bacterium = ?`
 * + fetchone() of sequenceExists / sequenceFind / sequenceLocate (metaMLST_functions.py:168-172, 196-203, 218-222):
 *   first_row[q] = lowest DB row (or lowest row_key[row], see mmlst_db_row_keys) inside the query's block (= the organism's row range, table order) whose sequence equals the
 *   query character for character -- same length AND same characters, case-sensitive like SQLite's `=` (H10); 0xFFFFFFFF when
 *   there is none (caller presets it for the _dev form).  Same DB / query layouts and `blocks` as mmlst_hamming_min_dev; the
 *   flagged (non-ACGT, bit 15 of the length) sequences compare their stored bytes (x*_ids ascending, x*_bytes [n][W*32]).
 *   Not "zip-Hamming distance 0": the truncating distance is also 0 against a prefix or an extension of the query.
 * --------------------------------------------------------------------------------------------------------------- */
int mmlst_exact_match_dev(const uint32_t* db_hi, const uint32_t* db_lo, const uint16_t* row_len, uint32_t n_rows, uint32_t W,
                          const uint32_t* q_hi, const uint32_t* q_lo, const uint16_t* q_len, uint32_t n_q,
                          const uint32_t* blocks, uint32_t n_blocks, uint32_t max_block_rows, uint32_t row_index_base,
                          const uint32_t* row_key /* NULL: key = row + row_index_base */, const uint32_t* xr_ids, const uint8_t* xr_bytes, uint32_t n_xr,
                          const uint32_t* xq_ids, const uint8_t* xq_bytes, uint32_t n_xq, uint32_t* first_row, void* stream);
/* host buffers, against the DB made resident by mmlst_db_upload[_x].  mmlst_db_row_keys attaches a key per resident row (its
 * position in table order when the rows are resident grouped by locus): first_row[q] is then the lowest KEY of an equal row,
 * which is what fetchone() returns when several genes of the organism hold the same sequence.  NULL detaches. */
int mmlst_db_row_keys(mmlst_ctx* ctx, const uint32_t* row_key, uint32_t n_rows);
int mmlst_exact_match(mmlst_ctx* ctx, const uint32_t* q_hi, const uint32_t* q_lo, const uint16_t* q_len, uint32_t n_q,
                      const uint32_t* xq_ids, const uint8_t* xq_bytes, uint32_t n_xq,
                      const uint32_t* blocks, uint32_t n_blocks, uint32_t* first_row);

/* ---------------------------------------------------------------------------------------------------------------
 * Seam S4 -- ST assignment (row a11).  Replaces the GROUP BY / HAVING statement of defineProfile (metaMLST_functions.py:205-216):
 * among the rows of `profiles` whose alleleCode is one of the query's allele codes, count per profileCode; answer = the
 * profiles whose count equals the maximum and that count.  The device list is ascending by profileCode; SQLite emits the ties of
 * `ORDER BY T DESC` in descending profileCode order, which the Python seam restores (api.ProfileIndex).
 *   prof_start[n_st+1], prof_allele[]: the `profiles` table grouped by profileCode, profiles ascending by code;
 *                                      prof_allele = alleleCode (alleles.recID) of every row of the group
 *   q_alleles[n_q][l_max], q_n[n_q]  : allele codes of every query (labels already resolved to recIDs; unknown labels dropped
 *                                      by the caller, H11).  A code listed twice counts a row once (`IN` is a set test).
 *   best[q] = the maximum count (0: no profile row matches), n_best[q] = number of profiles reaching it,
 *   out_idx[q][max_out] = their indices into the grouped table, ascending (the first max_out of them).
 *   count: device scratch n_q * n_st u32.  The percentage int(best / len(recs) * 100) stays on the host (Python floats, H6).
 * --------------------------------------------------------------------------------------------------------------- */
int mmlst_st_match_dev(const uint32_t* prof_start, const uint32_t* prof_allele, uint32_t n_st,
                       const uint32_t* q_alleles, const uint32_t* q_n, uint32_t l_max, uint32_t n_q,
                       uint32_t* count, uint32_t* best, uint32_t* n_best, uint32_t* out_idx, uint32_t max_out, void* stream);
int mmlst_profiles_upload(mmlst_ctx* ctx, const uint32_t* prof_start, const uint32_t* prof_allele, uint32_t n_st);
int mmlst_st_match(mmlst_ctx* ctx, const uint32_t* q_alleles, const uint32_t* q_n, uint32_t l_max, uint32_t n_q,
                   uint32_t* best, uint32_t* n_best, uint32_t* out_idx, uint32_t max_out);

/* Raw DEFLATE (RFC 1951) of ONE complete stream, e.g. the payload of a BGZF block, into a buffer of known size: the decoder
 * the BAM unpacker uses instead of zlib's inflate() (whole-buffer, 64-bit bit buffer, two-level tables; every access is
 * bounds-checked).  HOST.  Returns MMLST_OK and *produced = bytes written (<= out_capacity), or MMLST_E_BAM for a corrupt /
 * truncated stream or one that does not fit.  Exported for the tests (byte-for-byte against zlib). */
int mmlst_inflate_raw(const uint8_t* in, size_t n, uint8_t* out, size_t out_capacity, size_t* produced);

/* ---------------------------------------------------------------------------------------------------------------
 * BAM ingest (HOST, C++ threads + zlib).  Replaces the `samtools view -h -` text pipe of stage 1 (metamlst.py:96-110),
 * pysam's record access of stage 2 (cmseq/cmseq.py:54,527-545) and `samtools sort` + `samtools index`
 * (metaMLST_functions.py:237-247; the input file is never overwritten).  One pass: BGZF blocks inflated in
 * parallel, records walked once, streams emitted in `samtools sort` order (stable by tid, pos, reverse strand) with
 * the htslib depth cap applied.  Everything the reference would crash on is refused with MMLST_E_BAM and the
 * reference line named in mmlst_last_error(): RNAME '*' (metamlst.py:107), 1st/4th aux field missing or not an
 * integer (:109-110), a pileup record without integer AS/XM tags or without qualities (cmseq/cmseq.py:538,545);
 * proper-pair mates are refused with MMLST_E_PAIRED (H2).
 *   minqual       : pysam min_base_quality (20 at the only call site, metaMLST_functions.py:258)
 *   max_depth     : pysam pileup max_depth (8000 default reaches cmseq unchanged); 0 = no cap
 *   assume_sorted : metamlst.py --presorted -- keep the file order, MMLST_E_UNSORTED if it is not coordinate order
 *   want_qhash    : also emit the 128-bit QNAME hash (2 x u64) per score-stream record (coverage column, H7)
 * --------------------------------------------------------------------------------------------------------------- */
typedef struct mmlst_bam mmlst_bam;
typedef struct {
    int minqual; uint32_t max_depth; uint32_t sentinel_nodes; int n_threads; int pinned; int assume_sorted;
    int want_qhash; int check_crc;
    /* HOST unpacker only (mmlst_bam_ingest refuses it).  0 = MetaMLST's own crash rules: a record whose 1st / 4th aux field is missing or not an integer,
     * or a pileup record without integer AS:i / XM:i tags, is MMLST_E_BAM.  1 = what a cmseq user without a tag filter gets from pysam: such records are
     * kept -- positional fields read as -32768 / 255 (no stage-1 filter ever passes them; the Python side refuses to SCORE a stream unpacked this way),
     * missing named tags read as 0 and are counted in mmlst_bam_info_t.n_untagged, so that a caller who DOES pass a tag filter can raise the reference's
     * KeyError (cmseq/cmseq.py:545) instead of filtering on invented values.  Proper-pair mates stay refused (H2). */
    int lenient_tags;
} mmlst_unpack_opts;
typedef struct {
    mmlst_soa soa;              /* pointers into memory owned by the mmlst_bam handle, page-locked when opts.pinned */
    const uint64_t* qhash;      /* [n_rec][2] or NULL */
    const uint32_t* ref_len;    /* [n_ref] BAM header LN */
    const char* ref_names;      /* n_ref names joined by '\n' */
    const char* header_text;
    uint64_t n_dropped_by_cap, n_unmapped_flag;
    int presorted, minqual; uint32_t max_depth;
    double seconds[5];          /* read, inflate, parse, sort, pack */
    uint64_t n_untagged;        /* lenient_tags: pileup records without integer AS:i / XM:i (0 otherwise: they are refused) */
} mmlst_bam_info_t;
int mmlst_bam_unpack(const char* path, const mmlst_unpack_opts* opts /* NULL = defaults */, mmlst_bam** out);
int mmlst_bam_info(const mmlst_bam* bam, mmlst_bam_info_t* info);
void mmlst_bam_free(mmlst_bam* bam);

/* ---------------------------------------------------------------------------------------------------------------
 * BAM ingest ON THE DEVICE (csrc/ingest.cu).  Same replacement as mmlst_bam_unpack (metamlst.py:96-110, cmseq/cmseq.py:54,527-545,
 * metaMLST_functions.py:237-247), same streams, same refusals -- but only the COMPRESSED file crosses PCIe: BGZF blocks are
 * inflated by the hardware decompression engine (cuMemBatchDecompressAsync, DEFLATE), records are chained, parsed, put in
 * `samtools sort` order, depth-capped and packed by kernels, and the result stays in HBM.
 *   bam / n_bytes : the whole BAM file in HOST memory (page-locked memory from mmlst_pinned_alloc makes the copy one async DMA)
 *   opts          : as mmlst_bam_unpack (n_threads, pinned ignored).  The engine verifies the DEFLATE stream and a kernel the ISIZE of
 *                   every block; check_crc = 1 also checks every non-empty block's CRC32 against its trailer (MMLST_E_BAM, "CRC mismatch
 *                   in BGZF block k", k counting non-empty blocks as mmlst_bam_unpack does; its time is part of seconds[1]).  With
 *                   opts == NULL check_crc is 0, unlike mmlst_bam_unpack's default of 1.
 *   stream        : cudaStream_t the work is queued on (NULL = the default stream); the call returns after the last kernel finished
 * Every pointer of mmlst_dev_bam_info_t except contig_start / ref_len / ref_names / header_text is a DEVICE pointer owned by the
 * handle.  MMLST_E_CUDA when the device has no hardware DEFLATE (then use mmlst_bam_unpack).
 * --------------------------------------------------------------------------------------------------------------- */
typedef struct mmlst_dev_bam mmlst_dev_bam;
typedef struct {
    const uint32_t* tid; const int16_t* as0; const uint8_t* xm3; const uint16_t* qlen; const uint32_t* orig_idx; const uint64_t* qhash;
    const uint32_t* run_tid; const uint32_t* run_start; const uint32_t* chunk_run; const uint16_t* chunk_qlen; uint32_t n_runs;
    const mmlst_prec* p_recs; const uint32_t* planes;
    uint64_t n_rec, n_prec, n_plane_words; uint32_t max_row_words;
    const uint64_t* contig_start;   /* HOST [n_ref+1] */
    const uint32_t* ref_len;        /* HOST [n_ref] */
    const char* ref_names;          /* HOST, joined by '\n' */
    const char* header_text;        /* HOST */
    uint32_t n_ref;
    uint64_t n_dropped_by_cap, n_unmapped_flag, n_bgzf_blocks, compressed_bytes, inflated_bytes;
    int presorted, minqual; uint32_t max_depth; int boundary_repairs;
    double seconds[8];              /* device time: H2D, inflate, record chain, parse, sort, score stream, depth cap + compaction, pack */
} mmlst_dev_bam_info_t;
int mmlst_bam_ingest(int device, const uint8_t* bam, size_t n_bytes, const mmlst_unpack_opts* opts, void* stream, mmlst_dev_bam** out);
int mmlst_dev_bam_info(const mmlst_dev_bam* bam, mmlst_dev_bam_info_t* info);
void mmlst_dev_bam_free(mmlst_dev_bam* bam);
/* the ingest keeps its device workspace (a few allocations of up to the inflated size of the largest file seen) cached between calls;
 * this gives the idle blocks back to the driver */
int mmlst_ingest_trim(int device);

#ifdef __cplusplus
}
#endif
#endif /* MMLST_H */
