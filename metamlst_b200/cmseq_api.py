"""Seam S2' -- the slice of cmseq's API that sits on the pileup hot path (SURVEY.md 8b), over the GPU count tensor.

Mirrors `cmseq/cmseq.py` for users of cmseq other than MetaMLST: `BamFile(bam, filterInputList=...)`
(`cmseq/cmseq.py:35-88`) -> `get_contig_by_label(name)` -> `BamContig.get_base_stats` (`:507-569`),
`reference_free_consensus` (`:226-241`), `majority_rule` / `majority_rule_polymorphicLoci` (`:202-224`),
`polymorphism_rate` (`:430-456`), `breadth_and_depth_of_coverage` / `depth_of_coverage` / `breadth_of_coverage`
(`:459-505`), `get_all_base_values` (`:572-578`).  Same names, arguments, return shapes and key order.

What replaces pysam: the BAM is unpacked once per base-quality threshold by the native unpacker (`bam.unpack_bam`; the
threshold is folded into the bit-planes, H3) and a contig's five counters per column come from the bit-sliced pileup
kernel (`mmlst_pileup_consensus`).  Everything after the counters (ratio, binomial p-value, dict layout, the consensus
rule) is the reference's own per-column arithmetic in Python floats, so values are identical, not merely close.

Files MetaMLST itself would crash on are accepted the way pysam accepts them (`lenient_tags`): records without integer 1st / 4th aux fields
or without AS:i / XM:i tags take part in the pileup; only a call that passes a `BAM_tagFilter` on such a file raises the reference's KeyError.
Proper-pair mates are still refused (`MMLST_E_PAIRED`): pysam's `ignore_overlaps` handling (H2) is not implemented.

Whole-BAM methods on `BamFile` (`base_stats_all`, `base_stats_arrays`, `reference_free_consensus_all`, `polymorphism_rate_all`,
`breadth_and_depth_of_coverage_all`) return, for every contig the handle keeps, exactly what the per-contig method returns.  They cut
the contigs into batches under a column budget; per batch ONE library call (`mmlst_contig_stats`) uploads the batch's records, counts
them and selects / compacts the columns on the device, and only the compacted columns come back.  The per-contig methods and these
share one host definition of the reference's arithmetic (`_column_stats`, `_base_stats_dict`, `_poly_dict`, `_breadth_tuple`).

Not carried over (each raises, nothing degrades silently): `trimReads` (the bit-planes carry no read coordinate),
`BAM_tagFilter` entries other than `('AS','loc_gte',x)` / `('XM','loc_lte',y)` (the only ones MetaMLST passes,
`metaMLST_functions.py:259`), `stepper='all'`, the GFF/codon functions (`parse_gff`, `baseline_PSR`,
`get_base_stats_for_poly`, `easy_polymorphism_rate`) and the multiprocessing wrapper -- off the hot path.
"""
from __future__ import annotations

import math
import os
from collections import defaultdict
from typing import Dict, Iterable, List, NamedTuple, Optional, Sequence, Tuple
import ctypes as C

import numpy as np

from . import api, bam as bam_mod, native


class CMSEQ_DEFAULTS:  # cmseq/cmseq.py:25-32
    minqual = 30
    mincov = 1
    minlen = 0
    poly_error_rate = 0.001
    poly_pvalue_threshold = 0.01
    poly_dominant_frq_thrsh = 0.8
    trimReads = None


PYSAM_DEFAULT_MIN_BASE_QUALITY = 13  # what `pileup()` applies when cmseq does not pass one (cmseq/cmseq.py:469)
_NO_MINSCORE, _NO_MAX_XM = -32768, 255  # thresholds every record passes (as_named is i16, xm_named u8)


def _tag_filter(BAM_tagFilter) -> Tuple[int, int]:
    """(minscore, max_xM) of a cmseq BAM_tagFilter.  cmseq evaluates `all(func(tag value, limit))` per read
    (`cmseq/cmseq.py:545`); the kernels implement AS >= x and XM <= y."""
    minscore, max_xm = _NO_MINSCORE, _NO_MAX_XM
    for ent in (BAM_tagFilter or ()):
        tag, func, limit = ent
        if tag == "AS" and func == "loc_gte":
            minscore = max(minscore, int(limit))
        elif tag == "XM" and func == "loc_lte":
            max_xm = min(max_xm, int(limit))
        else:
            raise NotImplementedError("BAM_tagFilter entry %r: only ('AS','loc_gte',x) and ('XM','loc_lte',y) run on the device" % (ent,))
    return minscore, max(max_xm, -1)


def _contig_counts(ctx: native.Context, soa, tid: int, minscore: int, max_xm: int) -> np.ndarray:
    """counts[len][5] (A,C,G,T,N) of one contig from the pileup kernel.  The seam the CPU tests answer with the oracle."""
    ln = int(soa.ref_lens[tid])
    _seqs, _holes, _snps, counts, _off = api.pileup_consensus(ctx, soa, [tid], ["N" * ln], minscore, max_xm, 1, 0, True)
    return counts


class _BatchStats(NamedTuple):
    """What `mmlst_contig_stats` returns for a batch of contigs (include/mmlst.h): prefixes [n+1] of the selected columns, the
    low-dominance columns and the depth sum; the compacted columns (column inside the contig, `width` values each); the consensus bytes."""
    sel_off: np.ndarray
    low_off: np.ndarray
    depth_off: np.ndarray
    cols: np.ndarray
    vals: np.ndarray
    cons: Optional[np.ndarray]


_WIDTH = {native.STATS_COLUMNS: 5, native.STATS_DEPTH: 1, native.STATS_LOWDOM: 2}


def _bulk_stats(ctx: native.Context, soa, tids: Sequence[int], col_off: np.ndarray, minscore: int, max_xm: int,
                prm: native.ContigStatsParams, want_cons: bool) -> _BatchStats:
    """Pileup + column selection of a batch of contigs (tids ascending) in one library call.  The bulk seam the CPU tests answer with
    the oracle's counts and a numpy restatement of the column rule."""
    n, total = len(tids), int(col_off[-1])
    width = _WIDTH[prm.mode]
    sel_off, low_off, depth_off = np.zeros(n + 1, np.uint32), np.zeros(n + 1, np.uint32), np.zeros(n + 1, np.uint64)
    cols, vals = np.empty(max(total, 1), np.uint32), np.empty((max(total, 1), width), np.uint32)
    cons = np.empty(max(total, 1), np.uint8) if want_cons else None
    out = native.ContigStatsOut(native.ptr(sel_off), native.ptr(low_off), native.ptr(depth_off), native.ptr(cols), native.ptr(vals),
                                native.ptr(cons), total, 0)
    tid_arr = np.asarray(tids, dtype=np.uint32)
    cs = soa.c_struct()
    native.check(native.lib().mmlst_contig_stats(ctx.handle, C.byref(cs), native.ptr(tid_arr), n, native.ptr(col_off), int(minscore), int(max_xm),
                                                 C.byref(prm), C.byref(out)))
    k = int(out.n_out)
    return _BatchStats(sel_off, low_off, depth_off, cols[:k], vals[:k], cons[:total] if want_cons else None)


# ---- the reference's host arithmetic, one definition for the per-contig and the whole-BAM methods ----------------------------------
def _window(length: int, trunc) -> Tuple[int, int]:
    """cmseq/cmseq.py:459-490 as breadth_and_depth_of_coverage restates it: `trunc` columns dropped at both ends when the contig is long
    enough for that."""
    return (int(trunc), int(length - trunc)) if length > trunc * 2 else (0, int(length))


def _selected(counts: np.ndarray, mincov, lo: int = 0, hi: Optional[int] = None) -> Tuple[np.ndarray, np.ndarray]:
    """(0-based columns, A+C+G+T) of the columns of one contig's counts inside [lo, hi) whose A+C+G+T reaches mincov (cmseq/cmseq.py:551)."""
    depth = counts[lo:hi, :4].astype(np.int64).sum(axis=1)
    hit = np.nonzero(depth >= mincov)[0]
    return hit + lo, depth[hit]


def _pvalues(base_max: np.ndarray, base_sum: np.ndarray, error_rate) -> np.ndarray:
    """binom.cdf(base_max, base_sum, 1 - error_rate) per column (cmseq/cmseq.py:558), vectorised: the same ufunc per element."""
    from scipy import stats  # the reference imports it at module level (cmseq/cmseq.py:9)
    return stats.binom.cdf(np.asarray(base_max, dtype=np.float64), np.asarray(base_sum, dtype=np.int64), 1.0 - error_rate)


def _ratios(base_max: np.ndarray, base_sum: np.ndarray) -> np.ndarray:
    """base_max / base_sum as float64 division (cmseq/cmseq.py:556)."""
    return np.asarray(base_max, dtype=np.float64) / np.asarray(base_sum, dtype=np.int64)


def _column_stats(c5: np.ndarray, dominant_frq_thrsh, error_rate):
    """(base_cov, ratio_max2all, low, p) of selected columns with counts c5[k][5]: the binomial p-value only where the dominant base is
    under dominant_frq_thrsh (`low`), 1.0 elsewhere (cmseq/cmseq.py:553-562)."""
    acgt = np.asarray(c5)[:, :4].astype(np.int64)
    cov, mx = acgt.sum(axis=1), acgt.max(axis=1)
    ratio = _ratios(mx, cov)
    low = ratio < dominant_frq_thrsh
    p = np.ones(len(cov))
    if low.any():
        p[low] = _pvalues(mx[low], cov[low], error_rate)
    return cov, ratio, low, p


def _base_stats_dict(cols: np.ndarray, c5: np.ndarray, cov: np.ndarray, ratio: np.ndarray, low: np.ndarray, p: np.ndarray):
    """get_base_stats' dict (cmseq/cmseq.py:564-568): {1-based position: {'p', 'ratio_max2all', 'base_cov', 'base_freq'}}, p a numpy
    float64 where the binomial test ran and the literal 1.0 elsewhere, every other leaf a Python int / float."""
    base_stats = defaultdict(dict)
    for i, (pos, (a, c, g, t, n), s, r, lw) in enumerate(zip((np.asarray(cols, dtype=np.int64) + 1).tolist(), np.asarray(c5).tolist(),
                                                            np.asarray(cov).tolist(), np.asarray(ratio).tolist(), np.asarray(low).tolist())):
        col = base_stats[pos]
        col['p'] = p[i] if lw else 1.0
        col['ratio_max2all'] = r
        col['base_cov'] = s
        col['base_freq'] = {'A': a, 'T': t, 'C': c, 'G': g, 'N': n}
    return base_stats


def _poly_dict(n_cov: int, ratio_low: np.ndarray, p_low: np.ndarray, pvalue):
    """polymorphism_rate's dict (cmseq/cmseq.py:430-456) from the number of covered columns and the ratio / p-value of the columns
    whose dominant base is under the threshold, in column order."""
    rv = {'total_covered_bases': n_cov, 'total_polymorphic_bases': 0}
    if n_cov == 0:
        return rv
    ratios = np.asarray(ratio_low)[np.asarray(p_low) < pvalue].tolist()
    rv['total_polymorphic_bases'] = len(ratios)
    rv['total_polymorphic_rate'] = float(len(ratios)) / float(n_cov)
    if ratios:
        rv['ratios'] = ratios
        rv['dominant_allele_distr_mean'] = np.mean(ratios)
        rv['dominant_allele_distr_sd'] = np.std(ratios)
        for pct in (10, 20, 30, 40, 50, 60, 70, 80, 90, 95, 98, 99):
            rv['dominant_allele_distr_perc_' + str(pct)] = np.percentile(ratios, pct)
    return rv


def _breadth_tuple(lo: int, hi: int, cols: np.ndarray, depths: np.ndarray):
    """breadth_and_depth_of_coverage's tuple (cmseq/cmseq.py:480-490) from the covered columns of the window [lo, hi) and their depths."""
    if len(cols) == 0:
        return (np.nan, np.nan, np.nan, [np.nan])
    depth_at = dict(zip(np.asarray(cols).tolist(), np.asarray(depths).tolist()))   # {0-based column: depth}, ascending like upstream's dict
    vals = list(depth_at.values())
    return (float(len(cols)) / (hi - lo), np.mean(vals), np.median(vals), depth_at.values())


_POLY_MASK_P = 0.05   # majority_rule_polymorphicLoci masks a column whose p-value is at most this (cmseq/cmseq.py:214)


def _check_depth_args(trimReads, min_read_depth):
    if trimReads:
        raise NotImplementedError("trimReads is not carried by the packed pileup stream")
    if min_read_depth < 1:
        # upstream divides by base_sum for every column htslib visits, covered by counted bases or not (cmseq/cmseq.py:554-555)
        raise ValueError("min_read_depth must be >= 1")


class BamContig:
    coverage = None
    consensus = ''
    name = None
    length = None
    stepper = 'nofilter'
    annotations = None

    def __init__(self, bamHandle: "BamFile", contigName: str, contigLength: int, stepper: str = 'nofilter'):
        self.name = contigName
        self.length = contigLength
        self.bam_handle = bamHandle
        self.stepper = stepper
        self.annotations = []

    def set_stepper(self, ns):
        if ns in ['all', 'nofilter']:
            self.stepper = ns

    # Consensus rules (cmseq/cmseq.py:202-224).  Upstream takes `max(sorted(freq), key=freq.get)`: the keys sort to A, C, G, N, T and
    # max() keeps the first maximum, so ties resolve A > C > G > N > T and N competes with the bases (H8).  Written out here as
    # the scan it amounts to.  They are plain functions in the class body, as upstream, so `consensus_rule=BamContig.majority_rule`
    # and calling `rule(column)` both work.
    _TIE_ORDER = ("A", "C", "G", "N", "T")

    def _first_maximum(freq) -> str:
        best, best_n = None, None
        for base in BamContig._TIE_ORDER:
            if base in freq and (best is None or freq[base] > best_n):
                best, best_n = base, freq[base]
        return best

    def majority_rule(data_array):
        freq = data_array['base_freq']
        return BamContig._first_maximum(freq) if max(freq.values()) > 0 else 'N'

    def majority_rule_polymorphicLoci(data_array):
        if data_array['p'] <= _POLY_MASK_P:  # polymorphic under the binomial test: masked
            return "*"
        freq = data_array['base_freq']
        if max(n for base, n in freq.items() if base != 'N') > 0:
            return BamContig._first_maximum(freq)
        return 'N'

    def _check_stepper(self):
        if self.stepper != 'nofilter':
            raise NotImplementedError("stepper=%r: only 'nofilter' (what cmseq passes by default, cmseq/cmseq.py:40) is implemented" % (self.stepper,))

    def _counts(self, min_base_quality: int, BAM_tagFilter=None) -> np.ndarray:
        self._check_stepper()
        h = self.bam_handle
        soa, minscore, max_xm = h._stream(min_base_quality, BAM_tagFilter)
        return np.asarray(_contig_counts(h.ctx, soa, h._tid[self.name], minscore, max_xm))

    def get_base_stats(self, min_read_depth=CMSEQ_DEFAULTS.mincov, min_base_quality=CMSEQ_DEFAULTS.minqual, error_rate=CMSEQ_DEFAULTS.poly_error_rate,
                       dominant_frq_thrsh=CMSEQ_DEFAULTS.poly_dominant_frq_thrsh, BAM_tagFilter=None, trimReads=None):
        """cmseq/cmseq.py:507-569: {1-based position: {'p', 'ratio_max2all', 'base_cov', 'base_freq': {'A','T','C','G','N'}}} for
        the columns whose A+C+G+T count reaches min_read_depth, in ascending position order."""
        _check_depth_args(trimReads, min_read_depth)
        counts = self._counts(min_base_quality, BAM_tagFilter)
        cols, _depth = _selected(counts, min_read_depth)
        c5 = counts[cols]
        return _base_stats_dict(cols, c5, *_column_stats(c5, dominant_frq_thrsh, error_rate))

    def reference_free_consensus(self, consensus_rule=majority_rule, mincov=CMSEQ_DEFAULTS.mincov, minqual=CMSEQ_DEFAULTS.minqual,
                                 dominant_frq_thrsh=CMSEQ_DEFAULTS.poly_dominant_frq_thrsh, noneCharacter='-', BAM_tagFilter=None, trimReads=None):
        """cmseq/cmseq.py:226-241: the rule's call for every column that has statistics, `noneCharacter` elsewhere; the string is
        also kept in `self.consensus`."""
        stats = self.get_base_stats(min_read_depth=mincov, min_base_quality=minqual, dominant_frq_thrsh=dominant_frq_thrsh,
                                    BAM_tagFilter=BAM_tagFilter, trimReads=trimReads, error_rate=CMSEQ_DEFAULTS.poly_error_rate)
        calls = [noneCharacter] * self.length
        for pos1, column in stats.items():
            calls[pos1 - 1] = consensus_rule(column)
        self.consensus = ''.join(calls)
        return self.consensus

    def polymorphism_rate(self, mincov=CMSEQ_DEFAULTS.mincov, minqual=CMSEQ_DEFAULTS.minqual, pvalue=CMSEQ_DEFAULTS.poly_pvalue_threshold,
                          error_rate=CMSEQ_DEFAULTS.poly_error_rate, dominant_frq_thrsh=CMSEQ_DEFAULTS.poly_dominant_frq_thrsh):
        """cmseq/cmseq.py:430-456: a column is polymorphic when its p-value is under `pvalue` AND its dominant base is under
        `dominant_frq_thrsh`; the distribution keys appear only when there is at least one such column (same keys, same order)."""
        _check_depth_args(None, mincov)
        counts = self._counts(minqual)
        cols, _depth = _selected(counts, mincov)
        _cov, ratio, low, p = _column_stats(counts[cols], dominant_frq_thrsh, error_rate)
        return _poly_dict(len(cols), ratio[low], p[low], pvalue)

    def breadth_and_depth_of_coverage(self, mincov=10, minqual=30, trunc=0):
        """cmseq/cmseq.py:459-490.  Upstream calls pileup() WITHOUT min_base_quality, so pysam's default 13 drops reads first
        and the loop then asks for quality >= minqual: the effective threshold is max(13, minqual); N bases and deletions do
        not count; no tag filter."""
        if mincov < 1:
            raise ValueError("mincov must be >= 1")
        lo, hi = _window(self.length, trunc)
        counts = self._counts(max(PYSAM_DEFAULT_MIN_BASE_QUALITY, int(minqual)))
        return _breadth_tuple(lo, hi, *_selected(counts, mincov, lo, hi))

    def depth_of_coverage(self, mincov=10, minqual=30):
        return self.breadth_and_depth_of_coverage(mincov, minqual)[1]

    def breadth_of_coverage(self, mincov=10, minqual=30):
        return self.breadth_and_depth_of_coverage(mincov, minqual)[0]

    def get_all_base_values(self, stats_value, *f_args, **f_kwargs):
        """cmseq/cmseq.py:572-578."""
        base_stats = self.get_base_stats(*f_args, **f_kwargs)
        return [base_stats[k].get(stats_value, 'NaN') for k in base_stats]


def _wanted_contigs(spec):
    """cmseq/cmseq.py:58-66: `filterInputList` is a list of contig names, the path of a FASTA file (its record ids: first word of every
    '>' line), or a comma-separated string.  None = no filter."""
    if spec is None:
        return None
    if isinstance(spec, list):
        return set(spec)
    if os.path.isfile(spec):
        with open(spec, "r") as fh:
            heads = (ln[1:].split() for ln in fh if ln.startswith(">"))
            return {h[0] if h else "" for h in heads}
    return set(spec.split(","))


class BaseStatsArrays(NamedTuple):
    """`BamFile.base_stats_arrays`: get_base_stats of every contig in columnar form.  Contig i (`names[i]`) owns the columns
    offsets[i] .. offsets[i+1]; per covered column the 1-based position, the counts (A, C, G, T, N), A+C+G+T, the dominant base's share, whether
    that share is under dominant_frq_thrsh (the columns the binomial test ran on) and p (1.0 where it did not run)."""
    names: List[str]
    offsets: np.ndarray
    pos: np.ndarray
    counts: np.ndarray
    base_cov: np.ndarray
    ratio_max2all: np.ndarray
    low: np.ndarray
    p: np.ndarray


DEFAULT_COL_BUDGET = 1 << 26   # columns per batch: 1.3 GB of counts on the device, and at most as many compacted columns back


class BamFile:
    """cmseq/cmseq.py:35-88.  `sort` / `index` are accepted and need nothing: the unpacker puts the records in
    `samtools sort` order in memory and the pileup needs no `.bai` (no `.sorted` / `.bai` files are written)."""
    bam_handle = None
    bamFile = None
    contigs = {}

    def __init__(self, bamFile, sort=False, index=False, stepper='nofilter', minlen=CMSEQ_DEFAULTS.minlen, filterInputList=None,
                 minimumReadsAligning=None, ctx: Optional[native.Context] = None, device: int = 0, minqual: int = CMSEQ_DEFAULTS.minqual):
        if not os.path.isfile(bamFile):
            raise Exception(bamFile + ' is not accessible, or is not a file')
        self.bamFile = bamFile
        self.bam_handle = self
        self._own_ctx = ctx is None
        self.ctx = ctx if ctx is not None else native.Context(device)
        self._soas: Dict[int, object] = {}
        first = self._soa(int(minqual))  # header + the streams of the most likely threshold
        self.references = tuple(first.ref_names)
        self.lengths = tuple(int(x) for x in first.ref_lens)
        self._tid = {r: i for i, r in enumerate(self.references)}
        keep = _wanted_contigs(filterInputList)  # upstream scans a list per reference (O(n_ref x n)); a set gives the same answer
        n_on = np.bincount(np.asarray(first.tid, dtype=np.int64), minlength=len(self.references)) if minimumReadsAligning else None
        self.contigs = dict((r, BamContig(self, r, l, stepper)) for i, (r, l) in enumerate(zip(self.references, self.lengths))
                            if l > minlen and (keep is None or r in keep) and (not minimumReadsAligning or int(n_on[i]) >= minimumReadsAligning))

    def _stream(self, min_base_quality, BAM_tagFilter=None):
        """(pileup stream at min_base_quality, minscore, max_xm) of a call with this tag filter."""
        minscore, max_xm = _tag_filter(BAM_tagFilter)
        soa = self._soa(int(min_base_quality))
        if BAM_tagFilter and getattr(soa, "n_untagged", 0):
            # pysam's get_tag raises for the first read without the tag (cmseq/cmseq.py:545); the unpacker counts such reads per FILE, so this is
            # raised for any contig of a file that holds one -- stricter than upstream, never silently different
            raise KeyError("tag 'AS' / 'XM' not present in %d pileup records of %s: a BAM_tagFilter cannot be evaluated (cmseq/cmseq.py:545)" % (soa.n_untagged, self.bamFile))
        return soa, minscore, max_xm

    def _soa(self, minqual: int):
        s = self._soas.get(minqual)
        if s is None:
            s = self._soas[minqual] = bam_mod.unpack_bam(self.bamFile, minqual=minqual, want_qhash=False, lenient_tags=True)
        return s

    def get_contigs(self):
        return iter(self.contigs.keys())

    def get_contigs_obj(self):
        return iter(self.contigs.values())

    def get_contig_by_label(self, contigID):
        return (self.contigs[contigID] if contigID in self.contigs else None)

    # ---- whole-BAM methods: every contig the handle keeps (or `contigs`, a subset of them), in header order ----------------------------
    def _bulk(self, contigs, min_base_quality, BAM_tagFilter, mode, mincov, trunc, dominant_frq_thrsh, none_char, want_cons, col_budget):
        """(contig, n selected, columns, values, consensus bytes or None) per contig, header order.  Contigs are cut into batches of
        consecutive kept contigs under `col_budget` columns (a longer contig runs alone, none is split); contigs without pileup records need
        no launch and give the empty form."""
        if contigs is None:
            chosen = list(self.contigs.values())
        else:
            missing = [c for c in contigs if c not in self.contigs]
            if missing:
                raise KeyError("contigs not kept by this BamFile: %r" % (missing[:5],))
            wanted = set(contigs)
            chosen = [c for name, c in self.contigs.items() if name in wanted]
        for c in chosen:
            c._check_stepper()
        soa, minscore, max_xm = self._stream(min_base_quality, BAM_tagFilter)
        prm = native.ContigStatsParams(mode, min(int(math.ceil(mincov)), 0xFFFFFFFF), int(trunc), none_char, float(dominant_frq_thrsh))
        width = _WIDTH[mode]
        empty = (0, np.zeros(0, np.int64), np.zeros((0, width), np.uint32), None)
        cs = np.asarray(soa.contig_start, dtype=np.int64)
        budget = max(1, min(int(col_budget), native.CONTIG_STATS_MAX_COLS))
        batch: List[BamContig] = []
        n_cols = 0

        def run(batch):
            tids = [self._tid[c.name] for c in batch]
            col_off = np.zeros(len(batch) + 1, np.uint32)
            col_off[1:] = np.cumsum([c.length for c in batch], dtype=np.uint64)   # a batch past 2^32 columns is one contig, refused by the library
            if int(sum(c.length for c in batch)) > native.CONTIG_STATS_MAX_COLS:
                raise native.MmlstError(native.E_RANGE, "contig %s has %d columns, one batch holds at most %d (5 * column in 32 bits)"
                                        % (batch[0].name, batch[0].length, native.CONTIG_STATS_MAX_COLS))
            r = _bulk_stats(self.ctx, soa, tids, col_off, minscore, max_xm, prm, want_cons)
            out_off = r.low_off if mode == native.STATS_LOWDOM else r.sel_off
            for i, c in enumerate(batch):
                a, b = int(out_off[i]), int(out_off[i + 1])
                yield c, int(r.sel_off[i + 1]) - int(r.sel_off[i]), r.cols[a:b], r.vals[a:b], \
                    (r.cons[col_off[i]:col_off[i + 1]] if want_cons else None)

        for c in chosen:
            if cs[self._tid[c.name] + 1] <= cs[self._tid[c.name]]:
                if batch:
                    yield from run(batch)
                    batch, n_cols = [], 0
                yield (c,) + empty
                continue
            if batch and n_cols + c.length > budget:
                yield from run(batch)
                batch, n_cols = [], 0
            batch.append(c)
            n_cols += c.length
        if batch:
            yield from run(batch)

    def base_stats_arrays(self, min_read_depth=CMSEQ_DEFAULTS.mincov, min_base_quality=CMSEQ_DEFAULTS.minqual, error_rate=CMSEQ_DEFAULTS.poly_error_rate,
                          dominant_frq_thrsh=CMSEQ_DEFAULTS.poly_dominant_frq_thrsh, BAM_tagFilter=None, trimReads=None, contigs=None,
                          col_budget=DEFAULT_COL_BUDGET) -> BaseStatsArrays:
        """`get_base_stats` of every contig in columnar form (BaseStatsArrays): what a caller that walks millions of columns should use."""
        _check_depth_args(trimReads, min_read_depth)
        names, offs, cols, c5s = [], [0], [], []
        for c, _n, col, vals, _cons in self._bulk(contigs, min_base_quality, BAM_tagFilter, native.STATS_COLUMNS, min_read_depth, 0,
                                                  dominant_frq_thrsh, 0, False, col_budget):
            names.append(c.name)
            offs.append(offs[-1] + len(col))
            cols.append(np.asarray(col, dtype=np.int64))
            c5s.append(vals)
        col = np.concatenate(cols) if cols else np.zeros(0, np.int64)
        c5 = np.concatenate(c5s) if c5s else np.zeros((0, 5), np.uint32)
        cov, ratio, low, p = _column_stats(c5, dominant_frq_thrsh, error_rate)
        return BaseStatsArrays(names, np.asarray(offs, dtype=np.int64), col + 1, c5, cov, ratio, low, p)

    def base_stats_all(self, min_read_depth=CMSEQ_DEFAULTS.mincov, min_base_quality=CMSEQ_DEFAULTS.minqual, error_rate=CMSEQ_DEFAULTS.poly_error_rate,
                       dominant_frq_thrsh=CMSEQ_DEFAULTS.poly_dominant_frq_thrsh, BAM_tagFilter=None, trimReads=None, contigs=None,
                       col_budget=DEFAULT_COL_BUDGET):
        """{contig: BamContig.get_base_stats(...)} for every kept contig (or `contigs`), header order."""
        a = self.base_stats_arrays(min_read_depth, min_base_quality, error_rate, dominant_frq_thrsh, BAM_tagFilter, trimReads, contigs, col_budget)
        out = {}
        for i, name in enumerate(a.names):
            s = slice(int(a.offsets[i]), int(a.offsets[i + 1]))
            out[name] = _base_stats_dict(a.pos[s] - 1, a.counts[s], a.base_cov[s], a.ratio_max2all[s], a.low[s], a.p[s])
        return out

    def reference_free_consensus_all(self, consensus_rule=BamContig.majority_rule, mincov=CMSEQ_DEFAULTS.mincov, minqual=CMSEQ_DEFAULTS.minqual,
                                     dominant_frq_thrsh=CMSEQ_DEFAULTS.poly_dominant_frq_thrsh, noneCharacter='-', BAM_tagFilter=None,
                                     trimReads=None, contigs=None, col_budget=DEFAULT_COL_BUDGET):
        """{contig: BamContig.reference_free_consensus(...)} for every kept contig (or `contigs`), header order; also sets each contig's
        `.consensus`.  Only the module's two rules run on the device (the majority call of the consensus kernel; the '*' of
        majority_rule_polymorphicLoci from the host p-value of the low-dominance columns)."""
        masked = consensus_rule is BamContig.majority_rule_polymorphicLoci
        if not masked and consensus_rule is not BamContig.majority_rule:
            raise NotImplementedError("consensus_rule %r: only BamContig.majority_rule and BamContig.majority_rule_polymorphicLoci run on the device"
                                      % (consensus_rule,))
        _check_depth_args(trimReads, mincov)
        one = isinstance(noneCharacter, str) and len(noneCharacter) == 1 and 0 < ord(noneCharacter) < 256
        out = {}
        for c, _n, col, vals, cons in self._bulk(contigs, minqual, BAM_tagFilter, native.STATS_LOWDOM, mincov, 0, dominant_frq_thrsh,
                                                 ord(noneCharacter) if one else 0, True, col_budget):
            if cons is None:   # no pileup record: nothing is recorded
                seq = noneCharacter * c.length
            else:
                if masked and len(col):
                    p = _pvalues(vals[:, 0], vals[:, 1], CMSEQ_DEFAULTS.poly_error_rate)
                    cons = cons.copy()
                    cons[np.asarray(col, dtype=np.int64)[p <= _POLY_MASK_P]] = ord('*')
                seq = cons.tobytes().decode("latin-1")
                if not one:   # calls are never NUL: the unrecorded columns
                    seq = seq.replace('\0', noneCharacter)
            c.consensus = seq
            out[c.name] = seq
        return out

    def polymorphism_rate_all(self, mincov=CMSEQ_DEFAULTS.mincov, minqual=CMSEQ_DEFAULTS.minqual, pvalue=CMSEQ_DEFAULTS.poly_pvalue_threshold,
                              error_rate=CMSEQ_DEFAULTS.poly_error_rate, dominant_frq_thrsh=CMSEQ_DEFAULTS.poly_dominant_frq_thrsh, contigs=None,
                              col_budget=DEFAULT_COL_BUDGET):
        """{contig: BamContig.polymorphism_rate(...)} for every kept contig (or `contigs`), header order."""
        _check_depth_args(None, mincov)
        out = {}
        for c, n_cov, _col, vals, _cons in self._bulk(contigs, minqual, None, native.STATS_LOWDOM, mincov, 0, dominant_frq_thrsh, 0, False, col_budget):
            out[c.name] = _poly_dict(n_cov, _ratios(vals[:, 0], vals[:, 1]), _pvalues(vals[:, 0], vals[:, 1], error_rate), pvalue)
        return out

    def breadth_and_depth_of_coverage_all(self, mincov=10, minqual=30, trunc=0, contigs=None, col_budget=DEFAULT_COL_BUDGET):
        """{contig: BamContig.breadth_and_depth_of_coverage(...)} for every kept contig (or `contigs`), header order.  `trunc` must be a
        non-negative integer here."""
        if mincov < 1:
            raise ValueError("mincov must be >= 1")
        if int(trunc) != trunc or trunc < 0 or trunc > 0xFFFFFFFF:
            raise ValueError("trunc must be an integer in 0 .. 2^32 - 1")
        out = {}
        for c, _n, col, vals, _cons in self._bulk(contigs, max(PYSAM_DEFAULT_MIN_BASE_QUALITY, int(minqual)), None, native.STATS_DEPTH, mincov,
                                                  int(trunc), 0.0, 0, False, col_budget):
            lo, hi = _window(c.length, int(trunc))
            out[c.name] = _breadth_tuple(lo, hi, col, vals[:, 0])
        return out

    def close(self):
        if self._own_ctx and self.ctx is not None:
            self.ctx.close()
        self.ctx = None
        self._soas.clear()
