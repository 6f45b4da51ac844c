"""TEST INFRASTRUCTURE ONLY -- CPU restatement ("Leg A", SURVEY.md 8c) of MetaMLST's post-alignment hot path.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this module;
it is the checker, never the product.  Pure Python, record-at-a-time, written to be read next to the reference:
every function cites the reference lines it follows (paths relative to /root/reference).

PARITY STATUS
  * In-tree Python lines (stage 1, selection, buildConsensus driver, majority rule, .nfo/.out formatting, merge
    classification, stringDiff, defineProfile): PINNED -- oracle/make_golden.py runs the reference's unmodified
    scripts over import shims (oracle/shims) and tests/test_oracle_golden.py compares this module to those
    outputs byte for byte.
  * The pileup ENGINE below (`PileupEngine`: htslib bam_plp_push/bam_plp_next + pysam's min_base_quality skip)
    lives in pysam/htslib, which are third-party, un-vendored and un-pinned in the reference (cmseq/README.md:7-12
    asks for "pysam", no version) and absent from this image.  It is restated from the published htslib
    algorithm (sam.c, htslib >= 1.10) and pysam >= 0.15 (libcalignedsegment.pyx `pileup_base_qual_skip`); the
    reference ships no test or golden vector for it => "parity unpinned" for H1-H3 (SURVEY.md 8).
"""
from __future__ import annotations

import sqlite3
from typing import Dict, Iterable, Iterator, List, Optional, Sequence, Tuple

from .bamio import BamHeader, BamRecord

BAM_FUNMAP = 0x4
BAM_FPROPER_PAIR = 0x2
HTS_MAX_DEPTH_DEFAULT = 8000  # pysam AlignmentFile.pileup(max_depth=8000) default -> bam_mplp_set_maxcnt (H1)


# ------------------------------------------------------------------------------------------------
# Stage 1: metamlst.py:101-151
# ------------------------------------------------------------------------------------------------

def _positional_int(aux, k: int) -> int:
    """`int(read[11+k].split(':')[2])` (metamlst.py:109-110): the k-th aux field BY POSITION, whatever its tag
    (H4).  samtools prints every integer aux type as `:i:`; a non-integer field makes `int()` raise ValueError and
    a missing field IndexError -- both kill the reference run, so both raise here."""
    tag, typ, val = aux[k]  # IndexError like the reference
    if typ not in "cCsSiI":
        raise ValueError("invalid literal for int(): aux field %d is %s:%s" % (k, tag, typ))
    return int(val)


def stage1(header: BamHeader, records: Iterable[BamRecord], minscore: int = 80, max_xM: int = 5,
           min_read_len: int = 50, species_filter: Optional[str] = None, penalty: int = 100):
    """Returns (cel, sequenceBank, totalReads, ignoredReads) exactly as metamlst.py holds them at line 152.
    cel[species][gene][allele] = (localScore, n, round(avg, 1)); dict order = first passing record (H5)."""
    cel: Dict[str, Dict[str, Dict[str, object]]] = {}
    sequenceBank: Dict[str, Dict[str, int]] = {}
    ignoredReads = 0
    totalReads = 0
    for r in records:  # metamlst.py:101-104 (header lines skipped)
        rname = header.ref_names[r.tid] if r.tid >= 0 else "*"
        species, gene, allele = rname.split("_")  # :107 -- ValueError for '*' or a 2-/4-part name, as upstream
        score = _positional_int(r.aux, 0)  # :109
        xM = _positional_int(r.aux, 3)  # :110
        sequence = r.seq if len(r.seq) else "*"  # SAM column 10 is '*' when l_seq == 0
        if (species_filter and species in species_filter.split(",")) or not species_filter:  # :114
            if score >= minscore and len(sequence) >= min_read_len and xM <= max_xM:  # :115
                if species not in cel:
                    cel[species] = {}
                if gene not in cel[species]:
                    cel[species][gene] = {}
                    sequenceBank[species + "_" + gene] = {}
                if allele not in cel[species][gene]:
                    cel[species][gene][allele] = []
                cel[species][gene][allele].append(score)  # :125
                sequenceBank[species + "_" + gene][r.qname] = len(sequence)  # :127 (H7: last wins)
            else:
                ignoredReads += 1
            totalReads += 1
    for speciesKey, species in cel.items():  # :133-151
        for geneKey, geneInfo in species.items():
            maxLen = max(len(x) for x in geneInfo.values())
            for alleleCode, values in geneInfo.items():
                geneLen = len(values)
                localScore = sum(values)
                if geneLen != maxLen:
                    localScore = localScore - (maxLen - geneLen) * penalty
                averageScore = float(localScore) / float(geneLen)
                geneInfo[alleleCode] = (localScore, geneLen, round(averageScore, 1))  # H6
    return cel, sequenceBank, totalReads, ignoredReads


def out_log_rows(cel) -> List[str]:
    """Result rows of the --log .out file, metamlst.py:168-171."""
    rows = []
    for speciesKey, species in cel.items():
        for geneKey, geneInfo in species.items():
            for k, (score, geneLen, average) in sorted(geneInfo.items(), key=lambda x: x[1]):
                rows.append("\t".join(map(str, [speciesKey, geneKey, k, score, geneLen, average])) + "\r\n")
    return rows


def select_alleles(species_cel: Dict[str, Dict[str, tuple]]) -> List[Tuple[str, str]]:
    """metamlst.py:244 -- per locus (dict order) the alleles whose rounded avg equals the max, lowest int(allele)."""
    out = []
    for g1, g2 in species_cel.items():
        best = max(avg for (_v, _l, avg) in g2.values())
        cands = sorted((k for k, (_v, _l, avg) in g2.items() if avg == best), key=lambda x: int(x))
        out.append((g1, cands[0]))
    return out


def locus_table(species_cel, sequenceBank, speciesKey: str, db_max_len) -> List[tuple]:
    """metamlst.py:213-230: (gene, coverage, best avg, hits, closeAllelesList) per locus sorted by name."""
    rows = []
    for geneKey, geneInfo in sorted(species_cel.items(), key=lambda x: x[0]):
        minValue = max(avg for (_v, _l, avg) in geneInfo.values())
        aElements = {k: t for k, t in geneInfo.items() if t[2] == minValue}
        close = ",".join([str(a) for a in sorted(aElements.keys(), key=lambda x: int(x))][:5]) + \
                ("... (" + str(len(aElements)) + " more)" if len(aElements) > 5 else "")
        genL = db_max_len(speciesKey, geneKey)
        coverage = sum(sequenceBank[speciesKey + "_" + geneKey].values())
        rows.append((geneKey, round(float(coverage) / float(genL), 2), minValue, list(aElements.values())[0][1], close))
    return rows


# ------------------------------------------------------------------------------------------------
# Pileup engine: htslib bam_plp_push / bam_plp_next (sam.c) + pysam column.pileups  -- H1, H2, H3
# ------------------------------------------------------------------------------------------------

def resolve_record(r: BamRecord) -> List[Tuple[int, int]]:
    """For every reference offset covered by the record: (qpos, kind), kind 0 = M/=/X base, 1 = deletion (D),
    2 = reference skip (N).  htslib resolve_cigar2: M/=/X consume ref+query; I,S query only; D,N ref only; H,P
    nothing; qpos indexes the full SEQ including soft clips; for D/N qpos is the query index of the next base."""
    out = []
    y = 0
    for op, l in r.cigar:
        if op in (0, 7, 8):
            out.extend((y + i, 0) for i in range(l))
            y += l
        elif op in (1, 4):
            y += l
        elif op == 2:
            out.extend((y, 1) for _ in range(l))
        elif op == 3:
            out.extend((y, 2) for _ in range(l))
    return out


class PileupEngine:
    """State machine of htslib's pileup iterator for ONE contig fetch (pysam `AlignmentFile.pileup(contig,
    stepper='nofilter')`, cmseq/cmseq.py:527): records must arrive coordinate-sorted.

    push (bam_plp_push): unmapped-flag records are skipped; a record is DROPPED when its start equals the
    iterator's current column and the mempool count exceeds maxcnt (`iter->tid == b->core.tid && iter->pos ==
    b->core.pos && iter->mp->cnt > iter->maxcnt`); mp->cnt counts live buffered records + the tail sentinel
    (htslib >= 1.10 allocates no `dummy` node; older samtools had one more).  A record whose end <= pos is not
    linked.  next (bam_plp_next): emits column `pos` once a record starting beyond it has been pushed (or at
    EOF), freeing records with end <= pos during the scan.
    """

    def __init__(self, tid: int, maxcnt: int = HTS_MAX_DEPTH_DEFAULT, sentinel_nodes: int = 1):
        self.maxcnt = maxcnt
        self.buf: List[tuple] = []  # (beg, end, record, resolved, index)
        self.cnt = sentinel_nodes  # iter->head = iter->tail = mp_alloc()
        self.iter_tid = 0  # calloc'ed iterator
        self.iter_pos = 0
        self.max_tid = -1
        self.max_pos = -1
        self.is_eof = False
        self.tid = tid
        self.dropped: List[int] = []
        self.admitted: List[int] = []

    def push(self, r: Optional[BamRecord], index: int = -1) -> None:
        if r is None:
            self.is_eof = True
            return
        if r.tid < 0 or (r.flag & BAM_FUNMAP):
            return
        if self.iter_tid == r.tid and self.iter_pos == r.pos and self.cnt > self.maxcnt:
            self.dropped.append(index)
            return
        beg = r.pos
        end = r.pos + r.ref_len()  # raw rlen (bam_cigar2rlen), not bam_endpos
        if r.tid < self.max_tid or (r.tid == self.max_tid and beg < self.max_pos):
            raise ValueError("The input is not sorted (reads out of order)")
        self.max_tid, self.max_pos = r.tid, beg
        self.admitted.append(index)
        if end > self.iter_pos or r.tid > self.iter_tid:
            self.buf.append((beg, end, r, resolve_record(r), index))
            self.cnt += 1  # next = mp_alloc()

    def next(self):
        """One bam_plp_next call: returns (pos, [(record, qpos, kind)]) or None when more input is needed."""
        while self.is_eof or self.max_tid > self.iter_tid or (self.max_tid == self.iter_tid and self.max_pos > self.iter_pos):
            if self.is_eof and not self.buf:
                return None
            plp = []
            keep = []
            for node in self.buf:
                beg, end, r, res, _ = node
                if r.tid < self.iter_tid or (r.tid == self.iter_tid and end <= self.iter_pos):
                    self.cnt -= 1  # mp_free
                    continue
                keep.append(node)
                if r.tid == self.iter_tid and beg <= self.iter_pos:
                    qpos, kind = res[self.iter_pos - beg]
                    plp.append((r, qpos, kind))
            self.buf = keep
            col = (self.iter_tid, self.iter_pos)
            if self.buf:
                head = self.buf[0]
                if self.iter_tid < head[2].tid:
                    self.iter_tid, self.iter_pos = head[2].tid, head[0]
                elif self.iter_pos < head[0]:
                    self.iter_pos = head[0]
                else:
                    self.iter_pos += 1
            else:
                self.iter_pos += 1
            if plp:
                return col[1], plp
            if self.is_eof and not self.buf:
                break
        return None

    def columns(self, records: Sequence[BamRecord]) -> Iterator[Tuple[int, list]]:
        """bam_plp_auto: drain `next` before reading another record."""
        i = 0
        n = len(records)
        while True:
            col = self.next()
            if col is not None:
                yield col
                continue
            if self.is_eof:
                return
            if i < n:
                self.push(records[i], i)
                i += 1
            else:
                self.push(None)


def refuse_proper_pairs(records: Iterable[BamRecord]) -> None:
    """H2: pysam's default ignore_overlaps=True edits qualities of overlapping PROPER-PAIR mates.  MetaMLST's
    documented workflow aligns reads unpaired; neither this oracle nor the product implements the overlap rule, and
    both refuse loudly instead of silently differing."""
    for r in records:
        if r.flag & BAM_FPROPER_PAIR:
            raise NotImplementedError("proper-pair record %s: htslib overlap handling (H2) is not restated" % r.qname)


def get_base_stats(contig_records: Sequence[BamRecord], tid: int, min_read_depth: int = 1, min_base_quality: int = 30,
                   tag_filter: Optional[Sequence[Tuple[str, str, int]]] = None, max_depth: int = HTS_MAX_DEPTH_DEFAULT):
    """cmseq/cmseq.py:507-569 without the output-dead p / ratio (SURVEY 3.2): {pos1: {'base_cov', 'base_freq'}}.

    column.pileups omits reads whose base quality at qpos is < min_base_quality (pysam pileup_base_qual_skip: a
    qpos beyond l_qseq counts as quality 0) -- H3.  Tag predicates are by NAME (H4): a missing tag raises KeyError
    like pysam get_tag."""
    ops = {"loc_gte": lambda a, b: a >= b, "loc_lte": lambda a, b: a <= b, "loc_gt": lambda a, b: a > b,
           "loc_lt": lambda a, b: a < b, "loc_leq": lambda a, b: a == b}  # cmseq.py:582-595
    eng = PileupEngine(tid, max_depth)
    base_stats = {}
    for pos0, plp in eng.columns(contig_records):
        base_freq = {"A": 0, "T": 0, "C": 0, "G": 0, "N": 0}
        for r, qpos, kind in plp:
            c = r.qual[qpos] if (r.qual and qpos < len(r.seq)) else (255 if (not r.qual and qpos < len(r.seq)) else 0)
            if c < min_base_quality:
                continue  # not in column.pileups at all
            if kind != 0:
                continue  # is_del / is_refskip, cmseq.py:535
            b = r.seq[qpos].upper()
            this = "N"
            if b in ("A", "T", "C", "G"):
                if tag_filter is None or all(ops[f](_get_tag(r, tag), lim) for (tag, f, lim) in tag_filter):
                    this = b
            base_freq[this] += 1
        base_sum = sum(base_freq[b] for b in "ATCG")
        if base_sum >= min_read_depth:  # cmseq.py:554
            base_stats[pos0 + 1] = {"base_cov": base_sum, "base_freq": base_freq}
    return base_stats, eng


def _get_tag(r: BamRecord, tag: str):
    for t, _typ, v in r.aux:
        if t == tag:
            return v
    raise KeyError("tag '%s' not present" % tag)


def majority_rule(data_array) -> str:
    """cmseq/cmseq.py:202-209: `max(sorted(freq), key=freq.get)` => ties resolve A > C > G > N > T, N competes (H8)."""
    freq = data_array["base_freq"]
    if any(v > 0 for v in freq.values()):
        return max(sorted(freq), key=freq.get)
    return "N"


def reference_free_consensus(contig_records, tid: int, length: int, mincov: int = 1, minqual: int = 20,
                             none_char: str = "N", tag_filter=None, max_depth: int = HTS_MAX_DEPTH_DEFAULT) -> str:
    """cmseq/cmseq.py:226-241."""
    stats, _ = get_base_stats(contig_records, tid, mincov, minqual, tag_filter, max_depth)
    cons = {p: majority_rule(d) for p, d in stats.items()}
    if cons:
        return "".join(cons[p] if p in cons else none_char for p in range(1, length + 1))
    return none_char * length


class ConsRecord:
    """Plain stand-in for Bio.SeqRecord as buildConsensus' callers use it (metamlst.py:254-285)."""

    def __init__(self, seq: str, id: str, description: str):
        self.seq, self.id, self.description = seq, id, description


def build_consensus(header: BamHeader, sorted_records: Sequence[BamRecord], chromosome_list: Dict[str, str],
                    filter_score: int, max_xM: int, max_depth: int = HTS_MAX_DEPTH_DEFAULT) -> List[ConsRecord]:
    """metaMLST_functions.py:249-281.  `sorted_records` is the coordinate-sorted BAM content (after sort_index)."""
    refuse_proper_pairs(sorted_records)
    name2tid = {n: i for i, n in enumerate(header.ref_names)}
    by_tid: Dict[int, List[BamRecord]] = {}
    wanted = {name2tid[c] for c in chromosome_list if c in name2tid}
    for r in sorted_records:
        if r.tid in wanted:
            by_tid.setdefault(r.tid, []).append(r)
    out = []
    for chromo, dbSequen in chromosome_list.items():
        tid = name2tid[chromo]
        rSequen = list(reference_free_consensus(by_tid.get(tid, []), tid, header.ref_lens[tid], 1, 20, "N",
                                                [("AS", "loc_gte", filter_score), ("XM", "loc_lte", max_xM)], max_depth))
        cIndex = 0
        SNPs = 0
        for i, ch in enumerate(rSequen):
            if ch == "N":
                rSequen[i] = dbSequen[i].lower()  # IndexError if LN > len(db) as upstream (H10)
                cIndex += 1
            elif rSequen[i] != dbSequen[i]:
                SNPs += 1
        out.append(ConsRecord("".join(rSequen), chromo, "CI::" + str(cIndex) + "_SP::" + str(SNPs)))
    return out


# ------------------------------------------------------------------------------------------------
# Post-consensus accounting + .nfo line: metamlst.py:251-287
# ------------------------------------------------------------------------------------------------

def nfo_line(speciesKey: str, fileName: str, consenSeq: List[ConsRecord], min_accuracy: float, write_known: bool,
             sequence_find) -> Tuple[Optional[str], List[tuple]]:
    """Returns (line or None when the min_accuracy gate drops the organism, per-locus table rows)."""
    finWrite = 1
    rows = []
    for l in sorted(consenSeq, key=lambda x: x.id):
        holes = str(l.description.split("_")[0].split("::")[1])
        snps = int(l.description.split("_")[1].split("::")[1])
        leng = str(len(l.seq))
        leng_ns = str(round(1 - float(holes) / float(leng), 4) * 100) + " %"
        l.seqLen = len(l.seq)
        if (1 - float(holes) / float(leng)) <= min_accuracy:
            finWrite = 0
        if snps > 0:
            seqFind = sequence_find(speciesKey, l.seq)
            newAllele = seqFind if seqFind else "NEW"
        else:
            newAllele = "--"
            if not write_known:
                l.seq = ""
        rows.append((l.id, leng, holes, snps, leng_ns, newAllele))
    if not finWrite:
        return None, rows
    line = speciesKey + "\t" + fileName + "\t" + "\t".join(
        recd.id + "::" + str(recd.seq) + "::" + str(round(1 - float(recd.description.split("_")[0].split("::")[1]) / float(recd.seqLen), 4) * 100)
        + "::" + str(round(float(recd.description.split("_")[1].split("::")[1]) / float(recd.seqLen), 4) * 100) for recd in consenSeq) + "\r\n"
    return line, rows


class OracleDB:
    """The SQL lookups the path performs (metaMLST_functions.py:168-228), on the reference schema."""

    def __init__(self, path: str):
        self.conn = sqlite3.connect(path)
        self.conn.row_factory = sqlite3.Row

    def genes(self, bacterium: str) -> List[str]:  # metamlst.py:184
        return [r["geneName"] for r in self.conn.execute("SELECT geneName FROM genes WHERE bacterium = ?", (bacterium,))]

    def max_len(self, bacterium: str, gene: str) -> int:  # metamlst.py:225
        return self.conn.execute("SELECT MAX(LENGTH(sequence)) AS L FROM alleles WHERE bacterium = ? AND gene = ?", (bacterium, gene)).fetchone()["L"]

    def unal_sequence(self, bacterium: str, gene: str, allele: str):  # metaMLST_functions.py:186-194
        row = self.conn.execute("SELECT sequence FROM alleles WHERE bacterium = ? AND gene = ? AND alleleVariant = ?", (bacterium, gene, allele)).fetchone()
        return row["sequence"] if row is not None else None

    def sequence_find(self, bacterium: str, sequence: str):  # :196-203 (returns the GENE of the first exact match)
        row = self.conn.execute("SELECT gene FROM alleles WHERE sequence = ? AND bacterium = ?", (str(sequence), bacterium)).fetchone()
        return row["gene"] if row else 0

    def sequence_exists(self, bacterium: str, sequence: str) -> bool:  # :168-172
        return self.conn.execute("SELECT 1 FROM alleles WHERE sequence = ? AND bacterium = ?", (str(sequence), bacterium)).fetchone() is not None

    def sequence_locate(self, bacterium: str, sequence: str) -> str:  # :218-222
        return str(self.conn.execute("SELECT alleleVariant FROM alleles WHERE sequence = ? AND bacterium = ?", (str(sequence), bacterium)).fetchone()["alleleVariant"])

    def sequences_get_all(self, bacterium: str, gene: str) -> Dict[int, str]:  # :224-228
        return dict((r["alleleVariant"], r["sequence"]) for r in self.conn.execute(
            "SELECT sequence,alleleVariant FROM alleles WHERE gene = ? AND bacterium = ?", (gene, bacterium)))

    def define_profile(self, labels: Sequence[str]) -> List[Tuple[int, int]]:
        """metaMLST_functions.py:205-216 incl. its quirks (H11): unknown labels silently shrink the denominator;
        `[(0,0)]` only when the LAST lookup failed.  The ST statement is the reference's, verbatim: the order of tied profiles
        (`ORDER BY T DESC` leaves them in descending profileCode order in SQLite 3.x) is whatever that statement returns, and the
        merge takes the first of them."""
        recs = []
        result = None
        for label in labels:
            result = self.conn.execute("SELECT recID FROM alleles WHERE bacterium||'_'||gene||'_'||alleleVariant = ?", (label,)).fetchone()
            if result:
                recs.append(str(result["recID"]))
        if not result:
            return [(0, 0)]
        inl = ",".join(recs)
        q = ("SELECT profileCode, COUNT(*) as T FROM profiles WHERE alleleCode IN (" + inl + ") GROUP BY profileCode HAVING T = "
             "(SELECT COUNT(*) FROM profiles WHERE alleleCode IN (" + inl + ") GROUP BY profileCode ORDER BY COUNT(*) DESC LIMIT 1) ORDER BY T DESC")
        return [(row[0], int((float(row[1]) / float(len(recs))) * 100)) for row in self.conn.execute(q)]


def string_diff(s1: str, s2: str) -> int:
    """metaMLST_functions.py:230-234 (zip => compared over min(len), H9)."""
    c = 0
    for a, b in zip(s1, s2):
        if a != b:
            c += 1
    return c


def closest_allele(db: OracleDB, bacterium: str, gene: str, seq: str) -> Tuple[int, int]:
    """(min distance, alleleVariant of the first row reaching it in sequencesGetAll order) -- the quantity whose
    `<= z` test metamlst-merge.py:177-181 evaluates with an early exit."""
    best = (1 << 30, -1)
    for code, ref in db.sequences_get_all(bacterium, gene).items():
        d = string_diff(seq, ref)
        if d < best[0]:
            best = (d, code)
    return best


def type_sample(bam_header: BamHeader, records: Sequence[BamRecord], db: OracleDB, sample_name: str,
                minscore: int = 80, max_xM: int = 5, min_read_len: int = 50, min_accuracy: float = 0.90,
                nloci: int = 100, penalty: int = 100, species_filter: Optional[str] = None, write_known: bool = False,
                max_depth: int = HTS_MAX_DEPTH_DEFAULT, coord_sort=None):
    """metamlst.py:96-289 end to end on parsed records; returns dict with cel, counters, nfo lines, tables."""
    cel, bank, total, ignored = stage1(bam_header, records, minscore, max_xM, min_read_len, species_filter, penalty)
    if coord_sort is None:
        def coord_sort(recs):  # samtools sort (metaMLST_functions.py:244): stable by (tid, pos, reverse)
            return sorted(recs, key=lambda r: (r.tid, r.pos, (r.flag >> 4) & 1))
    sorted_records = None
    res = {"cel": cel, "total": total, "ignored": ignored, "nfo": [], "species": {}}
    for speciesKey, species in cel.items():  # :181
        tVar = dict((g, 0) for g in db.genes(speciesKey))
        if len(tVar) < len(species.keys()):
            res["broken"] = speciesKey
            break  # sys.exit(0) upstream
        for sk in species.keys():
            tVar[sk] = 1
        vals = sum(tVar.values())
        entry = {"detected": sorted(k for k, v in tVar.items() if v == 1), "missing": sorted(k for k, v in tVar.items() if v == 0)}
        res["species"][speciesKey] = entry
        if int((float(vals) / float(len(tVar))) * 100) >= nloci:  # :206
            entry["loci"] = locus_table(species, bank, speciesKey, db.max_len)
            if sorted_records is None:
                sorted_records = coord_sort(list(records))
            chosen = [(speciesKey + "_" + g + "_" + a, db.unal_sequence(speciesKey, g, a)) for g, a in select_alleles(species)]
            cons = build_consensus(bam_header, sorted_records, dict(chosen), minscore, max_xM, max_depth)
            entry["consensus"] = [(c.id, c.seq, c.description) for c in cons]
            line, rows = nfo_line(speciesKey, sample_name, cons, min_accuracy, write_known, db.sequence_find)
            entry["table"] = rows
            if line is not None:
                res["nfo"].append(line)
    return res


# ------------------------------------------------------------------------------------------------
# Cohort merge: metamlst-merge.py:93-292 (classification + ST table); report lines :298-340 without --meta
# ------------------------------------------------------------------------------------------------

def parse_nfo_folder(folder: str, species_filter: Optional[str] = None):
    """metamlst-merge.py:93-107 (os.listdir order, SEQ upper-cased)."""
    import os
    cel: Dict[str, list] = {}
    for file in os.listdir(folder):
        if file.split(".")[-1] != "nfo":
            continue
        for line in open(folder + "/" + file, "r"):
            organism = line.split()[0]
            sampleName = line.split()[1]
            genes = line.split()[2::]
            if species_filter and organism not in species_filter:
                continue
            cel.setdefault(organism, []).append(
                (dict((x.split("::")[0], (x.split("::")[1].upper(), x.split("::")[2], x.split("::")[3])) for x in genes), sampleName))
    return cel


def merge_bacterium(db: OracleDB, bacterium: str, bactRecord, z: Optional[int] = 5, closest=None):
    """metamlst-merge.py:121-239.  `closest(bacterium, gene, seq) -> (min_dist, allele)` replaces the early-exit
    loop :177-181 (flag = min_dist <= z); default = the stringDiff scan.  Returns the state the writers use."""
    conn = db.conn
    oldProfiles: Dict[int, list] = {}
    genesBase: Dict[str, str] = {}
    encounteredProfiles: Dict[int, list] = {}
    isolates = []
    newSequences: Dict[str, list] = {}
    lastProfile = 100000
    lastGenes = dict((row["gene"], 100000) for row in conn.execute(
        "SELECT gene, MAX(alleleVariant) as maxGene FROM alleles WHERE bacterium = ? GROUP BY gene", (bacterium,)))
    for row in conn.execute("SELECT profileCode,gene,alleleVariant FROM profiles,alleles WHERE alleleCode = alleles.recID AND alleles.bacterium = ?", (bacterium,)):
        if row["profileCode"] not in oldProfiles:
            oldProfiles[row["profileCode"]] = [0, {}]
        oldProfiles[row["profileCode"]][1][row["gene"]] = row["alleleVariant"]
    if closest is None:
        def closest(b, g, s):
            return closest_allele(db, b, g, s)
    for bacteriumLine, sampleRecord in bactRecord:
        profileLine = {}
        newAlleles = []
        flagRecurrent = False
        sum_of_accuracies = 0.0
        for geneLabel, (geneSeq, geneAccur, percent_snps) in bacteriumLine.items():
            geneOrganism, geneName, geneAllele = geneLabel.split("_")
            sum_of_accuracies += float(geneAccur)
            if geneSeq == "" or db.sequence_exists(bacterium, geneSeq):
                if geneSeq != "":
                    geneAllele = db.sequence_locate(bacterium, geneSeq)
                profileLine[geneName] = (geneAllele, 0)
            elif geneSeq in genesBase:
                profileLine[geneName] = (genesBase[geneSeq].split("_")[2], 2)
                flagRecurrent = True
            else:
                geneCategoryCode = 1
                if z is not None:
                    geneCategoryCode = 3
                    if closest(bacterium, geneName, geneSeq)[0] <= z:
                        geneCategoryCode = 1
                geneNewAlleleNumber = str(lastGenes[geneName] + 1)
                lastGenes[geneName] += 1
                geneNewLabel = geneOrganism + "_" + geneName + "_" + geneNewAlleleNumber
                genesBase[geneSeq] = geneNewLabel
                profileLine[geneName] = (geneNewAlleleNumber, geneCategoryCode)
                newAlleles.append(geneName)
                newSequences.setdefault(geneName, []).append((geneNewLabel, geneSeq))
        meanAccuracy = sum_of_accuracies / float(len(bacteriumLine))
        if len(newAlleles) == 0:
            if not flagRecurrent:
                tryDefine = db.define_profile([bacterium + "_" + k + "_" + v[0] for k, v in profileLine.items()])
                if tryDefine and tryDefine[0][1] == 100:
                    oldProfiles[tryDefine[0][0]][0] += 1
                    isolates.append((tryDefine[0][0], meanAccuracy, sampleRecord))
                    continue
            foundExistant = 0
            for key, (element, abundance, isNewProfile) in encounteredProfiles.items():
                if [k + str(v[0]) for k, v in sorted(profileLine.items())] == [k + str(v[0]) for k, v in sorted(element.items())]:
                    foundExistant = key
            if foundExistant:
                encounteredProfiles[foundExistant][1] += 1
                isolates.append((foundExistant, meanAccuracy, sampleRecord))
            else:
                lastProfile += 1
                encounteredProfiles[lastProfile] = [profileLine, 1, 2]
                isolates.append((lastProfile, meanAccuracy, sampleRecord))
        else:
            lastProfile += 1
            profileCategoryCode = 1
            if z is not None:
                for k, (v, cat) in profileLine.items():
                    if cat == 3:
                        profileCategoryCode = 3
                        break
            encounteredProfiles[lastProfile] = [profileLine, 1, profileCategoryCode]
            if profileCategoryCode != 3:
                isolates.append((lastProfile, meanAccuracy, sampleRecord))
    return {"oldProfiles": oldProfiles, "encounteredProfiles": encounteredProfiles, "isolates": isolates,
            "lastGenes": lastGenes, "newSequences": newSequences}


def st_table_text(state) -> str:
    """merged/<org>_ST.txt, metamlst-merge.py:253-277 (note the mixed \\r\\n / \\n line ends)."""
    out = "ST\t" + "\t".join(sorted(state["lastGenes"].keys())) + "\r\n"
    for profileCode, (hits, profile) in state["oldProfiles"].items():
        out += str(profileCode) + "\t" + "\t".join(str(v) for k, v in sorted(profile.items())) + "\r\n"
    for profileID, (profile, hits, code) in state["encounteredProfiles"].items():
        if code not in (1, 2):
            continue
        out += str(profileID) + "\t" + "\t".join(str(v[0]) for k, v in sorted(profile.items())) + "\n"
    return out


def report_text(state) -> str:
    """merged/<org>_report.txt without --meta, metamlst-merge.py:316-339."""
    out = "ST\tConfidence\t\n"
    for profileST, meanAccur, sampleName in state["isolates"]:
        if sampleName.endswith(".fna"):
            sampleName = sampleName.split(".")[0]
        out += str(profileST) + "\t" + str(round(meanAccur, 2)) + "\t" + str(sampleName) + "\n"
    return out
