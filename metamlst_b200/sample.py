"""Whole-sample and cohort driver (SURVEY.md 8f rank 2): what `metamlst.py` does between opening the BAM and closing the DB
(metamlst.py:85-299), with every per-record / per-base step on the GPU.

    typer = SampleTyper("db.sqlite", device=0)            # DB connection, GPU context and device tables stay open across samples
    res   = typer.type_bam("sample.bam", out_dir)         # appends out_dir/sample.nfo, optional .out log
    type_cohort(bams, "db.sqlite", out_dir, devices=[0, 1, ...])   # the implicit `for bam in cohort: metamlst.py bam`

Structure (not the reference's): a sample is first reduced to a list of `SpeciesCall`s -- one per organism of the score table, each
holding its `LocusCall`s (contig, consensus, holes, SNPs) -- by one of three engines:

  engine="device" (default)  BAM -> unpack -> streams.DeviceStreams.from_soa -> pipeline.DevicePipeline.step(): score, selection,
                             pileup and consensus are ONE chain of kernels with a single D2H of the result block; the score tables
                             leave the device only when the `.out` log or the screen text is asked for.  With torch.distributed
                             (one process per GPU) every rank types its record range of the same sample and the integer tables are
                             all-reduced (`mode="ranges"`): the ranks end with identical results, rank 0 writes the files.
  engine="onecall"           the sample stays in host memory: ONE library call per sample (api.type_soa -> mmlst_sample), only the chosen
                             contigs' pileup records cross the bus
  engine="host"              the four seams one by one through the host-buffer C-ABI (api.score_soa, api.build_consensus): the
                             path a maintainer gets by rebinding the reference's names (INTEGRATION.md).

and then rendered by pure functions into the three texts the reference emits: the `.nfo` line (metamlst.py:284-285, append mode,
'\\r\\n'), the `.out` log (:160-172) and the screen output (:176-296, colour escapes and coverage column included, returned as a
string, never printed).  Formatting uses the reference's own Python float / str operations so the bytes are identical (H6).
"""
from __future__ import annotations

import os
import queue
import sqlite3
import threading
import time
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

from . import api, bam, native

# terminal colours of the reference (metaMLST_functions.py: class bcolors)
HEADER, OKBLUE, OKGREEN, WARNING, FAIL, ENDC = "\033[95m", "\033[94m", "\033[92m", "\033[93m", "\033[91m", "\033[0m"


# ----------------------------------------------------------------------------------------------------------------
# the typed sample
# ----------------------------------------------------------------------------------------------------------------
@dataclass
class LocusCall:
    """One reconstructed locus: what buildConsensus returns per contig (metaMLST_functions.py:276) as plain fields."""
    contig: str            # organism_gene_allele of the chosen reference allele
    sequence: str          # consensus, holes filled with the lower-case DB base
    holes: int
    snps: int
    known_as: Optional[str] = None   # gene of an exact DB match when snps > 0 (screen note only, metamlst.py:264-269)

    @property
    def gene(self) -> str:
        return self.contig.split("_")[1]

    @property
    def allele(self) -> str:
        return self.contig.split("_")[2]

    @property
    def length(self) -> int:
        return len(self.sequence)

    def completeness(self) -> float:       # metamlst.py:258,261
        return 1 - float(self.holes) / float(self.length)

    def confidence_text(self) -> str:      # metamlst.py:258,285 (H6)
        return str(round(self.completeness(), 4) * 100)

    def snp_text(self) -> str:             # metamlst.py:285
        return str(round(float(self.snps) / float(self.length), 4) * 100)

    def nfo_field(self, write_known: bool) -> str:
        seq = self.sequence if (self.snps > 0 or write_known) else ""   # metamlst.py:271-273
        return self.contig + "::" + seq + "::" + self.confidence_text() + "::" + self.snp_text()


@dataclass
class SpeciesCall:
    species: str
    db_genes: List[str]                    # rows of `genes` for the organism (metamlst.py:184)
    detected: List[str]                    # loci with at least one passing record, score-table order (H5)
    passed_gate: bool = False              # --nloci
    loci: List[LocusCall] = field(default_factory=list)   # chosen loci in score-table order (= chromosomeList order)

    def accepted(self, min_accuracy: float) -> bool:
        """metamlst.py:261: one locus at or under min_accuracy discards the organism for this sample."""
        return all(l.completeness() > min_accuracy for l in self.loci)


@dataclass
class SampleResult:
    sample: str
    nfo_lines: List[str] = field(default_factory=list)   # one per organism that passed every gate, in score-table order
    out_log: Optional[str] = None                        # text of the .out file (when log=True)
    stdout: str = ""                                     # what metamlst.py would have printed (quiet=False)
    cel: Optional[dict] = None
    total_reads: int = 0
    ignored_reads: int = 0
    broken_db: bool = False                              # the reference's sys.exit(0) at metamlst.py:190
    calls: List[SpeciesCall] = field(default_factory=list)
    seconds: Dict[str, float] = field(default_factory=dict)
    records: int = 0


# ----------------------------------------------------------------------------------------------------------------
# renderers (pure functions of the typed sample)
# ----------------------------------------------------------------------------------------------------------------
def _status_line(mesg: str, label: str, colour: str) -> str:
    """metamlst_print(mesg, label, type) for messages under 65 characters (metaMLST_functions.py:122-128)."""
    assert len(mesg) < 65
    return mesg.ljust(66) + (colour + "[ - " + label.center(5) + " - ]" + ENDC).ljust(14) + "\r\n"


def render_nfo(call: SpeciesCall, sample: str, write_known: bool) -> str:
    return call.species + "\t" + sample + "\t" + "\t".join(l.nfo_field(write_known) for l in call.loci) + "\r\n"


def render_out_log(bam_path: str, penalty: int, minscore: int, total: int, ignored: int, cel) -> str:
    head = [("SAMPLE:\t\t\t\t\t", bam_path), ("VERSION:\t\t\t\t\t", "1.1"), ("PENALTY:\t\t\t\t", repr(penalty)), ("MIN-THRESHOLD SCORE:\t\t\t\t", repr(minscore)),
            ("TOTAL ALIGNED READS:\t\t\t\t", repr(total)), (" - OF WHICH IGNORED:\t\t\t\t", repr(ignored) + " BAM READS\r\n")]
    text = "".join(k + v + "\r\n" for k, v in head) + "------------------------------  RESULTS ------------------------------\r\n"
    for species, genes in cel.items():
        for gene, alleles in genes.items():
            for allele, triple in sorted(alleles.items(), key=lambda kv: kv[1]):
                text += "\t".join(map(str, (species, gene, allele) + tuple(triple))) + "\r\n"
    return text


def _screen_species_header(call: SpeciesCall) -> str:
    found = set(call.detected)
    names = sorted(set(call.db_genes) | found)
    text = (OKGREEN if call.passed_gate else FAIL) + " " + call.species.ljust(18, " ") + ENDC + " Detected Loci: " + \
        ", ".join(OKGREEN + g + ENDC for g in names if g in found) + "\n"
    if any(g not in found for g in names):
        text += (" " * 20) + "Missing Loci : " + ", ".join(FAIL + g + ENDC for g in names if g not in found) + "\n"
    return text + "\n"


def _screen_allele_table(call: SpeciesCall, genes: Dict[str, dict], coverage: Dict[str, int], longest) -> str:
    text = _status_line("Closest allele identification", "...", HEADER)
    text += "\r\n  " + "Locus".ljust(7) + "Avg. Coverage".rjust(15) + "Score".rjust(7) + "Hits".rjust(6) + " Reference Allele(s)".ljust(36) + "\n"
    for gene in sorted(genes):
        info = genes[gene]
        top = max(t[2] for t in info.values())
        tied = [a for a, t in info.items() if t[2] == top]
        shown = ",".join(sorted(tied, key=int)[:5]) + ("... (" + str(len(tied)) + " more)" if len(tied) > 5 else "")
        cov = round(float(coverage[call.species + "_" + gene]) / float(longest(call.species, gene)), 2)
        text += "  " + WARNING + gene.ljust(7) + ENDC + str(cov).rjust(15) + ENDC + HEADER + str(top).rjust(7) + str(info[tied[0]][1]).rjust(6) + \
            ENDC + OKBLUE + " " + shown.ljust(36) + ENDC + "\n"
    return text + "\n" + _status_line("Building Consensus Sequences", "...", HEADER)


def _screen_consensus_table(call: SpeciesCall, min_accuracy: float) -> str:
    text = "\r"  # buildConsensus ends with print('\r', end='') (metaMLST_functions.py:278)
    text += "\r\n  " + "Locus".ljust(7) + "Ref.".ljust(7) + "Length".rjust(7) + "Ns".rjust(7) + "SNPs".rjust(7) + "Confidence".rjust(15) + "Notes".rjust(10) + "\n"
    for l in sorted(call.loci, key=lambda x: x.contig):
        note = "--" if l.snps == 0 else (l.known_as or "NEW")
        text += "  " + WARNING + l.gene.ljust(7) + ENDC + l.allele.ljust(7) + str(l.length).rjust(7) + str(l.holes).rjust(7) + str(l.snps).rjust(7) + \
            (l.confidence_text() + " %").rjust(15) + note.rjust(10) + "\n"
    text += "\n"
    if call.accepted(min_accuracy):
        return text + _status_line("Reconstruction Successful", "WRITE", OKGREEN)
    return text + _status_line("Accuracy lower than " + str(round(min_accuracy * 100, 2)) + "%", "SKIP", FAIL)


# ----------------------------------------------------------------------------------------------------------------
class SampleTyper:
    """One SQLite connection + one GPU, reused for every sample typed through it."""

    def __init__(self, db_path: str, device: int = 0, minscore: int = 80, max_xM: int = 5, min_read_len: int = 50,
                 min_accuracy: float = 0.90, penalty: int = 100, nloci: int = 100, species_filter: Optional[str] = None,
                 write_known: bool = False, log: bool = False, presorted: bool = False, debug: bool = False,
                 unpack_threads: int = 0, ctx: Optional[native.Context] = None, engine: str = "device", group=None,
                 ingest: str = "host", check_crc: bool = False):
        """check_crc: with ingest="device", also check every BGZF block's CRC32 on the GPU (bam.ingest_bam); the host unpacker
        (ingest="host") always checks it."""
        if not os.path.isfile(db_path):
            raise IOError("Failed to connect to the database: please check your database file!")  # metamlst.py:72-73
        if engine not in ("device", "host", "onecall"):
            raise ValueError("engine must be 'device', 'host' or 'onecall'")
        if ingest not in ("device", "host"):
            raise ValueError("ingest must be 'device' (BGZF inflate + record parse on the GPU) or 'host' (C++ threads)")
        self.db_path = db_path
        self.conn = sqlite3.connect(db_path, check_same_thread=False)
        self.conn.row_factory = sqlite3.Row
        self.device = int(device)
        self._ctx = ctx
        self._own_ctx = ctx is None
        self.engine, self.group, self.ingest, self.check_crc = engine, group, ingest, bool(check_crc)
        self.minscore, self.max_xM, self.min_read_len = int(minscore), int(max_xM), int(min_read_len)
        self.min_accuracy, self.penalty, self.nloci = float(min_accuracy), int(penalty), int(nloci)
        self.species_filter, self.write_known, self.log, self.presorted, self.debug = species_filter, write_known, log, presorted, debug
        self.unpack_threads = int(unpack_threads)
        self._pipe = None          # pipeline.DevicePipeline of the last BAM header seen (a cohort shares one)
        self._pipe_key = None
        self._sidx = None          # api.SampleIndex of the last BAM header seen (engine="onecall")
        self._sidx_key = None
        self._alleles: Optional[Dict[str, str]] = None

    @property
    def ctx(self) -> native.Context:
        if self._ctx is None:
            self._ctx = native.Context(self.device)
        return self._ctx

    def close(self):
        self.conn.close()
        self._pipe = None
        if self._own_ctx and self._ctx is not None:
            self._ctx.close()
            self._ctx = None

    # -- the SQL the reference runs on this path -------------------------------------------------------------------
    def _genes(self, bacterium: str) -> List[str]:  # metamlst.py:184
        return [r["geneName"] for r in self.conn.execute("SELECT geneName FROM genes WHERE bacterium = ?", (bacterium,))]

    def _longest_allele(self, bacterium: str, gene: str) -> int:  # metamlst.py:225-226
        return self.conn.execute("SELECT LENGTH(sequence) as L FROM alleles WHERE bacterium = ? AND gene = ? ORDER BY L DESC LIMIT 1",
                                 (bacterium, gene)).fetchone()["L"]

    def _unal_sequence(self, bacterium: str, gene: str, allele: str):  # metaMLST_functions.py:186-194
        row = self.conn.execute("SELECT sequence FROM alleles WHERE bacterium = ? AND gene = ? AND alleleVariant = ?",
                                (bacterium, gene, allele)).fetchone()
        return row["sequence"] if row is not None else None

    def _sequence_find(self, bacterium: str, sequence: str):  # metaMLST_functions.py:196-203
        row = self.conn.execute("SELECT gene,alleleVariant FROM alleles WHERE sequence = ? AND bacterium = ?", (str(sequence), bacterium)).fetchone()
        return row["gene"] if row else None

    def _allele_table(self) -> Dict[str, str]:
        """{'organism_gene_allele': sequence} of the whole `alleles` table, first row wins (what db_getUnalSequence's fetchone
        returns): read once, it feeds the device copy of the DB sequences."""
        if self._alleles is None:
            t: Dict[str, str] = {}
            for r in self.conn.execute("SELECT bacterium, gene, alleleVariant, sequence FROM alleles ORDER BY recID"):
                t.setdefault("%s_%s_%s" % (r[0], r[1], r[2]), r[3])
            self._alleles = t
        return self._alleles

    # ---------------------------------------------------------------------------------------------------------------
    def unpack(self, bam_path: str):
        """Phase 1: BAM -> packed streams.  Safe to call from another thread than type_unpacked."""
        return bam.unpack_bam(bam_path, presorted=self.presorted, threads=self.unpack_threads)

    def load(self, bam_path: str):
        """Host half of phase 1, safe on a prefetch thread: ingest="host" -> the unpacked streams (C++ threads); ingest="device" -> the
        file's bytes in page-locked memory (the GPU does the rest: `ingest`)."""
        if self.ingest == "device" and self.engine == "device":
            return bam.read_pinned(bam_path, bam.POOL)
        return self.unpack(bam_path)

    def ingest_loaded(self, loaded, want_qhash: bool = False):
        """Device half of phase 1 for ingest="device": compressed bytes cross PCIe; inflate / parse / sort / depth cap / packing happen
        in HBM (csrc/ingest.cu).  A host-unpacked sample passes through."""
        if hasattr(loaded, "c_struct"):
            return loaded
        st = bam.ingest_bam(loaded, self.device, presorted=self.presorted, want_qhash=want_qhash, check_crc=self.check_crc)
        bam.POOL.put(loaded)  # the call is synchronous: the staging buffer has been consumed
        return st

    def type_bam(self, bam_path: str, out_dir: str, want_stdout: bool = False, timestamp: Optional[int] = None) -> SampleResult:
        t0 = time.perf_counter()
        soa = self.ingest_loaded(self.load(bam_path), want_qhash=want_stdout)
        t1 = time.perf_counter()
        res = self.type_unpacked(soa, bam_path, want_stdout=want_stdout)
        res.seconds["unpack"] = t1 - t0
        if self._rank() == 0:
            self.write(res, bam_path, out_dir, timestamp)
        return res

    def _rank(self) -> int:
        if self.engine != "device":
            return 0
        import torch
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            return torch.distributed.get_rank(self.group)
        return 0

    # -- engines: sample -> (calls, cel or None, totals) ------------------------------------------------------------
    def _pipeline(self, soa, want_qhash: bool):
        import numpy as np
        import torch
        from . import pipeline, streams
        dev = torch.device("cuda", self.device)
        dist_on = torch.distributed.is_available() and torch.distributed.is_initialized() and torch.distributed.get_world_size(self.group) > 1
        rank = torch.distributed.get_rank(self.group) if dist_on else 0
        world = torch.distributed.get_world_size(self.group) if dist_on else 1
        if isinstance(soa, streams.DeviceStreams):  # already resident (bam.ingest_bam)
            if world > 1:
                raise ValueError("a device-ingested sample is typed by one GPU; shard a host-unpacked sample (ingest='host') over several")
            st = soa
        else:
            st = streams.DeviceStreams.from_soa(soa, dev, rank=rank, world=world, mode="ranges", want_qhash=want_qhash)
        key = (tuple(soa.ref_names), np.asarray(soa.ref_lens).tobytes())
        if self._pipe is None or self._pipe_key != key:
            index = api.AlleleIndex(soa.ref_names)
            table = self._allele_table()
            genes_in_db = {sp: len(self._genes(sp)) for sp in dict.fromkeys(index.species)}
            self._pipe = pipeline.DevicePipeline(st, index, lambda t: table.get(index.ref_names[t]) or "", minscore=self.minscore, max_xM=self.max_xM,
                                                 min_read_len=self.min_read_len, penalty=self.penalty, species_filter=self.species_filter,
                                                 nloci=self.nloci, genes_in_db=genes_in_db, exchange="allreduce", group=self.group)
            self._pipe_key = key
        else:
            self._pipe.rebind(st)
        return self._pipe

    def _calls_device(self, soa, want_tables: bool, want_cov: bool):
        import torch
        with torch.cuda.device(self.device):
            pipe = self._pipeline(soa, want_cov)
            pipe.want_tables = want_tables
            try:
                per_species = pipe.step()
            except RuntimeError as e:
                if "Database is broken" not in str(e):
                    raise
                # the reference stops at the organism that shows it, earlier organisms are complete (metamlst.py:188-190): rare enough
                # to replay on the host-driven seams from the score tables of a score-only pass
                pipe.want_tables = True
                pipe.run_score()
                pipe._enqueue_tables()
                torch.cuda.current_stream(pipe.dev).synchronize()
                cel = api.finish_scores(pipe.index, *pipe.tables(), self.penalty)
                c = pipe.counters.cpu().numpy().view("uint64")
                pipe.reset_tables()
                if not hasattr(soa, "c_struct"):  # device-resident sample: the host-driven seams want it in host memory
                    qh = soa.qhash
                    soa = soa.to_host(pinned=False)
                    soa.qhash = None if qh is None else qh.cpu().numpy().view("uint64")
                cov = api.coverage_sums(self.ctx, soa, pipe.index, self.minscore, self.max_xM, self.min_read_len, self.species_filter) if want_cov else None
                return self._calls_host_from_cel(soa, cel), cel, int(c[0]), int(c[1]), cov
            cel = api.finish_scores(pipe.index, *pipe.tables(), self.penalty) if want_tables else None
            coverage = pipe.run_coverage() if (want_cov and per_species) else None
        calls = []
        for sp in (cel.keys() if cel is not None else per_species.keys()):  # the log / screen text walk the organisms the gate drops too
            detected = list(cel[sp].keys()) if cel is not None else [c.split("_")[1] for (c, _s, _h, _n) in per_species[sp]]
            call = SpeciesCall(sp, self._genes(sp), detected, passed_gate=sp in per_species)
            call.loci = [LocusCall(c, s, int(h), int(n)) for (c, s, h, n) in per_species.get(sp, [])]
            calls.append(call)
        return calls, cel, pipe.total_reads, pipe.ignored_reads, coverage

    def _calls_onecall(self, soa, want_tables: bool, want_cov: bool):
        """engine="onecall": the sample stays in host memory and goes through ONE library call (api.type_soa -> mmlst_sample): score stream up, score,
        selection on the device, only the chosen contigs' pileup records up, pileup, consensus, results down."""
        import numpy as np
        key = (tuple(soa.ref_names), np.asarray(soa.ref_lens).tobytes())
        if self._sidx is None or self._sidx_key != key:
            index = api.AlleleIndex(soa.ref_names)
            table = self._allele_table()
            genes_in_db = {sp: len(self._genes(sp)) for sp in dict.fromkeys(index.species)}
            self._sidx = api.SampleIndex(self.ctx, index, soa.ref_lens, lambda t: table.get(index.ref_names[t]) or "", genes_in_db)
            self._sidx_key = key
        sidx = self._sidx
        try:
            r = api.type_soa(sidx, soa, self.minscore, self.max_xM, self.min_read_len, self.penalty, self.nloci, self.species_filter, want_tables=want_tables)
        except RuntimeError as e:
            if "Database is broken" not in str(e):
                raise
            return self._calls_host(soa, want_cov)   # rare: replayed seam by seam, the reference stops at the organism that shows it
        per_species = dict(r["species"])
        cel = api.finish_scores(sidx.index, *r["tables"], self.penalty) if want_tables else None
        coverage = None
        if want_cov and per_species:
            coverage = api.coverage_sums(self.ctx, soa, sidx.index, self.minscore, self.max_xM, self.min_read_len, self.species_filter)
        calls = []
        for sp in (cel.keys() if cel is not None else per_species.keys()):
            detected = list(cel[sp].keys()) if cel is not None else [c.split("_")[1] for (c, _s, _h, _n) in per_species[sp]]
            call = SpeciesCall(sp, self._genes(sp), detected, passed_gate=sp in per_species)
            call.loci = [LocusCall(c, s, int(h), int(n)) for (c, s, h, n) in per_species.get(sp, [])]
            calls.append(call)
        return calls, cel, r["totalReads"], r["ignoredReads"], coverage

    def _calls_host_from_cel(self, soa, cel) -> List[SpeciesCall]:
        """Gate, selection (metamlst.py:244) and seam S2 per organism from a finished score table."""
        calls = []
        for sp, genes in cel.items():
            db_genes = self._genes(sp)
            call = SpeciesCall(sp, db_genes, list(genes.keys()))
            calls.append(call)
            if len(db_genes) < len(genes):  # metamlst.py:188-190: message, then sys.exit(0) -- the sample ends here
                call.passed_gate = None  # type: ignore[assignment]
                break
            listed = len(set(db_genes) | set(genes))  # tVar: the DB's genes plus every detected one (metamlst.py:186,192-194)
            call.passed_gate = int((float(len(genes)) / float(listed)) * 100) >= self.nloci
            if not call.passed_gate:
                continue
            chromosomeList = {sp + "_" + g + "_" + a: self._unal_sequence(sp, g, a) for g, a in api.select_alleles(genes)}
            recs = api.build_consensus(self.ctx, soa, chromosomeList, self.minscore, self.max_xM, self.debug)
            for r in recs:
                holes, snps = (int(x.split("::")[1]) for x in r.description.split("_"))
                call.loci.append(LocusCall(r.id, str(r.seq), holes, snps))
        return calls

    def _calls_host(self, soa, want_cov: bool):
        index = api.AlleleIndex(soa.ref_names)
        cel, total, ignored, _raw = api.score_soa(self.ctx, soa, index, self.minscore, self.max_xM, self.min_read_len, self.species_filter, self.penalty)
        calls = self._calls_host_from_cel(soa, cel)
        coverage = None
        if want_cov and any(c.passed_gate for c in calls):
            coverage = api.coverage_sums(self.ctx, soa, index, self.minscore, self.max_xM, self.min_read_len, self.species_filter)
        return calls, cel, total, ignored, coverage

    # ---------------------------------------------------------------------------------------------------------------
    def type_unpacked(self, soa, bam_path: str, want_stdout: bool = False) -> SampleResult:
        """Phase 2 (GPU + per-locus host formatting): metamlst.py:101-296 on an unpacked sample."""
        t_start = time.perf_counter()
        sample = bam_path.split("/")[-1].split(".")[0]  # metamlst.py:89
        res = SampleResult(sample=sample)
        want_tables = bool(self.log or want_stdout)
        if self.engine == "device":
            calls, cel, res.total_reads, res.ignored_reads, coverage = self._calls_device(soa, want_tables, want_stdout)
        elif self.engine == "onecall":
            calls, cel, res.total_reads, res.ignored_reads, coverage = self._calls_onecall(soa, want_tables, want_stdout)
        else:
            calls, cel, res.total_reads, res.ignored_reads, coverage = self._calls_host(soa, want_stdout)
        t_gpu = time.perf_counter()
        res.cel, res.calls = cel, calls
        if self.log:
            res.out_log = render_out_log(bam_path, self.penalty, self.minscore, res.total_reads, res.ignored_reads, cel)
        screen: List[str] = []
        if want_stdout:
            screen.append(OKBLUE + "Sample file: " + ENDC + os.path.realpath(sample) + "\n")
            screen.append(OKBLUE + "MetaMLST Database file: " + ENDC + os.path.basename(self.db_path) + "\n\n")
        for call in calls:
            if call.passed_gate is None:  # "Database is broken": the reference prints and exits (metamlst.py:189-190)
                screen.append("Database is broken for" + call.species + FAIL + "[ - EXITING - ]".rjust(75, " ") + ENDC + "\n")
                res.broken_db = True
                break
            if want_stdout:
                screen.append(_screen_species_header(call))
            if not call.passed_gate:
                continue
            if want_stdout:
                for l in call.loci:
                    if l.snps > 0:
                        l.known_as = self._sequence_find(call.species, l.sequence)
                screen.append(_screen_allele_table(call, cel[call.species], coverage, self._longest_allele))
                screen.append(_screen_consensus_table(call, self.min_accuracy))
            if call.accepted(self.min_accuracy):
                res.nfo_lines.append(render_nfo(call, sample, self.write_known))
        if want_stdout:
            if calls and not res.broken_db:
                screen.append("\033[92m" + "[ - Completed - ]".rjust(80, " ") + "\033[0m" + "\n")
            res.stdout = "".join(screen)
        res.seconds.update({"gpu": t_gpu - t_start, "format": time.perf_counter() - t_gpu})
        return res

    def write(self, res: SampleResult, bam_path: str, out_dir: str, timestamp: Optional[int] = None) -> None:
        """Phase 3: the files metamlst.py leaves in its -o folder."""
        if not os.path.isdir(out_dir):
            os.mkdir(out_dir)  # metamlst.py:91
        if res.out_log is not None:
            ts = int(time.time()) if timestamp is None else int(timestamp)
            with open(out_dir + "/" + res.sample + "_" + str(ts) + ".out", "w", newline="") as f:
                f.write(res.out_log)
        for line in res.nfo_lines:
            with open(out_dir + "/" + res.sample + ".nfo", "a", newline="") as f:  # append mode, one line per organism
                f.write(line)


def type_cohort(bam_paths: Sequence[str], db_path: str, out_dir: str, devices: Sequence[int] = (0,), prefetch: int = 2,
                typers: Optional[Dict[int, "SampleTyper"]] = None, loaders: int = 2, **params) -> List[SampleResult]:
    """Type a cohort back to back (BASELINE.json configs[3]): per device one worker thread owning a SampleTyper (one DB
    connection, one set of device tables for the whole cohort); a loader thread per device runs `prefetch` samples ahead (host
    unpack, or with ingest="device" just the file read into page-locked memory).  Samples are dealt round-robin to the devices;
    results come back in input order.  `typers` ({device: SampleTyper}): reuse warm typers (they stay open) instead of making new ones."""
    results: List[Optional[SampleResult]] = [None] * len(bam_paths)
    errors: List[BaseException] = []

    def worker(slot: int, device: int):
        mine = [i for i in range(len(bam_paths)) if i % len(devices) == slot]
        if not mine:
            return
        typer = typers[device] if typers is not None else SampleTyper(db_path, device=device, **params)
        q: "queue.Queue" = queue.Queue(maxsize=max(1, prefetch))
        stop = threading.Event()

        def put(item) -> bool:
            while not stop.is_set():
                try:
                    q.put(item, timeout=0.1)
                    return True
                except queue.Full:
                    pass
            return False

        todo: "queue.Queue" = queue.Queue()
        for i in mine:
            todo.put(i)
        n_load = max(1, min(int(loaders), len(mine)))

        def unpacker():
            # `loaders` threads per device pull the next sample of this device: reading a file into page-locked memory (or unpacking it
            # on the host) takes longer than typing it on the GPU, one thread would be the bottleneck
            while not stop.is_set():
                try:
                    i = todo.get_nowait()
                except queue.Empty:
                    break
                try:
                    t0 = time.perf_counter()
                    soa = typer.load(bam_paths[i])
                    if not put((i, soa, time.perf_counter() - t0, None)):
                        return
                except BaseException as e:  # noqa: BLE001
                    put((i, None, 0.0, e))
                    return
            put(None)

        ths = [threading.Thread(target=unpacker, daemon=True) for _ in range(n_load)]
        for th in ths:
            th.start()
        finished = 0
        try:
            while True:
                item = q.get()
                if item is None:
                    finished += 1
                    if finished == n_load:
                        break
                    continue
                i, soa, t_unpack, err = item
                if err is not None:
                    raise err
                t0 = time.perf_counter()
                soa = typer.ingest_loaded(soa)
                t_ing = time.perf_counter() - t0
                res = typer.type_unpacked(soa, bam_paths[i])
                res.seconds["load"] = t_unpack
                res.seconds["device_ingest"] = t_ing
                res.records = int(soa.tid.shape[0]) if hasattr(soa, "tid") else 0
                del soa
                typer.write(res, bam_paths[i], out_dir)
                res.seconds["typed_and_written"] = time.perf_counter() - t0
                results[i] = res
        except BaseException as e:  # noqa: BLE001
            errors.append(e)
        finally:
            stop.set()  # a failing worker releases its unpacker (and the page-locked sample it may be holding)
            while True:
                try:
                    q.get_nowait()
                except queue.Empty:
                    break
            for th in ths:
                th.join(timeout=5)
            if typers is None:
                typer.close()

    threads = [threading.Thread(target=worker, args=(s, d)) for s, d in enumerate(devices)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        raise errors[0]
    return [r for r in results if r is not None]


# ----------------------------------------------------------------------------------------------------------------
# one PROCESS per GPU (the B200 way to run a box: no interpreter lock and no driver lock shared between the devices)
# ----------------------------------------------------------------------------------------------------------------
def _pool_worker(slot: int, device: int, db_path: str, params: dict, tasks, results):
    try:
        import torch
        torch.cuda.set_device(device)
        typer = SampleTyper(db_path, device=device, **params)
    except BaseException as e:  # noqa: BLE001
        results.put(("error", slot, repr(e)))
        return
    results.put(("ready", slot, None))
    while True:
        task = tasks.get()
        if task is None:
            break
        ids, paths, out_dir = task
        try:
            res = type_cohort(paths, db_path, out_dir, devices=(device,), typers={device: typer})
            for r in res:
                r.cel = None  # large and rebuilt on demand; keep the reply small
            results.put(("done", slot, list(zip(ids, res))))
        except BaseException as e:  # noqa: BLE001
            results.put(("error", slot, repr(e)))
    typer.close()


class CohortPool:
    """Persistent workers, one PROCESS per entry of `devices` (a device may be listed twice: two processes then share the GPU and the
    host-side part of one sample -- file read, block table, launches -- runs under the kernels of the other), each owning a warm
    SampleTyper (DB connection, device tables, ingest workspace).  `type(bam_paths, out_dir)` deals the samples round-robin and returns
    the SampleResults in input order -- what a shell loop of `metamlst.py` runs over a cohort (BASELINE.json configs[3]) becomes one
    call per cohort."""

    def __init__(self, db_path: str, devices: Sequence[int], **params):
        import multiprocessing as mp
        ctx = mp.get_context("spawn")
        self.devices = list(devices)
        self.db_path = db_path
        self._results = ctx.Queue()
        self._tasks = [ctx.Queue() for _ in self.devices]
        self._procs = [ctx.Process(target=_pool_worker, args=(i, d, db_path, dict(params), self._tasks[i], self._results), daemon=True)
                       for i, d in enumerate(self.devices)]
        for p in self._procs:
            p.start()
        for _ in self.devices:
            kind, slot, info = self._results.get()
            if kind != "ready":
                self.close()
                raise RuntimeError("cohort worker %s (device %s) failed to start: %s" % (slot, self.devices[slot], info))

    def type(self, bam_paths: Sequence[str], out_dir: str) -> List[SampleResult]:
        if not os.path.isdir(out_dir):
            os.mkdir(out_dir)
        share: List[list] = [[] for _ in self.devices]
        for i, p in enumerate(bam_paths):
            share[i % len(self.devices)].append((i, p))
        busy = 0
        for slot, items in enumerate(share):
            if items:
                self._tasks[slot].put(([i for i, _p in items], [p for _i, p in items], out_dir))
                busy += 1
        out: List[Optional[SampleResult]] = [None] * len(bam_paths)
        for _ in range(busy):
            kind, slot, info = self._results.get()
            if kind == "error":
                raise RuntimeError("cohort worker %s (device %s): %s" % (slot, self.devices[slot], info))
            for i, r in info:
                out[i] = r
        return [r for r in out if r is not None]

    def close(self):
        for q in self._tasks:
            try:
                q.put(None)
            except Exception:  # noqa: BLE001
                pass
        for p in self._procs:
            p.join(timeout=10)
            if p.is_alive():
                p.terminate()
