"""Device-resident driver of the hot path: score -> best-allele selection -> pileup -> consensus.

One instance per GPU / process.  Inputs are the packed streams already in HBM (torch tensors); the kernels are
launched through the `*_dev` C-ABI on torch's current stream.  With torch.distributed initialised (NCCL, one process
per GPU) the partial integer tables are combined with all-reduce (SUM for scores/hits/counts, MIN for first indices),
exactly the exchange SURVEY.md 8e names; shards must be contig-aligned so that the htslib depth cap stays local.
"""
from __future__ import annotations

import os
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import api, dist, native

def build_chunks(contig_start: np.ndarray, chosen_tid: Sequence[int], col_off: np.ndarray) -> np.ndarray:
    """mmlst_chunk descriptors (8 x u32 each) for the chosen contigs of a device-resident pileup stream."""
    out = []
    total = sum(int(contig_start[t + 1]) - int(contig_start[t]) for t in chosen_tid)
    CHUNK_RECORDS = int(native.lib().mmlst_chunk_records(total))  # whole tiles, <= 63 tiles, >= 4 chunks per SM
    for l, t in enumerate(chosen_tid):
        r0, r1 = int(contig_start[t]), int(contig_start[t + 1])
        for b in range(r0, r1, CHUNK_RECORDS):
            out.append((b, min(r1, b + CHUNK_RECORDS), int(col_off[l]), int(col_off[l + 1] - col_off[l]), 0, 0, 0, 0))
    return np.asarray(out, dtype=np.uint32).reshape(-1, 8)


class DevicePipeline:
    def __init__(self, streams, index: api.AlleleIndex, dbseq_of: Callable[[int], str], minscore: int = 80, max_xM: int = 5,
                 min_read_len: int = 50, penalty: int = 100, species_filter: Optional[str] = None, mincov: int = 1,
                 impl: int = 0, idx_base: int = 0, group=None, nloci: int = 100, genes_in_db: Optional[Dict[str, int]] = None,
                 db_ascii: Optional[np.ndarray] = None, db_off: Optional[np.ndarray] = None, exchange: str = "allreduce",
                 use_runs: Optional[bool] = None):
        """exchange (only with torch.distributed, world > 1): "allreduce" = partial score / count tensors are all-reduced
        (any record sharding whose depth cap was resolved beforehand); "gather" = owner mode for contig-aligned shards:
        each rank finishes its own loci and ONE all-gather of the result blocks ends the pass (dist.merge_owner_blocks);
        "p2p" = owner mode with the all-gather done by our own kernels over NVLink peer memory (csrc/exchange.cu): the
        block is stored straight into every peer's symmetric buffer, no NCCL call inside the pass."""
        api.refuse_lenient(streams)
        self.s = streams
        self._use_runs_arg, self._idx_base_arg = use_runs, idx_base
        self.index = index
        self.dbseq_of = dbseq_of
        self.minscore, self.max_xM, self.min_read_len, self.penalty = int(minscore), api.check_max_xm(max_xM), int(min_read_len), int(penalty)
        self.mincov, self.impl = int(mincov), int(impl)
        self.idx_base = int(idx_base) if idx_base else int(getattr(streams, "idx_base", 0) or 0)
        self.group = group
        self.dist = torch.distributed.is_available() and torch.distributed.is_initialized() and torch.distributed.get_world_size() > 1
        if exchange not in ("allreduce", "gather", "p2p"):
            raise ValueError("exchange must be 'allreduce', 'gather' or 'p2p'")
        self.owner = self.dist and exchange in ("gather", "p2p")
        self.p2p = self.dist and exchange == "p2p"
        self.world = torch.distributed.get_world_size() if self.dist else 1
        dev = streams.as0.device
        self.dev = dev
        self.use_runs = bool(use_runs) if use_runs is not None else getattr(streams, "run_tid", None) is not None
        self.use_qc = self.use_runs and getattr(streams, "chunk_qlen", None) is not None  # len(SEQ) per chunk: 3 B / record
        n_ref = len(index.ref_names)
        self.n_ref = n_ref
        self.allow = torch.from_numpy(index.allow_mask(species_filter)).to(dev)
        self.locus_of = torch.from_numpy(index.locus_of.astype(np.int32)).to(dev)
        # every accumulator that must start at zero lives in ONE int64 block => one memset node per pass
        self.max_cols = int(np.sort(np.asarray(streams.ref_lens))[::-1][: index.n_loci].sum())
        w_hit, w_cnt = (n_ref + 1) // 2, (self.max_cols * 5 + 8 + 1) // 2
        self.zblock = torch.zeros(n_ref + 2 + w_hit + w_cnt, dtype=torch.int64, device=dev)
        self.zscore = self.zblock[: n_ref + 2 + w_hit]  # [sum_as | counters | n_hit]: one SUM all-reduce
        self.sum_as = self.zblock[:n_ref]
        self.counters = self.zblock[n_ref:n_ref + 2]
        self.n_hit = self.zblock[n_ref + 2:n_ref + 2 + w_hit].view(torch.int32)[:n_ref]
        self.counts = self.zblock[n_ref + 2 + w_hit:].view(torch.int32)[: self.max_cols * 5 + 8]
        self.first_idx = torch.zeros(n_ref, dtype=torch.int32, device=dev)
        self._db_cache: Dict[Tuple[int, ...], tuple] = {}
        self.lib = native.lib()
        # ---- device-side selection (mmlst_select_dev): look-up tables + output block
        self.nloci = int(nloci)
        species_names: List[str] = []
        sp_id: Dict[str, int] = {}
        sol = np.zeros(index.n_loci, dtype=np.int32)
        for l, (sp, _g) in enumerate(index.locus_names):
            if sp not in sp_id:
                sp_id[sp] = len(species_names)
                species_names.append(sp)
            sol[l] = sp_id[sp]
        self.species_names = species_names
        gdb = np.zeros(len(species_names), dtype=np.int32)
        for sp, i in sp_id.items():
            gdb[i] = (genes_in_db or {}).get(sp, int((sol == i).sum()))  # rows of `genes` for the organism (metamlst.py:184)
        if db_ascii is None:
            seqs = [dbseq_of(t).encode("latin-1") for t in range(n_ref)]
            db_off = np.zeros(n_ref + 1, dtype=np.int64)
            db_off[1:] = np.cumsum([len(x) for x in seqs])
            db_ascii = np.frombuffer(b"".join(seqs), dtype=np.uint8)
        self.bad_len = np.asarray(streams.ref_lens, dtype=np.int64) > (db_off[1:] - db_off[:-1])  # H10
        t32 = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        self.allele_num = t32(np.asarray([int(a) for a in index.allele], dtype=np.int64).astype(np.uint32).view(np.int32))
        self.species_of_locus = t32(sol)
        self.genes_in_db = t32(gdb)
        self.ref_len_d = t32(np.asarray(streams.ref_lens, dtype=np.int32))
        self.contig_start_d = torch.zeros(n_ref + 1, dtype=torch.int64, device=dev)
        self.max_chunks = 0
        self.rebind(streams)
        self.db_ascii_d = t32(np.concatenate([db_ascii, np.zeros(8, np.uint8)]))
        self.db_off_d = t32(np.asarray(db_off, dtype=np.int64))
        nl = index.n_loci
        self.scratch = torch.zeros(nl * 12 + 64, dtype=torch.uint8, device=dev)
        order = np.argsort(index.locus_of, kind="stable").astype(np.uint32)  # allele rows grouped by locus
        # rows already grouped by locus (a DB dumped gene by gene): no row list, the selection kernel saves a dependent trip to memory
        self.locus_rows = None if np.array_equal(order, np.arange(order.shape[0], dtype=order.dtype)) else t32(order.view(np.int32))
        self.locus_start = t32(np.searchsorted(index.locus_of[order], np.arange(nl + 1)).astype(np.int32))
        # ONE output block => one D2H node per pass: int32 header[16] | chosen_tid[nl] | chosen_species[nl] | col_off[nl+1] |
        # holes[nl] | snps[nl] | pad, then the consensus bytes
        self.o_hdr, self.o_tid, self.o_sp, self.o_col, self.o_holes, self.o_snps = 0, 16, 16 + nl, 16 + 2 * nl, 17 + 3 * nl, 17 + 4 * nl
        self.o_first = 17 + 5 * nl
        self.n_small = (17 + 6 * nl + 7) // 4 * 4
        self.out = torch.zeros((self.n_small * 4 + self.max_cols + 16 + 15) // 16 * 16, dtype=torch.uint8, device=dev)
        self.small = self.out[: self.n_small * 4].view(torch.int32)
        self.cons = self.out[self.n_small * 4:]
        self.holes = self.small[self.o_holes:self.o_holes + nl]
        self.snps = self.small[self.o_snps:self.o_snps + nl]
        self.db_start_d = torch.zeros(nl + 1, dtype=torch.int64, device=dev)
        self.out_bytes = int(self.out.shape[0])
        if self.owner:  # every rank's block, gathered (+ 16 B: status word of the peer-memory exchange)
            self.out_all = torch.zeros(self.world * self.out_bytes + 16, dtype=torch.uint8, device=dev)
            self.out_h = torch.zeros(self.world * self.out_bytes + 16, dtype=torch.uint8).pin_memory()
            if self.p2p:
                self._init_p2p()
        else:
            self.out_h = torch.zeros(self.out_bytes, dtype=torch.uint8).pin_memory()
        self.small_h = self.out_h[: self.n_small * 4].view(torch.int32)
        self.cons_h = self.out_h[self.n_small * 4: self.out_bytes]
        self.genes_in_db_h = gdb
        self.ticket = torch.zeros(nl + 8, dtype=torch.int32, device=dev)   # fused consensus: chunks finished per chosen locus (self-resetting)
        # pileup + consensus as ONE launch: built, parity-tested, measured on B200 (profiles/r2y_bench_fused{0,1}.json): serial pass 76.9 us fused against
        # 74.3 us as two launches (the last chunk of every locus finishes at the end of the grid, so the fused consensus is a serial tail of one CTA per
        # locus, and every chunk pays two CTA barriers and a ticket) -- off unless MMLST_FUSED_TAIL=1
        self.fused_tail = os.environ.get("MMLST_FUSED_TAIL", "0") == "1"
        self.want_tables = False  # step() also brings (sum_as, n_hit, first_idx) to the host: tables()
        self._tables_h = None
        self._clean = False  # score tables / counts / scratch hold the "nothing accumulated" state
        self.timers: Optional[Dict[str, list]] = None  # name -> [(start_event, end_event)]
        self.launches = 0

    # ------------------------------------------------------------------------------------------------------------
    def rebind(self, streams):
        """Point the pipeline at ANOTHER sample unpacked against the same BAM header (a cohort typed against one index: every
        look-up table, accumulator and the output block are reused; only the record streams and their contig ranges change).
        A captured CUDA graph is dropped (it holds the old streams' addresses)."""
        if list(streams.ref_names) != self.index.ref_names or not np.array_equal(np.asarray(streams.ref_lens), np.asarray(self.s.ref_lens)):
            raise ValueError("rebind: the sample was aligned against a different reference set")
        api.refuse_lenient(streams)
        self.s = streams
        self.use_runs = getattr(streams, "run_tid", None) is not None if self._use_runs_arg is None else bool(self._use_runs_arg)
        self.use_qc = self.use_runs and getattr(streams, "chunk_qlen", None) is not None
        self.idx_base = int(self._idx_base_arg) if self._idx_base_arg else int(getattr(streams, "idx_base", 0) or 0)
        self.contig_start_d.copy_(torch.from_numpy(np.asarray(streams.contig_start, dtype=np.uint64).view(np.int64)), non_blocking=False)
        self._pack16()
        need = int(streams.n_prec) // 512 + self.index.n_loci + 8
        if need > self.max_chunks:
            self.max_chunks = need
            self.chunks_d = torch.zeros(self.max_chunks * 8, dtype=torch.int32, device=self.dev)
        self.graph = None

    def _pack16(self):
        """The compact score stream (2 B / record, mmlst_score_pack16_dev) of a run-length sample with len(SEQ) per chunk and no
        file-order index: code[] / head[] derived from the resident as0 / xm3 / chunk_qlen, which stay resident (the chunks the compact
        code cannot decide, the partial last chunk, the coverage column and to_host() read them).  Derived again for every sample bound."""
        s = self.s
        self.code16 = self.head16 = None
        n = int(s.as0.shape[0])
        if not self.use_qc or getattr(s, "orig_idx", None) is not None or n == 0:
            return
        nch = (n + 255) // 256
        self.code16 = torch.empty(nch * 256, dtype=torch.int16, device=self.dev)  # whole chunks: the kernel's bulk copies read 512 B per chunk
        self.head16 = torch.empty(nch, dtype=torch.int32, device=self.dev)
        native.check(self.lib.mmlst_score_pack16_dev(native.ptr(s.as0), native.ptr(s.xm3), native.ptr(s.chunk_qlen), n, native.ptr(self.code16),
                                                     native.ptr(self.head16), self._stream()))

    def compact_fallback_chunks(self) -> int:
        """Full chunks of the bound sample that form 7 reduces from the 3-byte arrays at this pipeline's minscore (code 0, "as0 <= top - 1023",
        could pass there); -1 without a compact stream."""
        if self.code16 is None:
            return -1
        n = int(self.s.as0.shape[0])
        top = (self.head16[: n // 256] & 0xFFFF).to(torch.int32)
        top = top - ((top & 0x8000) << 1)  # u16 -> int16
        return int((top - 1023 >= self.minscore).sum().item())

    def _timed(self, name: str, fn):
        if self.timers is None:
            fn()
            return
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        self.timers.setdefault(name, []).append((a, b))

    def _stream(self):
        return torch.cuda.current_stream(self.dev).cuda_stream

    def reset_tables(self):
        """Score tables, counters, count tensor and the selection ticket back to the empty state.  The device-driven
        pass (`_enqueue`) leaves them that way itself (MMLST_SELECT_CONSUME / MMLST_CONSENSUS_CONSUME)."""
        self.zblock.zero_(); self.first_idx.fill_(-1); self.scratch.zero_(); self.ticket.zero_()
        self._clean = True

    def _score_call(self):
        """Stage 1 over the resident score stream: the run-length form when the streams carry it (2 B / record compact or 3 B / record
        with len(SEQ) per chunk, else 5 B / record), else the explicit-tid form (9 B / record)."""
        s = self.s
        n = int(s.as0.shape[0])
        oi = native.ptr(getattr(s, "orig_idx", None))  # file-order index per record (BAM that was not coordinate-sorted, locus shards); NULL = identity + idx_base
        if n == 0:
            return
        if self.use_runs and self.use_qc and self.code16 is not None:  # the library picks form 7 or the 3-byte call (another form, max_xM >= 15)
            native.check(self.lib.mmlst_score_runs16_dev(native.ptr(s.run_tid), native.ptr(s.run_start), int(s.run_tid.shape[0]), native.ptr(s.chunk_run),
                                                         native.ptr(s.chunk_qlen), native.ptr(s.as0), native.ptr(s.xm3), native.ptr(self.code16),
                                                         native.ptr(self.head16), n, self.idx_base, native.ptr(self.allow), self.n_ref, self.minscore,
                                                         self.max_xM, self.min_read_len, native.ptr(self.sum_as), native.ptr(self.n_hit),
                                                         native.ptr(self.first_idx), native.ptr(self.counters), self._stream()))
        elif self.use_runs and self.use_qc:
            native.check(self.lib.mmlst_score_runs_qc_dev(native.ptr(s.run_tid), native.ptr(s.run_start), int(s.run_tid.shape[0]), native.ptr(s.chunk_run),
                                                          native.ptr(s.chunk_qlen), native.ptr(s.as0), native.ptr(s.xm3), oi, n, self.idx_base,
                                                          native.ptr(self.allow), self.n_ref, self.minscore, self.max_xM, self.min_read_len,
                                                          native.ptr(self.sum_as), native.ptr(self.n_hit), native.ptr(self.first_idx),
                                                          native.ptr(self.counters), self._stream()))
        elif self.use_runs:
            native.check(self.lib.mmlst_score_runs_dev(native.ptr(s.run_tid), native.ptr(s.run_start), int(s.run_tid.shape[0]), native.ptr(s.chunk_run),
                                                       native.ptr(s.as0), native.ptr(s.xm3), native.ptr(s.qlen), oi, n, self.idx_base,
                                                       native.ptr(self.allow), self.n_ref, self.minscore, self.max_xM, self.min_read_len,
                                                       native.ptr(self.sum_as), native.ptr(self.n_hit), native.ptr(self.first_idx),
                                                       native.ptr(self.counters), self._stream()))
        else:
            native.check(self.lib.mmlst_score_dev(native.ptr(s.tid), native.ptr(s.as0), native.ptr(s.xm3), native.ptr(s.qlen), oi, n, self.idx_base,
                                                  native.ptr(self.allow), native.ptr(self.locus_of), self.n_ref, self.minscore, self.max_xM,
                                                  self.min_read_len, native.ptr(self.sum_as), native.ptr(self.n_hit), native.ptr(self.first_idx),
                                                  native.ptr(self.counters), self._stream()))

    def run_score(self, reset: bool = True):
        s = self.s
        if reset:
            self.reset_tables()
        self._clean = False
        self._timed("score", self._score_call)
        self.launches += 1
        if self.dist and not self.owner:
            dist.allreduce_score_block(self.zscore, self.first_idx, self.group)

    # -- coverage column (H7, metamlst.py:127,228), csrc/coverage.cu.  run_coverage is the whole of it; the four steps below are
    # what it runs on a record shard that cuts through loci, exposed so that shards can be driven one after another in one process.
    def _cov_call(self, fn):
        s = self.s
        native.check(fn(native.ptr(s.tid), native.ptr(s.as0), native.ptr(s.xm3), native.ptr(s.qlen),
                        native.ptr(getattr(s, "orig_idx", None)),  # file-order index per record, exactly as _score_call passes it
                        native.ptr(s.qhash), int(s.tid.shape[0]), self.idx_base, native.ptr(self.allow), native.ptr(self.locus_of), self.n_ref,
                        self.minscore, self.max_xM, self.min_read_len, native.ptr(self._cov_table), self._cov_slots, native.ptr(self._cov),
                        self._stream()))

    def _coverage_reset(self):
        s = self.s
        if getattr(s, "qhash", None) is None:
            raise ValueError("streams were packed without QNAME keys (want_qhash)")
        self._cov_slots = int(self.lib.mmlst_coverage_table_slots(int(s.tid.shape[0])))
        if getattr(self, "_cov_table", None) is None or self._cov_table.shape[0] < self._cov_slots * 3:
            self._cov_table = torch.empty(self._cov_slots * 3, dtype=torch.int64, device=self.dev)
            self._cov = torch.zeros(self.index.n_loci, dtype=torch.int64, device=self.dev)
        self._cov_table[: self._cov_slots * 3].zero_(); self._cov.zero_()

    def coverage_insert(self, reset: bool = True):
        """Zeroes the (locus, QNAME) table and the per-locus sums (unless `reset` is False), then inserts every passing record
        of this shard: afterwards each slot holds the largest value word, (file index + 1) << 16 | len(SEQ), among this
        shard's records of the name."""
        if reset:
            self._coverage_reset()
        self._cov_call(self.lib.mmlst_coverage_insert_dev)
        self.launches += 1

    def coverage_entries(self) -> torch.Tensor:
        """The occupied slots of the table as one int64 tensor [m][3]: key words (2) and value word."""
        n = self._cov_slots
        keys = self._cov_table[: 2 * n].view(n, 2)
        occ = (keys != 0).any(1)
        return torch.cat([keys[occ], self._cov_table[2 * n: 3 * n][occ].view(-1, 1)], 1)

    def coverage_merge(self, entries: torch.Tensor):
        """Raise this shard's slots to the value words of the same keys in `entries` (another shard's coverage_entries, any
        number of rows; rows of zeros are skipped).  Keys this shard does not hold are ignored."""
        m = int(entries.shape[0])
        if m == 0:
            return
        keys = entries[:, :2].contiguous()
        vals = entries[:, 2].contiguous()
        native.check(self.lib.mmlst_coverage_merge_dev(native.ptr(keys), native.ptr(vals), m, native.ptr(self._cov_table), self._cov_slots,
                                                       self._stream()))
        self.launches += 1

    def coverage_sum(self) -> torch.Tensor:
        """Sum pass: every record that IS the last of its name (value word equal to its slot's) adds len(SEQ) to its locus.
        Returns the per-locus sums of this shard (int64 [n_loci], on the device)."""
        self._cov_call(self.lib.mmlst_coverage_sum_dev)
        self.launches += 1
        return self._cov

    def _exchange_coverage_entries(self):
        """Every rank's occupied slots to every rank (all-gather, padded with zero rows to the largest rank), merged here."""
        mine = self.coverage_entries()
        cnt = torch.tensor([int(mine.shape[0])], dtype=torch.int64, device=self.dev)
        cnts = torch.zeros(self.world, dtype=torch.int64, device=self.dev)
        torch.distributed.all_gather_into_tensor(cnts, cnt, group=self.group)
        m = int(cnts.max().item())
        if m == 0:
            return
        pad = torch.zeros((m, 3), dtype=torch.int64, device=self.dev)
        pad[: mine.shape[0]] = mine
        every = torch.zeros((self.world * m, 3), dtype=torch.int64, device=self.dev)
        torch.distributed.all_gather_into_tensor(every, pad, group=self.group)
        rank = torch.distributed.get_rank(self.group)
        for r in range(self.world):
            if r != rank:
                self.coverage_merge(every[r * m:(r + 1) * m])

    def run_coverage(self, timed: bool = False):
        """Coverage column (H7, metamlst.py:127,228) of the resident score stream: {'species_gene': bases}.  Needs streams
        packed with the 128-bit QNAME keys.  Owner-mode shards ("loci") hold whole loci, so ranks just add their sums.  Record
        shards ("ranges") can split the records of one name over several ranks: between the insert and the sum pass every rank
        merges the others' table entries, so that exactly one rank -- the one holding the name's last record in file order --
        adds it, and the sums add up again."""
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        ev[0].record()
        self._coverage_reset()
        ev[1].record()
        self.coverage_insert(reset=False)
        if self.dist and not self.owner:
            self._exchange_coverage_entries()
        self.coverage_sum()
        ev[2].record()
        if self.dist:
            torch.distributed.all_reduce(self._cov, group=self.group)
        cov = self._cov.cpu().numpy()
        out = {sp + "_" + g: int(cov[l]) for l, (sp, g) in enumerate(self.index.locus_names) if cov[l]}
        if timed:
            return out, {"memset_ms": ev[0].elapsed_time(ev[1]), "kernels_ms": ev[1].elapsed_time(ev[2]), "table_bytes": self._cov_slots * 24}
        return out

    def select(self):
        sum_as = self.sum_as.cpu().numpy()
        n_hit = self.n_hit.cpu().numpy().view(np.uint32)
        first = self.first_idx.cpu().numpy().view(np.uint32)
        return api.fast_select(self.index, sum_as, n_hit, first, self.penalty), (sum_as, n_hit, first)

    def _db_for(self, tids: Tuple[int, ...]):
        hit = self._db_cache.get(tids)
        if hit is None:
            lens = [int(self.s.ref_lens[t]) for t in tids]
            col_off = np.zeros(len(tids) + 1, dtype=np.uint32)
            col_off[1:] = np.cumsum(lens)
            db = np.zeros(int(col_off[-1]) + 8, dtype=np.uint8)
            for i, t in enumerate(tids):
                sq = self.dbseq_of(t)
                if len(sq) < lens[i]:
                    raise IndexError("string index out of range: BAM LN > DB sequence length for %s" % self.index.ref_names[t])
                db[col_off[i]:col_off[i + 1]] = np.frombuffer(sq[:lens[i]].encode("latin-1"), dtype=np.uint8)
            hit = (col_off, torch.from_numpy(db).to(self.dev), torch.from_numpy(col_off.view(np.int32)).to(self.dev))
            if len(self._db_cache) > 64:
                self._db_cache.clear()
            self._db_cache[tids] = hit
        return hit

    def run_pileup_consensus(self, tids: Sequence[int]):
        tids = tuple(int(t) for t in tids)
        s = self.s
        col_off, db_d, col_off_d = self._db_for(tids)
        total = int(col_off[-1])
        chunks = build_chunks(s.contig_start, tids, col_off)
        self.counts[: total * 5].zero_()
        if chunks.shape[0]:
            chunks_d = torch.from_numpy(chunks.view(np.int32)).to(self.dev, non_blocking=True)
            def k():
                native.check(self.lib.mmlst_pileup_dev(native.ptr(s.p_recs), native.ptr(s.planes), native.ptr(chunks_d), int(chunks.shape[0]),
                                                       int(s.max_row_words), self.minscore, self.max_xM, native.ptr(self.counts), total,
                                                       self.impl, self._stream()))
            self._timed("pileup", k)
            self.launches += 1
        if self.dist:
            dist.allreduce_counts(self.counts[: total * 5], self.group)
        def k2():
            native.check(self.lib.mmlst_consensus_dev(native.ptr(self.counts), native.ptr(db_d), native.ptr(col_off_d), len(tids), self.mincov,
                                                      native.ptr(self.cons), native.ptr(self.holes), native.ptr(self.snps), self._stream()))
        self._timed("consensus", k2)
        self.launches += 1
        cons = self.cons[:total].cpu().numpy()
        holes = self.holes[: len(tids)].cpu().numpy()
        snps = self.snps[: len(tids)].cpu().numpy()
        return [cons[col_off[i]:col_off[i + 1]].tobytes().decode("latin-1") for i in range(len(tids))], holes, snps, col_off

    def _select_call(self, flags: int):
        sm, nl = self.small, self.index.n_loci
        base = sm.data_ptr()
        native.check(self.lib.mmlst_select_dev(native.ptr(self.sum_as), native.ptr(self.n_hit), native.ptr(self.first_idx), native.ptr(self.locus_rows),
                                               native.ptr(self.locus_start), native.ptr(self.allele_num), self.n_ref, native.ptr(self.species_of_locus),
                                               native.ptr(self.genes_in_db), nl, len(self.species_names), self.penalty, self.nloci,
                                               native.ptr(self.contig_start_d), native.ptr(self.ref_len_d), native.ptr(self.db_off_d),
                                               int(os.environ.get("MMLST_CHUNK_RECORDS", "0")),   # 0 = the library's rule (mmlst_chunk_records); profiling knob
                                               native.ptr(self.scratch), int(self.scratch.shape[0]), base + 4 * self.o_hdr, base + 4 * self.o_tid,
                                               base + 4 * self.o_sp, base + 4 * self.o_col, native.ptr(self.db_start_d), native.ptr(self.chunks_d),
                                               self.max_chunks, flags | (native.SELECT_LOCAL if self.owner else 0), native.ptr(self.counters),
                                               base + 4 * self.o_first, self._stream()))

    def _consensus_call(self, flags: int):
        nl = self.index.n_loci
        base = self.small.data_ptr()
        native.check(self.lib.mmlst_consensus_indirect_dev(native.ptr(self.counts), native.ptr(self.db_ascii_d), native.ptr(self.db_start_d),
                                                           base + 4 * self.o_col, nl, base + 4 * self.o_hdr, self.mincov, native.ptr(self.cons),
                                                           base + 4 * self.o_holes, base + 4 * self.o_snps, flags, self._stream()))

    def _pileup_call(self):
        s = self.s
        native.check(self.lib.mmlst_pileup_indirect_dev(native.ptr(s.p_recs), native.ptr(s.planes), native.ptr(self.chunks_d),
                                                        self.small.data_ptr() + 4 * self.o_hdr, int(s.max_row_words), self.minscore, self.max_xM,
                                                        native.ptr(self.counts), self.impl, self._stream()))

    def _pileup_consensus_call(self, flags: int):
        """Pileup and consensus of the pass in ONE launch (csrc/pileup.cuh FusedConsensus): the CTA finishing the last chunk of a locus calls it."""
        s, nl = self.s, self.index.n_loci
        base = self.small.data_ptr()
        native.check(self.lib.mmlst_pileup_consensus_indirect_dev(
            native.ptr(s.p_recs), native.ptr(s.planes), native.ptr(self.chunks_d), base + 4 * self.o_hdr, int(s.max_row_words), self.minscore, self.max_xM,
            native.ptr(self.counts), native.ptr(self.db_ascii_d), native.ptr(self.db_start_d), base + 4 * self.o_col, nl, self.mincov, native.ptr(self.cons),
            base + 4 * self.o_holes, base + 4 * self.o_snps, flags, native.ptr(self.ticket), self._stream()))

    def _enqueue(self):
        """Everything of one pass on the current stream, no host synchronisation and no memset: score -> [all-reduce] ->
        select -> pileup -> [all-reduce] -> consensus -> ONE D2H into a pinned buffer.  Selection and consensus reset
        what they read, so the pass starts from and ends in the empty-table state."""
        if not self._clean:
            self.reset_tables()
        self.run_score(reset=False)
        if self.want_tables:  # the score tables leave the device before the selection consumes them (`.out` log / screen table)
            self._enqueue_tables()
        self._timed("select", lambda: self._select_call(native.SELECT_CONSUME | native.SELECT_SCRATCH_CLEAN))
        self.launches += 1
        if self.fused_tail and self.impl != 1 and not (self.dist and not self.owner):
            # no exchange between the two: pileup + consensus as one launch
            self._timed("pileup+consensus", lambda: self._pileup_consensus_call(native.CONSENSUS_CONSUME))
            self.launches += 1
        else:
            self._timed("pileup", self._pileup_call)
            self.launches += 1
            if self.dist and not self.owner:
                dist.allreduce_counts(self.counts, self.group)
            self._timed("consensus", lambda: self._consensus_call(native.CONSENSUS_CONSUME))
            self.launches += 1
        if self.p2p:  # the pass's only exchange, by our own kernels: block -> every peer's memory, then wait for theirs
            native.check(self.lib.mmlst_xchg_publish_dev(native.ptr(self.out), self.out_bytes, native.ptr(self.peer_base), self.rank, self.world,
                                                         self.x_half, self.x_slot, self.x_flag_off, native.ptr(self.x_epoch), self._stream()))
            native.check(self.lib.mmlst_xchg_await_dev(native.ptr(self.xbuf), self.out_bytes, self.world, self.x_half, self.x_slot, self.x_flag_off,
                                                       native.ptr(self.out_all), native.ptr(self.x_epoch), native.ptr(self.x_ticket),
                                                       self.out_all.data_ptr() + self.world * self.out_bytes, self._stream()))
            self.launches += 2
            self.out_h.copy_(self.out_all, non_blocking=True)
        elif self.owner:  # the same exchange as ONE NCCL all-gather
            torch.distributed.all_gather_into_tensor(self.out_all[: self.world * self.out_bytes], self.out, group=self.group)
            self.out_h.copy_(self.out_all, non_blocking=True)
        else:
            self.out_h.copy_(self.out, non_blocking=True)
        self._clean = True

    def time_kernels(self, reps: int = 20, alt: Optional["DevicePipeline"] = None, flush: Optional[torch.Tensor] = None) -> Dict[str, float]:
        """Average device time (ms) of every kernel of the pass, always from a cold L2.
        score: `reps` back-to-back launches between two CUDA events on the launching stream, alternating between this
        pipeline's sample and `alt`'s (two samples together exceed the L2, so every launch streams from HBM; back-to-back
        amortises the event/launch gap a single launch would carry).
        select / pileup / consensus work on tables and a depth-capped pileup stream that FIT the L2: `flush` (a buffer
        larger than the L2) is rewritten before every launch and each launch gets its own event pair (the ~2 us event
        gap is included: an upper bound).  Without `flush` they are timed back to back like the score kernel (warm L2).
        The tables hold a finished pass when this is called; they are garbage afterwards (the next step resets them)."""
        pipes = [self] + ([alt] if alt is not None else [])
        for p in pipes:
            p.reset_tables()
            p.run_score(reset=False)  # tables of a finished scoring pass (all-reduced when distributed)
            p._select_call(native.SELECT_SCRATCH_CLEAN)
        torch.cuda.current_stream(self.dev).synchronize()
        out: Dict[str, float] = {}
        saved = [p.dist for p in pipes]
        for p in pipes:
            p.dist = False  # kernels only: no collectives inside the loops
        try:
            for name in ("select", "pileup", "consensus", "score"):
                for p in pipes:
                    p._launch_one(name)  # warm
                if name == "score" or flush is None:
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    for i in range(reps):
                        pipes[i % len(pipes)]._launch_one(name)
                    b.record()
                    b.synchronize()
                    out[name] = a.elapsed_time(b) / reps
                else:
                    pairs = []
                    for i in range(reps):
                        flush.zero_()
                        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        a.record()
                        pipes[i % len(pipes)]._launch_one(name)
                        b.record()
                        pairs.append((a, b))
                    torch.cuda.current_stream(self.dev).synchronize()
                    out[name] = float(np.mean([a.elapsed_time(b) for a, b in pairs]))
        finally:
            for p, d in zip(pipes, saved):
                p.dist = d
                p._clean = False
        return out

    def time_score_variants(self, reps: int = 20, alt: Optional["DevicePipeline"] = None) -> Dict[str, float]:
        """Average device time (ms) of the run-length score kernel in each of its forms (mmlst_set_score_variant), timed like
        time_kernels() times it (back to back, alternating two samples, cold L2); every form must leave the same tables.
        Keys: the form, plus 'h' when the L2 residency hints are on.  Leaves the library on the last form tried: the caller restores its own."""
        pipes = [self] + ([alt] if alt is not None else [])
        out: Dict[str, float] = {}
        want = None
        keys = ["0", "1", "2", "3", "4", "5", "2h", "3h", "4h", "5h"]  # "h": ring form with the L2 residency hints
        if self.use_qc:
            keys += ["6", "6h", "6g10", "6g12"]  # pair-fused ring (per-chunk len(SEQ) streams only); gNN: grid of NN/8 resident waves
        if self.code16 is not None:
            keys += ["7", "7h"]  # form 6 over the compact 2 B / record stream
        grid0 = self.lib.mmlst_set_score_grid_scale(-1)
        for key in keys:
            v = int(key[0])
            self.lib.mmlst_set_score_variant(v)
            self.lib.mmlst_set_score_l2_hints(1 if key[1:2] == "h" else 0)
            self.lib.mmlst_set_score_grid_scale(int(key.split("g")[1]) if "g" in key else grid0)
            self.reset_tables()
            self._score_call()
            torch.cuda.current_stream(self.dev).synchronize()
            got = [self.zscore.clone(), self.first_idx.clone()]
            if want is None:
                want = got
            assert all(torch.equal(a, b) for a, b in zip(got, want)), "score kernel form %s disagrees with form 0" % key
            for p in pipes:
                p._score_call()  # warm
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(reps):
                pipes[i % len(pipes)]._score_call()
            b.record()
            b.synchronize()
            out[key] = a.elapsed_time(b) / reps
        self.lib.mmlst_set_score_grid_scale(grid0)
        for p in pipes:
            p._clean = False
        return out

    def time_score_half(self, reps: int = 20, alt: Optional["DevicePipeline"] = None) -> Dict[str, float]:
        """The score kernel over the first half / quarter of the resident stream (timing only; the tables are garbage
        afterwards): t(n) at three sizes separates the per-launch fixed cost from the streaming rate."""
        pipes = [self] + ([alt] if alt is not None else [])
        out: Dict[str, float] = {}
        full = [p.s.as0 for p in pipes]
        n = int(self.s.as0.shape[0])
        try:
            for frac in (1, 2, 4):
                m = (n // frac) & ~255
                for p, f in zip(pipes, full):
                    p.s.as0 = f[:m]
                for p in pipes:
                    p._score_call()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for i in range(reps):
                    pipes[i % len(pipes)]._score_call()
                b.record()
                b.synchronize()
                out["1/%d" % frac] = a.elapsed_time(b) / reps
        finally:
            for p, f in zip(pipes, full):
                p.s.as0 = f
                p._clean = False
        return out

    def _launch_one(self, name: str):
        s = self.s
        if name == "score":
            self._score_call()
        elif name == "select":
            self._select_call(native.SELECT_SCRATCH_CLEAN)  # tables left intact: every repetition does the same work
        elif name == "pileup":
            self._pileup_call()
        elif name == "consensus":
            self._consensus_call(0)
        else:
            raise ValueError(name)

    def _init_p2p(self):
        """Symmetric (peer-mapped) exchange buffer of this pipeline: torch's symmetric-memory allocator provides the
        allocation and the address exchange; the data path is csrc/exchange.cu."""
        import torch.distributed._symmetric_memory as symm
        grp = self.group if self.group is not None else torch.distributed.group.WORLD
        self.rank = torch.distributed.get_rank(grp)
        self.x_slot = (self.out_bytes + 127) // 128 * 128
        self.x_half = self.world * self.x_slot
        self.x_flag_off = 2 * self.x_half
        self.xbuf = symm.empty(self.x_flag_off + 128 * ((8 * self.world + 127) // 128), dtype=torch.uint8, device=self.dev)
        self.xbuf.zero_()
        torch.cuda.synchronize(self.dev)
        self.xhdl = symm.rendezvous(self.xbuf, grp)  # collective: exchanges the handles, maps every peer's buffer
        ptrs = [int(x) for x in self.xhdl.buffer_ptrs]
        assert len(ptrs) == self.world and ptrs[self.rank] == self.xbuf.data_ptr(), "symmetric buffer: unexpected peer table"
        self.peer_base = torch.tensor(ptrs, dtype=torch.int64, device=self.dev)
        self.x_epoch = torch.zeros(1, dtype=torch.int64, device=self.dev)
        self.x_ticket = torch.zeros(1, dtype=torch.int32, device=self.dev)
        torch.cuda.synchronize(self.dev)
        torch.distributed.barrier(grp)  # every buffer is zeroed and mapped before anyone publishes

    def _finish_owner(self):
        nl = self.index.n_loci
        blocks, total, ignored = [], 0, 0
        if self.p2p and int(self.out_h[self.world * self.out_bytes:].view(torch.int32)[0]) != 0:
            raise RuntimeError("peer-memory exchange timed out waiting for a peer's result block")
        for r in range(self.world):
            blk = self.out_h[r * self.out_bytes:(r + 1) * self.out_bytes]
            h = blk[: self.n_small * 4].view(torch.int32).numpy()
            cons = blk[self.n_small * 4:].numpy()
            n = int(h[0])
            total += int(h[6:8].view(np.uint64)[0]); ignored += int(h[8:10].view(np.uint64)[0])
            if h[3] & 2:
                raise RuntimeError("chunk list overflow")
            tids = h[self.o_tid:self.o_tid + n]
            if self.bad_len[tids].any():
                raise IndexError("string index out of range: BAM LN > DB sequence length (metaMLST_functions.py:267)")
            col = h[self.o_col:self.o_col + n + 1]
            blocks.append({"tid": tids.tolist(), "species": h[self.o_sp:self.o_sp + n].tolist(),
                           "first": h[self.o_first:self.o_first + n].view(np.uint32).tolist(),
                           "payload": [(cons[col[i]:col[i + 1]].tobytes().decode("latin-1"), int(h[self.o_holes + i]), int(h[self.o_snps + i])) for i in range(n)]})
        self.total_reads, self.ignored_reads = total, ignored
        merged = dist.merge_owner_blocks(blocks, self.species_names, self.genes_in_db_h, self.nloci)
        return {sp: [(self.index.ref_names[t], seq, holes, snps) for t, (seq, holes, snps) in lst] for sp, lst in merged}

    def _finish(self):
        if self.owner:
            return self._finish_owner()
        h = self.small_h.numpy()
        n = int(h[0])
        self.total_reads = int(h[6:8].view(np.uint64)[0])      # metamlst.py:130 totalReads
        self.ignored_reads = int(h[8:10].view(np.uint64)[0])   # metamlst.py:129 ignoredReads
        if h[3] & 1:
            raise RuntimeError("Database is broken: a species has more detected loci than the genes table lists (metamlst.py:188)")
        if h[3] & 2:
            raise RuntimeError("chunk list overflow")
        tids = h[self.o_tid:self.o_tid + n]
        if self.bad_len[tids].any():
            raise IndexError("string index out of range: BAM LN > DB sequence length (metaMLST_functions.py:267)")
        col = h[self.o_col:self.o_col + n + 1]
        cons = self.cons_h.numpy()
        out: Dict[str, list] = {}
        for i in range(n):
            out.setdefault(self.species_names[int(h[self.o_sp + i])], []).append(
                (self.index.ref_names[int(tids[i])], cons[col[i]:col[i + 1]].tobytes().decode("latin-1"), int(h[self.o_holes + i]), int(h[self.o_snps + i])))
        return out

    def _enqueue_tables(self):
        if self._tables_h is None:
            self._tables_h = (torch.zeros(self.zscore.shape[0], dtype=torch.int64).pin_memory(), torch.zeros(self.n_ref, dtype=torch.int32).pin_memory())
        self._tables_h[0].copy_(self.zscore, non_blocking=True)
        self._tables_h[1].copy_(self.first_idx, non_blocking=True)

    def tables(self):
        """(sum_as int64, n_hit uint32, first_idx uint32) of the last finished pass run with `want_tables` (host numpy views)."""
        z, f = self._tables_h
        n = self.n_ref
        return z[:n].numpy(), z[n + 2:].view(torch.int32)[:n].numpy().view(np.uint32), f.numpy().view(np.uint32)

    def step(self):
        """One pass of the hot path, no host round trip between the stages.
        Returns {species: [(contig, consensus, holes, snps)]} in the reference's dict order."""
        self._enqueue()
        torch.cuda.current_stream(self.dev).synchronize()
        return self._finish()

    def capture(self):
        """Record the pass once into a CUDA graph (one launch per step afterwards; kernels, memsets, NCCL calls and
        the D2H copies are all graph nodes)."""
        assert self.timers is None, "per-kernel timers are not capturable"
        self._enqueue()  # warm-up outside capture (lazy attribute setting, NCCL channels)
        torch.cuda.synchronize(self.dev)
        n0 = self.launches
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self._enqueue()
        self.launches_per_step = self.launches - n0
        self.launches = n0

    def step_graph(self):
        if not self._clean:
            self.reset_tables()  # the captured pass contains no memset: it starts from the empty-table state it leaves behind
        self.graph.replay()
        self.launches += self.launches_per_step
        torch.cuda.current_stream(self.dev).synchronize()
        return self._finish()

    def enqueue_step(self):
        """Queue one pass without waiting for it (cohort mode: passes run back to back, results are read from the pinned
        output block after a synchronisation with `collect()`)."""
        if getattr(self, "graph", None) is not None:
            if not self._clean:
                self.reset_tables()
            self.graph.replay()
            self.launches += self.launches_per_step
        else:
            self._enqueue()

    def collect(self):
        torch.cuda.current_stream(self.dev).synchronize()
        return self._finish()

    def step_host_select(self):
        """Same pass with the selection done on the host in Python floats (cross-check of the device selection)."""
        self.run_score()
        chosen, _raw = self.select()
        tids = [t for _sp, ts in chosen for t in ts]
        out: Dict[str, list] = {}
        if tids:
            seqs, holes, snps, _ = self.run_pileup_consensus(tids)
            i = 0
            for sp, ts in chosen:
                for t in ts:
                    out.setdefault(sp, []).append((self.index.ref_names[t], seqs[i], int(holes[i]), int(snps[i])))
                    i += 1
        return out


class CohortLanes:
    """Cohort mode (BASELINE.json configs[3], SURVEY.md 8f rank 2): consecutive samples are independent, so pass i+1 is
    queued on another stream than pass i -- the latency-bound tail of a pass (selection, capped pileup, consensus: small
    grids) runs underneath the HBM-bound scoring kernel of the next one.  Every lane is a DevicePipeline with its own
    accumulators / output block and its own CUDA graph; lanes may share the input streams (the bench re-types one sample)
    or hold different samples (a real cohort)."""

    def __init__(self, make_pipe: Callable[[int], "DevicePipeline"], n_lanes: int = 2):
        """make_pipe(lane) -> DevicePipeline.  With torch.distributed every lane must get its OWN process group
        (communicator): collectives of consecutive passes overlap, and NCCL serialises nothing across communicators."""
        self.pipes = [make_pipe(lane) for lane in range(n_lanes)]
        self.dev = self.pipes[0].dev
        self.streams = [torch.cuda.Stream(device=self.dev) for _ in range(n_lanes)]
        self.captured = False

    def warm_and_capture(self, graph: bool = True):
        res = []
        for p, st in zip(self.pipes, self.streams):
            with torch.cuda.stream(st):
                r = p.step()
                if graph:
                    p.capture()
                    assert p.step_graph() == r, "graph replay differs from the eager pass"
                res.append(r)
        self.captured = graph
        torch.cuda.synchronize(self.dev)
        return res

    def enqueue(self, i: int) -> None:
        lane = i % len(self.pipes)
        with torch.cuda.stream(self.streams[lane]):
            self.pipes[lane].enqueue_step()

    def fork(self, event: "torch.cuda.Event") -> None:
        """All lanes start after `event` (recorded on the timing stream)."""
        for st in self.streams:
            st.wait_event(event)

    def join(self) -> None:
        """The current stream waits for everything queued on the lanes."""
        cur = torch.cuda.current_stream(self.dev)
        for st in self.streams:
            ev = torch.cuda.Event()
            ev.record(st)
            cur.wait_event(ev)

    def collect(self):
        out = []
        for p, st in zip(self.pipes, self.streams):
            with torch.cuda.stream(st):
                out.append(p.collect())
        return out

    @property
    def launches(self) -> int:
        return sum(p.launches for p in self.pipes)


def device_select(index: api.AlleleIndex, sum_as: np.ndarray, n_hit: np.ndarray, first_idx: np.ndarray, penalty: int = 100,
                  nloci: int = 100, genes_in_db: Optional[Dict[str, int]] = None, device: str = "cuda:0"):
    """mmlst_select_dev on given score tables -> [(species, [tid per locus])] in the reference's dict order
    (same shape as api.fast_select; used by the parity tests of the device-side rounding / ordering)."""
    lib = native.lib()
    dev = torch.device(device)
    n_ref, nl = len(index.ref_names), index.n_loci
    names: List[str] = []
    sid: Dict[str, int] = {}
    sol = np.zeros(nl, np.int32)
    for l, (sp, _g) in enumerate(index.locus_names):
        if sp not in sid:
            sid[sp] = len(names)
            names.append(sp)
        sol[l] = sid[sp]
    gdb = np.asarray([(genes_in_db or {}).get(sp, int((sol == i).sum())) for i, sp in enumerate(names)], np.int32)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    t_sum, t_n, t_f = d(sum_as.astype(np.int64)), d(n_hit.astype(np.uint32).view(np.int32)), d(first_idx.astype(np.uint32).view(np.int32))
    order = np.argsort(index.locus_of, kind="stable").astype(np.uint32)
    identity = np.array_equal(order, np.arange(order.shape[0], dtype=order.dtype))   # rows already grouped by locus: no row list (include/mmlst.h)
    t_rows, t_start = (None if identity else d(order.view(np.int32))), d(np.searchsorted(index.locus_of[order], np.arange(nl + 1)).astype(np.int32))
    t_an = d(np.asarray([int(a) for a in index.allele], np.int64).astype(np.uint32).view(np.int32))
    t_sol, t_gdb = d(sol), d(gdb)
    t_cs, t_rl, t_dbo = d(np.zeros(n_ref + 1, np.int64)), d(np.ones(n_ref, np.int32)), d(np.zeros(n_ref + 1, np.int64))
    scratch = torch.zeros(nl * 12 + 64, dtype=torch.uint8, device=dev)
    small = torch.zeros(16 + 3 * nl + 8, dtype=torch.int32, device=dev)
    dbs = torch.zeros(nl + 1, dtype=torch.int64, device=dev)
    chunks = torch.zeros(8 * (nl + 8), dtype=torch.int32, device=dev)
    base = small.data_ptr()
    native.check(lib.mmlst_select_dev(native.ptr(t_sum), native.ptr(t_n), native.ptr(t_f), native.ptr(t_rows), native.ptr(t_start), native.ptr(t_an),
                                      n_ref, native.ptr(t_sol), native.ptr(t_gdb), nl, len(names), int(penalty), int(nloci), native.ptr(t_cs),
                                      native.ptr(t_rl), native.ptr(t_dbo), 0, native.ptr(scratch), int(scratch.shape[0]), base,
                                      base + 4 * 16, base + 4 * (16 + nl), base + 4 * (16 + 2 * nl), native.ptr(dbs), native.ptr(chunks), nl + 8,
                                      0, 0, 0, torch.cuda.current_stream(dev).cuda_stream))
    h = small.cpu().numpy()
    n = int(h[0])
    out: Dict[str, List[int]] = {}
    for i in range(n):
        out.setdefault(names[int(h[16 + nl + i])], []).append(int(h[16 + i]))
    return list(out.items()), int(h[3])
