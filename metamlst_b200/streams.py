"""Packed record streams resident in HBM (torch tensors on one device), in the layouts of include/mmlst.h.

`DeviceStreams.from_soa` is the bridge between a real sample and the device pipeline: BAM -> `bam.unpack_bam` (SoaHost,
page-locked) -> `from_soa` (one async copy per array) -> `pipeline.DevicePipeline`.  With several GPUs it also cuts the
shard a rank types:

  "ranges"  any record sharding (SURVEY.md 8e, north_star: "reads are sharded across the GPUs ... partial pileup-count and score
            tensors are allreduced"): rank r takes a contiguous range of the score stream (file-order indices kept through
            idx_base / orig_idx) and a contiguous range of the pileup stream.  The htslib depth cap was resolved at unpack over
            the WHOLE sample, i.e. before sharding, so counts add up exactly.  Goes with exchange="allreduce".  The records of one
            read name can fall on both sides of a cut: the coverage column merges the ranks' name tables before it adds their sums
            (DevicePipeline.run_coverage).
  "loci"    contig-aligned shards: rank r takes the score-stream records of loci l with l % world == r (orig_idx made explicit)
            and keeps the whole (depth-capped, hence small) pileup stream; it only ever chooses -- and piles up -- contigs of
            its own loci.  Goes with the owner-mode exchanges ("p2p", "gather").
"""
from __future__ import annotations

from typing import List, Optional

import numpy as np
import torch

from . import packing


class DeviceStreams:
    """Coordinate-sorted streams as torch tensors on one device (+ helpers to mirror them into a pinned SoaHost)."""

    def __init__(self):
        self.ref_names: List[str] = []
        self.ref_lens: Optional[np.ndarray] = None

    def to_host(self, pinned: bool = True) -> packing.SoaHost:
        def h(t, dt):
            a = t.detach().cpu().numpy()
            return a.view(dt) if a.dtype != dt else a
        recs = self.p_recs.detach().cpu().numpy().reshape(-1).view(packing.PREC_DTYPE)
        oi = getattr(self, "orig_idx", None)
        soa = packing.SoaHost(self.ref_names, self.ref_lens, h(self.tid, np.uint32), h(self.as0, np.int16), h(self.xm3, np.uint8),
                              h(self.qlen, np.uint16), None if oi is None else h(oi, np.uint32), recs, h(self.planes, np.uint32),
                              int(self.max_row_words), self.contig_start.copy(), self.minqual, self.max_depth, self.n_dropped)
        if getattr(self, "run_tid", None) is not None:
            soa.run_tid, soa.run_start, soa.chunk_run = h(self.run_tid, np.uint32), h(self.run_start, np.uint32), h(self.chunk_run, np.uint32)
            if getattr(self, "chunk_qlen", None) is not None:
                soa.chunk_qlen = h(self.chunk_qlen, np.uint16)
        return soa.pin() if pinned else soa

    def build_runs(self) -> "DeviceStreams":
        """Run-length form of the score stream on the device (include/mmlst.h, mmlst_score_runs_dev): run_tid, run_start,
        chunk_run as int32 tensors (bit patterns of the u32 arrays)."""
        n = int(self.tid.shape[0])
        self.run_tid = self.run_start = self.chunk_run = self.chunk_qlen = None
        if n == 0:
            return self
        assert n < 0xffffff00
        vals, counts = torch.unique_consecutive(self.tid, return_counts=True)
        start = torch.zeros(vals.shape[0] + 1, dtype=torch.int64, device=self.tid.device)
        start[1:] = torch.cumsum(counts, 0)
        first = torch.arange(0, n, 256, dtype=torch.int64, device=self.tid.device)
        self.chunk_run = (torch.searchsorted(start, first, right=True) - 1).to(torch.int32).contiguous()
        self.run_tid = vals.to(torch.int32).contiguous()
        self.run_start = start.to(torch.int32).contiguous()  # n < 2^32 - 256: the u32 bit pattern
        # len(SEQ) once per 256-record chunk when every chunk is uniform (mmlst_score_runs_qc_dev)
        nc = (n + 255) // 256
        q = self.qlen.to(torch.int32)
        pad = torch.full((nc * 256 - n,), int(q[-1].item()), dtype=torch.int32, device=q.device)
        q2 = torch.cat([q, pad]).view(nc, 256)
        if bool((q2 == q2[:, :1]).all().item()):
            self.chunk_qlen = q2[:, 0].to(torch.int16).contiguous()  # bit pattern of the u16
        return self

    def slice_ranges(self, rank: int, world: int) -> "DeviceStreams":
        """This rank's shard of device-resident streams, mode "ranges" (module text): a contiguous range of the score stream
        (file-order indices kept through idx_base / orig_idx) and a contiguous range of the pileup stream, rows rebased.  The
        depth cap was resolved over the whole sample when the streams were packed."""
        if world <= 1:
            return self
        dev = self.as0.device
        n, P = int(self.tid.shape[0]), int(self.n_prec)
        a, b = (n * rank) // world, (n * (rank + 1)) // world
        p0, p1 = (P * rank) // world, (P * (rank + 1)) // world
        s = DeviceStreams()
        s.ref_names, s.ref_lens = self.ref_names, self.ref_lens
        s.minqual, s.max_depth, s.n_dropped = self.minqual, self.max_depth, getattr(self, "n_dropped", 0)
        s.tid, s.as0, s.xm3, s.qlen = self.tid[a:b].contiguous(), self.as0[a:b].contiguous(), self.xm3[a:b].contiguous(), self.qlen[a:b].contiguous()
        oi = getattr(self, "orig_idx", None)
        s.orig_idx = None if oi is None else oi[a:b].contiguous()
        s.idx_base = (int(getattr(self, "idx_base", 0) or 0) + a) if oi is None else 0
        qh = getattr(self, "qhash", None)
        s.qhash = None if qh is None else qh[a:b].contiguous()
        total_words = int(self.planes.shape[0]) - packing.PLANE_SLACK_WORDS
        off = lambda j: (int(self.p_recs[j, 1].item()) & 0xFFFFFFFF) if j < P else total_words
        w0, w1 = (off(p0), off(p1)) if p1 > p0 else (0, 0)
        recs = self.p_recs[p0:p1].clone()
        if w0 and p1 > p0:
            recs[:, 1] = ((recs[:, 1].to(torch.int64) & 0xFFFFFFFF) - w0).to(torch.int32)
        s.p_recs = recs
        s.planes = torch.cat([self.planes[w0:w1], torch.zeros(packing.PLANE_SLACK_WORDS, dtype=torch.int32, device=dev)])
        s.n_prec, s.max_row_words = p1 - p0, int(self.max_row_words)
        cs = np.asarray(self.contig_start, dtype=np.int64)
        s.contig_start = (np.clip(cs, p0, p1) - p0).astype(np.uint64)
        s.run_tid = s.run_start = s.chunk_run = s.chunk_qlen = None
        if getattr(self, "run_tid", None) is not None and b > a:
            s.build_runs()
            if int(s.run_tid.shape[0]) > 0.125 * (b - a):
                s.run_tid = s.run_start = s.chunk_run = s.chunk_qlen = None
        return s

    # ------------------------------------------------------------------------------------------------------------
    @classmethod
    def from_soa(cls, soa: packing.SoaHost, device, rank: int = 0, world: int = 1, mode: str = "ranges",
                 locus_of: Optional[np.ndarray] = None, want_qhash: bool = False, stream=None) -> "DeviceStreams":
        """Upload an unpacked sample (or this rank's shard of it, see the module text).  Copies are asynchronous when the
        SoaHost is page-locked (`bam.unpack_bam(pinned=True)`, `SoaHost.pin()`); `idx_base` of the returned streams is the
        file-order index of its first score-stream record when no explicit orig_idx is carried."""
        dev = torch.device(device)
        s = cls()
        s.ref_names = list(soa.ref_names)
        s.ref_lens = np.asarray(soa.ref_lens, dtype=np.int32)
        s.minqual, s.max_depth, s.n_dropped = int(soa.minqual), int(soa.max_depth or 0), int(soa.n_dropped_by_cap)
        n, P = soa.n_rec, soa.n_prec
        s.idx_base = 0
        s.orig_idx = None
        s.qhash = None

        def up(a, dt=None):
            a = np.ascontiguousarray(a)
            if dt is not None and a.dtype != dt:
                a = a.view(dt)
            t = torch.from_numpy(a)
            return t.to(dev, non_blocking=True)

        if world > 1 and mode not in ("ranges", "loci"):
            raise ValueError("mode must be 'ranges' or 'loci'")
        if world > 1 and mode == "loci":
            if locus_of is None:
                raise ValueError("mode='loci' needs locus_of[tid]")
            keep = (np.asarray(locus_of)[soa.tid] % world) == rank
            sel = np.nonzero(keep)[0]
            tid, as0, xm3, qlen = soa.tid[sel], soa.as0[sel], soa.xm3[sel], soa.qlen[sel]
            oi = (soa.orig_idx[sel] if soa.orig_idx is not None else sel).astype(np.uint32)
            p0, p1 = 0, P
            qh = soa.qhash[sel] if (want_qhash and soa.qhash is not None) else None
            whole_runs = False
        else:
            a, b = (n * rank) // world, (n * (rank + 1)) // world
            tid, as0, xm3, qlen = soa.tid[a:b], soa.as0[a:b], soa.xm3[a:b], soa.qlen[a:b]
            oi = soa.orig_idx[a:b] if soa.orig_idx is not None else None
            s.idx_base = a if oi is None else 0
            p0, p1 = (P * rank) // world, (P * (rank + 1)) // world
            qh = soa.qhash[a:b] if (want_qhash and soa.qhash is not None) else None
            whole_runs = world == 1
        s.tid, s.as0, s.xm3, s.qlen = up(tid, np.int32), up(as0), up(xm3), up(qlen, np.int16)
        if oi is not None:
            s.orig_idx = up(oi, np.int32)
        if qh is not None:
            s.qhash = up(qh, np.int64)
        # pileup stream: records [p0, p1) and their plane rows (one contiguous word range), row offsets rebased
        recs = soa.p_recs[p0:p1]
        if p1 > p0:
            off = soa.p_row_off
            w0, w1 = int(off[p0]), int(off[p1])
            if w0:
                recs = recs.copy()
                recs["row_off"] -= np.uint32(w0)
            planes = soa.planes[w0:w1]
        else:
            planes = soa.planes[:0]
        s.p_recs = up(recs.view(np.int32).reshape(-1, 4)) if p1 > p0 else torch.zeros((0, 4), dtype=torch.int32, device=dev)
        s.planes = torch.cat([up(planes, np.int32), torch.zeros(packing.PLANE_SLACK_WORDS, dtype=torch.int32, device=dev)])
        s.n_prec = p1 - p0
        s.max_row_words = int(soa.max_row_words)
        cs = np.asarray(soa.contig_start, dtype=np.int64)
        s.contig_start = (np.clip(cs, p0, p1) - p0).astype(np.uint64)
        # run-length form of the score stream: taken over when the whole stream is uploaded, rebuilt on the device for a shard
        s.run_tid = s.run_start = s.chunk_run = s.chunk_qlen = None
        if whole_runs and soa.run_tid is not None:
            s.run_tid, s.run_start, s.chunk_run = up(soa.run_tid, np.int32), up(soa.run_start, np.int32), up(soa.chunk_run, np.int32)
            if soa.chunk_qlen is not None:
                s.chunk_qlen = up(soa.chunk_qlen, np.int16)
        elif soa.run_tid is not None and int(s.tid.shape[0]):
            s.build_runs()
            if int(s.run_tid.shape[0]) > 0.125 * int(s.tid.shape[0]):
                s.run_tid = s.run_start = s.chunk_run = s.chunk_qlen = None
        return s
