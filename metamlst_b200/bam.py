"""BAM -> SoaHost through the native unpacker (`mmlst_bam_unpack`, csrc/bam_unpack.cpp).

Stands where the reference shells out to `samtools view -h -` (metamlst.py:96), opens the file with pysam
(cmseq/cmseq.py:54) and rewrites it with `samtools sort` / `samtools index` (metaMLST_functions.py:237-247).  The
arrays are views of memory owned by the native handle (page-locked when a CUDA device is present), kept alive by the
returned SoaHost.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np

from . import native, packing


class UnpackOpts(C.Structure):
    _fields_ = [("minqual", C.c_int), ("max_depth", C.c_uint32), ("sentinel_nodes", C.c_uint32), ("n_threads", C.c_int),
                ("pinned", C.c_int), ("assume_sorted", C.c_int), ("want_qhash", C.c_int), ("check_crc", C.c_int), ("lenient_tags", C.c_int)]


class BamInfo(C.Structure):
    _fields_ = [("soa", native.Soa), ("qhash", C.c_void_p), ("ref_len", C.c_void_p), ("ref_names", C.c_char_p),
                ("header_text", C.c_char_p), ("n_dropped_by_cap", C.c_uint64), ("n_unmapped_flag", C.c_uint64),
                ("presorted", C.c_int), ("minqual", C.c_int), ("max_depth", C.c_uint32), ("seconds", C.c_double * 5), ("n_untagged", C.c_uint64)]


class _Handle:
    def __init__(self, h):
        self.h = h

    def __del__(self):
        try:
            if self.h:
                native.lib().mmlst_bam_free(self.h)
                self.h = None
        except Exception:  # noqa: BLE001
            pass


def _view(addr: Optional[int], n: int, dtype) -> np.ndarray:
    dt = np.dtype(dtype)
    if not addr or n == 0:
        return np.zeros(0, dtype=dt)
    buf = (C.c_uint8 * (n * dt.itemsize)).from_address(addr)
    return np.frombuffer(buf, dtype=dt, count=n)


def unpack_bam(path: str, minqual: int = packing.DEFAULT_MINQUAL, max_depth: Optional[int] = packing.DEFAULT_MAX_DEPTH,
               presorted: bool = False, threads: int = 0, pinned: bool = True, want_qhash: bool = True,
               sentinel_nodes: int = 1, lenient_tags: bool = False) -> packing.SoaHost:
    """Unpack a BAM once into the score stream + pileup stream (include/mmlst.h).  `presorted` = metamlst.py --presorted
    (file order is kept and must be coordinate order); otherwise records are put in `samtools sort` order and
    `orig_idx` carries the file order stage 1 saw (H5).  max_depth=None disables the htslib depth cap.  lenient_tags: keep records
    MetaMLST itself would crash on (no integer 1st / 4th aux field, no AS:i / XM:i) -- for cmseq users without a tag filter; the stream
    is then marked `lenient` (it cannot be scored) and `n_untagged` counts the pileup records without the two tags."""
    lib = native.lib()
    o = UnpackOpts(int(minqual), int(max_depth or 0), int(sentinel_nodes), int(threads), 1 if pinned else 0,
                   1 if presorted else 0, 1 if want_qhash else 0, 1, 1 if lenient_tags else 0)
    h = C.c_void_p()
    native.check(lib.mmlst_bam_unpack(path.encode(), C.byref(o), C.byref(h)))
    keep = _Handle(h)
    info = BamInfo()
    native.check(lib.mmlst_bam_info(h, C.byref(info)))
    s = info.soa
    n, P, n_ref = int(s.n_rec), int(s.n_prec), int(s.n_ref)
    names = info.ref_names.decode("latin-1").split("\n") if n_ref else []
    soa = packing.SoaHost(
        names, _view(info.ref_len, n_ref, np.uint32).astype(np.int32),
        _view(s.tid, n, np.uint32), _view(s.as0, n, np.int16), _view(s.xm3, n, np.uint8), _view(s.qlen, n, np.uint16),
        _view(s.orig_idx, n, np.uint32) if s.orig_idx else None,
        _view(s.p_recs, P, packing.PREC_DTYPE), _view(s.planes, int(s.n_plane_words), np.uint32), int(s.max_row_words),
        _view(s.contig_start, n_ref + 1, np.uint64), int(info.minqual), int(info.max_depth), int(info.n_dropped_by_cap))
    if s.run_tid:
        nr = int(s.n_runs)
        soa.run_tid, soa.run_start = _view(s.run_tid, nr, np.uint32), _view(s.run_start, nr + 1, np.uint32)
        soa.chunk_run = _view(s.chunk_run, (n + 255) // 256, np.uint32)
        soa.chunk_qlen = _view(s.chunk_qlen, (n + 255) // 256, np.uint16) if s.chunk_qlen else None
        if nr > 0.125 * n:  # name-grouped input: the explicit tid form is the smaller one
            soa.run_tid = soa.run_start = soa.chunk_run = soa.chunk_qlen = None
    soa.qhash = _view(info.qhash, 2 * n, np.uint64).reshape(n, 2) if info.qhash else None
    soa.header_text = (info.header_text or b"").decode("latin-1")
    soa.unpack_seconds = dict(zip(("read", "inflate", "parse", "sort", "pack"), [float(x) for x in info.seconds]))
    soa.lenient, soa.n_untagged = bool(lenient_tags), int(info.n_untagged)
    soa._keep = (keep,)
    return soa


# ----------------------------------------------------------------------------------------------------------------
# device-side ingest (csrc/ingest.cu): compressed bytes in, packed streams resident in HBM out
# ----------------------------------------------------------------------------------------------------------------
class DevBamInfo(C.Structure):
    _fields_ = [("tid", C.c_void_p), ("as0", C.c_void_p), ("xm3", C.c_void_p), ("qlen", C.c_void_p), ("orig_idx", C.c_void_p), ("qhash", C.c_void_p),
                ("run_tid", C.c_void_p), ("run_start", C.c_void_p), ("chunk_run", C.c_void_p), ("chunk_qlen", C.c_void_p), ("n_runs", C.c_uint32),
                ("p_recs", C.c_void_p), ("planes", C.c_void_p),
                ("n_rec", C.c_uint64), ("n_prec", C.c_uint64), ("n_plane_words", C.c_uint64), ("max_row_words", C.c_uint32),
                ("contig_start", C.c_void_p), ("ref_len", C.c_void_p), ("ref_names", C.c_char_p), ("header_text", C.c_char_p), ("n_ref", C.c_uint32),
                ("n_dropped_by_cap", C.c_uint64), ("n_unmapped_flag", C.c_uint64), ("n_bgzf_blocks", C.c_uint64), ("compressed_bytes", C.c_uint64),
                ("inflated_bytes", C.c_uint64), ("presorted", C.c_int), ("minqual", C.c_int), ("max_depth", C.c_uint32), ("boundary_repairs", C.c_int),
                ("seconds", C.c_double * 8), ("n_untagged", C.c_uint64)]


class _DevHandle:
    def __init__(self, h):
        self.h = h

    def __del__(self):
        try:
            if self.h:
                native.lib().mmlst_dev_bam_free(self.h)
                self.h = None
        except Exception:  # noqa: BLE001
            pass


class _DevArray:
    """A device array owned by the native handle, handed to torch through the CUDA array interface (no copy)."""

    def __init__(self, addr: int, n: int, typestr: str, keep):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (addr, False), "version": 2, "strides": None}
        self._keep = keep


class PinnedPool:
    """Page-locked staging buffers, reused: cudaHostAlloc costs milliseconds per call (tens for a large file), a cohort reads hundreds
    of files.  get(n) hands out a uint8 tensor of at least n bytes, put(t) takes it back."""

    def __init__(self):
        import threading
        self._lock = threading.Lock()
        self._free = []

    def get(self, n: int):
        import torch
        with self._lock:
            best = None
            for i, t in enumerate(self._free):
                if t.numel() >= n and (best is None or t.numel() < self._free[best].numel()):
                    best = i
            if best is not None:
                return self._free.pop(best)
        return torch.empty(max(int(n * 1.25), 1 << 20), dtype=torch.uint8, pin_memory=torch.cuda.is_available())

    def put(self, t) -> None:
        base = getattr(t, "_pool_base", None)
        if base is not None:
            with self._lock:
                if len(self._free) < 16:
                    self._free.append(base)


POOL = PinnedPool()


def read_pinned(path: str, pool: Optional[PinnedPool] = None):
    """The file's bytes in page-locked memory (one async DMA to the device): a uint8 torch tensor.  With a pool the buffer is a
    recycled one: give it back with pool.put(tensor) once the ingest has consumed it."""
    import torch
    size = os.path.getsize(path)
    if pool is not None:
        base = pool.get(size)
    else:
        base = torch.empty(max(size, 1), dtype=torch.uint8, pin_memory=torch.cuda.is_available())
    with open(path, "rb") as fh:
        got = fh.readinto(memoryview(base.numpy())[:size]) if size else 0
    if got != size:
        raise IOError("short read on %s" % path)
    view = base[:size]
    if pool is not None:
        view._pool_base = base
    return view


def ingest_bam(source, device=0, minqual: int = packing.DEFAULT_MINQUAL, max_depth: Optional[int] = packing.DEFAULT_MAX_DEPTH,
               presorted: bool = False, want_qhash: bool = True, sentinel_nodes: int = 1, check_crc: bool = False, lenient_tags: bool = False):
    """BAM -> streams.DeviceStreams WITHOUT the sample ever being unpacked on the host: the compressed file crosses PCIe, the
    hardware decompression engine inflates the BGZF blocks, kernels chain / parse / sort / depth-cap / pack the records
    (csrc/ingest.cu).  `source`: a path, or a uint8 torch tensor / numpy array holding the file's bytes (page-locked for an
    asynchronous copy: `read_pinned`).  Same streams, same refusals as `unpack_bam`; raises MmlstError(MMLST_E_CUDA) on a device
    without hardware DEFLATE.  `check_crc`: also check every BGZF block's CRC32 against its trailer on the device, as `unpack_bam`
    always does (MmlstError(MMLST_E_BAM) "CRC mismatch in BGZF block k"); without it the DEFLATE stream and ISIZE are still checked.
    `lenient_tags`: as `unpack_bam` -- the streams are marked `lenient` (they cannot be scored) and carry `n_untagged`."""
    import torch
    dev = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
    data = read_pinned(source) if isinstance(source, str) else source
    addr = data.data_ptr() if hasattr(data, "data_ptr") else data.ctypes.data
    nbytes = int(data.numel() if hasattr(data, "numel") else data.size)
    lib = native.lib()
    o = UnpackOpts(int(minqual), int(max_depth or 0), int(sentinel_nodes), 0, 1, 1 if presorted else 0, 1 if want_qhash else 0,
                  1 if check_crc else 0, 1 if lenient_tags else 0)
    h = C.c_void_p()
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        native.check(lib.mmlst_bam_ingest(dev.index or 0, addr, nbytes, C.byref(o), stream, C.byref(h)))
    return _dev_streams(_DevHandle(h), dev, want_qhash, lenient_tags)


def _dev_streams(keep, dev, want_qhash: bool, lenient_tags: bool = False):
    """streams.DeviceStreams over the arrays of an mmlst_dev_bam handle (no copy: the handle stays alive with the streams)."""
    import torch
    from . import streams
    info = DevBamInfo()
    native.check(native.lib().mmlst_dev_bam_info(keep.h, C.byref(info)))
    n, P, n_ref, nr = int(info.n_rec), int(info.n_prec), int(info.n_ref), int(info.n_runs)

    def t(addr_, count, typestr, dtype):
        if not addr_ or count == 0:
            return torch.zeros(0, dtype=dtype, device=dev)
        return torch.as_tensor(_DevArray(addr_, count, typestr, keep), device=dev)

    s = streams.DeviceStreams()
    s._keep = keep
    s.ref_names = info.ref_names.decode("latin-1").split("\n") if n_ref else []
    s.ref_lens = _view(info.ref_len, n_ref, np.uint32).astype(np.int32)
    s.header_text = (info.header_text or b"").decode("latin-1")
    s.minqual, s.max_depth, s.n_dropped = int(info.minqual), int(info.max_depth), int(info.n_dropped_by_cap)
    s.idx_base = 0
    s.tid, s.as0 = t(info.tid, n, "<i4", torch.int32), t(info.as0, n, "<i2", torch.int16)
    s.xm3, s.qlen = t(info.xm3, n, "|u1", torch.uint8), t(info.qlen, n, "<i2", torch.int16)
    s.orig_idx = t(info.orig_idx, n, "<i4", torch.int32) if info.orig_idx else None
    s.qhash = t(info.qhash, 2 * n, "<i8", torch.int64).view(n, 2) if (info.qhash and want_qhash) else None
    s.p_recs = t(info.p_recs, 4 * P, "<i4", torch.int32).view(P, 4)
    s.planes = t(info.planes, int(info.n_plane_words), "<i4", torch.int32)
    s.n_prec, s.max_row_words = P, int(info.max_row_words)
    s.contig_start = _view(info.contig_start, n_ref + 1, np.uint64).copy()
    s.run_tid = s.run_start = s.chunk_run = s.chunk_qlen = None
    if nr and nr <= 0.125 * n:  # name-grouped streams keep the explicit tid form (as unpack_bam does)
        s.run_tid, s.run_start = t(info.run_tid, nr, "<i4", torch.int32), t(info.run_start, nr + 1, "<i4", torch.int32)
        s.chunk_run = t(info.chunk_run, (n + 255) // 256, "<i4", torch.int32)
        s.chunk_qlen = t(info.chunk_qlen, (n + 255) // 256, "<i2", torch.int16) if info.chunk_qlen else None
    s.presorted = bool(info.presorted)
    s.ingest_seconds = dict(zip(("h2d", "inflate", "chain", "parse", "sort", "score_stream", "cap_compact", "pack"), [float(x) for x in info.seconds]))
    s.ingest_stats = {"bgzf_blocks": int(info.n_bgzf_blocks), "compressed_bytes": int(info.compressed_bytes), "inflated_bytes": int(info.inflated_bytes),
                      "boundary_repairs": int(info.boundary_repairs), "unmapped_flag": int(info.n_unmapped_flag)}
    if lenient_tags:   # pileup only: DevicePipeline refuses to score it, as the host score seams refuse a lenient SoaHost
        s.lenient, s.n_untagged = True, int(info.n_untagged)
    return s


def ingest_bam_sharded(path: str, device=0, group=None, locus_of=None, minqual: int = packing.DEFAULT_MINQUAL,
                       max_depth: Optional[int] = packing.DEFAULT_MAX_DEPTH, presorted: bool = False, want_qhash: bool = True,
                       sentinel_nodes: int = 1, check_crc: bool = False, lenient_tags: bool = False):
    """One BAM ingested by every rank of a torch.distributed group (metamlst_b200/shard.py): this rank inflates and parses a 1/W share
    of the BGZF blocks and returns its streams.DeviceStreams, the records of the loci it owns (locus_of[tid] % W == rank; default:
    the loci of api.AlleleIndex over the header's reference names) -- what `DeviceStreams.from_soa(unpack_bam(path), mode="loci")`
    gives, with orig_idx the explicit file index and the pileup stream of the owned contigs only.  Same options and the same refusals
    as `ingest_bam`: every rank raises the refusal the whole file gives, after the ranks agreed on it.  With `lenient_tags` each rank's
    `n_untagged` counts the untagged pileup records of its own contigs (their sum over the ranks is the file's)."""
    from . import shard
    coll = shard.TorchCollective(group)
    return coll.run(shard.ingest_steps(path, device, coll.rank, coll.world, locus_of=locus_of, minqual=minqual, max_depth=max_depth,
                                       presorted=presorted, want_qhash=want_qhash, sentinel_nodes=sentinel_nodes, check_crc=check_crc,
                                       lenient_tags=lenient_tags))


def ingest_bam_local(path: str, world: int, device=0, **kw):
    """Every rank of a `world`-rank sharded ingest (ingest_bam_sharded) run in turn in this process on one device: the list of the
    ranks' streams."""
    from . import shard
    return shard.run_local([shard.ingest_steps(path, device, r, world, **kw) for r in range(world)])
