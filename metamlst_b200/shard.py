"""One BAM file ingested by W ranks (bam.ingest_bam_sharded): every rank inflates and parses 1/W of the BGZF blocks and receives the
records of the loci it owns (include/mmlst.h, "ONE BAM over W ranks").

The ingest is a generator of collective requests, so that one text serves two drivers:
  TorchCollective  one rank per process, the requests go to torch.distributed (all_gather_object, all_to_all_single);
  LocalCollective  W ranks in turn in ONE process (tests drive every rank on one GPU): run_local() steps the W generators.
Requests: ("gather", obj) -> [obj of every rank]; ("a2a", 1-D tensor grouped by destination, [elements for every destination],
[elements from every source]) -> 1-D tensor of what every source sent here, in rank order.

Shard planning (host, from the file alone): rank r searches a BGZF header from byte size*r/W; the guess is verified by walking the
block headers of rank r-1's range, which must land on it exactly; where it does not, rank r takes the landing point and the walk is
repeated, until nothing changes (rank 0 starts at byte 0, so every accepted boundary is a true one, by induction).  The record
boundaries follow the same rule one level down (mmlst_ingest_front_walk).
"""
from __future__ import annotations

import ctypes as C
import os
import struct
import zlib
from typing import List, Optional, Tuple

import numpy as np

from . import native

BROKEN = (1 << 64) - 1          # an exit / entry past a malformed record (and "guess" as the entry of a front walk)
_MAGIC = b"\x1f\x8b\x08"


class FrontInfo(C.Structure):
    _fields_ = [("n_blocks", C.c_uint64), ("n_own_blocks", C.c_uint64), ("own_inflated", C.c_uint64), ("inflated", C.c_uint64),
                ("compressed", C.c_uint64), ("block_error", C.c_uint64), ("entry", C.c_uint64), ("exit", C.c_uint64), ("need", C.c_uint64),
                ("n_rec", C.c_uint64), ("chain_error", C.c_uint64), ("repairs", C.c_uint32), ("world", C.c_int),
                ("send", C.c_void_p), ("send_len", C.c_void_p), ("send_idx", C.c_void_p), ("dest_records", C.c_void_p), ("dest_bytes", C.c_void_p),
                ("unsorted", C.c_int), ("first_key", C.c_uint64), ("last_key", C.c_uint64), ("seconds", C.c_double * 3)]


class BackArgs(C.Structure):
    _fields_ = [("ref_len", C.c_void_p), ("ref_names", C.c_char_p), ("header_text", C.c_char_p), ("n_ref", C.c_int32), ("unsorted", C.c_int)]


# ---------------------------------------------------------------------------------------------------------------------
# BGZF block headers on disk
# ---------------------------------------------------------------------------------------------------------------------
def block_check(fd: int, off: int, size: int) -> Tuple[int, Optional[str]]:
    """(total size, None) of the BGZF block whose header starts at byte `off` of the file, or (0, the refusal text of the whole-file
    ingest's block table for it): gzip magic and FEXTRA, a BC subfield, a size that fits header + trailer and the file, ISIZE <= 64 KiB."""
    h = os.pread(fd, 12, off) if size - off >= 18 else b""
    if len(h) < 12 or h[:3] != _MAGIC or not (h[3] & 4):
        return 0, "not a BGZF block at byte %d (plain gzip / truncated file?)" % off
    xlen = struct.unpack_from("<H", h, 10)[0]
    if size - off < 12 + xlen + 8:
        return 0, "truncated BGZF header at %d" % off
    x = os.pread(fd, xlen, off + 12)
    bsize, q = -1, 0
    while q + 4 <= xlen:
        slen = struct.unpack_from("<H", x, q + 2)[0]
        if x[q] == 66 and x[q + 1] == 67 and slen == 2:
            bsize = struct.unpack_from("<H", x, q + 4)[0]
        q += 4 + slen
    if bsize < 0:
        return 0, "BGZF block without BC subfield at %d" % off
    total = bsize + 1
    if total < 12 + xlen + 8 or size - off < total:
        return 0, "truncated BGZF block at %d" % off
    isize = block_isize(fd, off, total)
    if isize > 65536:
        return 0, "BGZF block with ISIZE %d > 64 KiB at %d" % (isize, off)
    return total, None


def block_size_at(fd: int, off: int, size: int) -> int:
    """Total size of a valid BGZF block starting at byte `off` (block_check), 0 when there is none."""
    return block_check(fd, off, size)[0]


def block_isize(fd: int, off: int, total: int) -> int:
    return struct.unpack("<I", os.pread(fd, 4, off + total - 4))[0]


def find_block(fd: int, size: int, start: int) -> int:
    """First offset >= start where a BGZF block header is followed by another one (or by the end of the file); `size` when there is
    none.  A guess: the caller verifies it against the walk of the previous range."""
    p = start
    while p < size:
        buf = os.pread(fd, min(1 << 20, size - p), p)
        i = 0
        while True:
            i = buf.find(_MAGIC, i)
            if i < 0:
                break
            t = block_size_at(fd, p + i, size)
            if t and (p + i + t == size or block_size_at(fd, p + i + t, size)):
                return p + i
            i += 1
        p += max(len(buf) - 2, 1)
    return size


def walk_blocks(fd: int, size: int, start: int, stop: int):
    """Walk the block headers from `start` to the first block boundary >= stop: that offset, or (offset, refusal text) of the first
    header on the way that is not valid."""
    p = start
    while p < stop and p < size:
        t, msg = block_check(fd, p, size)
        if not t:
            return (p, msg)
        p += t
    return p


def next_starts(starts: List[int], lands: list) -> List[int]:
    """One verification round: rank r starts where the walk of rank r-1's range landed (a rank whose predecessor's walk failed keeps
    its start until that walk is repaired)."""
    out = [0]
    for r in range(1, len(starts)):
        out.append(lands[r - 1] if isinstance(lands[r - 1], int) else starts[r])
    return out


def plan_refusal(starts: List[int], lands: list) -> Optional[str]:
    """The refusal of a failed walk whose range start is verified (rank 0, or the landing point of every earlier rank): its first
    invalid header is the file's first, the one the whole-file ingest names.  None while no such walk failed."""
    for r, land in enumerate(lands):
        if not isinstance(land, int):
            return land[1]
        if r + 1 < len(starts) and land != starts[r + 1]:
            return None
    return None


def read_header(path: str) -> Tuple[str, List[str], np.ndarray, int]:
    """BAM header from the first BGZF blocks (host inflate): text, reference names, lengths, and the inflated offset of the first record."""
    def bad(msg):
        return native.MmlstError(native.E_BAM, "mmlst_bam_ingest: " + msg)
    size = os.path.getsize(path)
    u = bytearray()
    fd = os.open(path, os.O_RDONLY)
    try:
        p = 0
        while True:
            if p >= size:
                raise bad("truncated BAM header" if u else "not a BAM file (empty)")
            t = block_size_at(fd, p, size)
            if not t:
                raise bad("not a BGZF block at byte %d (plain gzip / truncated file?)" % p)
            raw = os.pread(fd, t, p)
            xlen = struct.unpack_from("<H", raw, 10)[0]
            try:
                u += zlib.decompress(raw[12 + xlen:t - 8], -15)
            except zlib.error:
                raise bad("a BGZF block did not inflate to its ISIZE (corrupt file?)") from None
            p += t
            if len(u) < 12:
                continue
            if u[:4] != b"BAM\1":
                raise bad("not a BAM file (magic)")
            l_text = struct.unpack_from("<i", u, 4)[0]
            if l_text < 0:
                raise bad("bad l_text")
            q = 8 + l_text
            if q + 4 > len(u):
                continue
            n_ref = struct.unpack_from("<i", u, q)[0]
            if n_ref < 0:
                raise bad("bad n_ref")
            q += 4
            names, lens, done = [], [], True
            for _ in range(n_ref):
                if q + 4 > len(u):
                    done = False
                    break
                ln = struct.unpack_from("<i", u, q)[0]
                if ln < 1:
                    raise bad("truncated reference dictionary")
                if q + 4 + ln + 4 > len(u):
                    done = False
                    break
                names.append(bytes(u[q + 4:q + 4 + ln]).split(b"\0", 1)[0].decode("latin-1"))
                lens.append(struct.unpack_from("<I", u, q + 4 + ln)[0])
                q += 8 + ln
            if done:
                text = bytes(u[8:8 + l_text]).split(b"\0", 1)[0].decode("latin-1")
                return text, names, np.asarray(lens, dtype=np.uint32), q
    finally:
        os.close(fd)


# ---------------------------------------------------------------------------------------------------------------------
# collectives
# ---------------------------------------------------------------------------------------------------------------------
class TorchCollective:
    """The requests of one rank, served by torch.distributed (NCCL for the tensors)."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.group = group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)

    def run(self, gen):
        import torch
        import torch.distributed as dist
        reply = None
        while True:
            try:
                req = gen.send(reply)
            except StopIteration as e:
                return e.value
            if req[0] == "gather":
                out = [None] * self.world
                dist.all_gather_object(out, req[1], group=self.group)
                reply = out
            else:   # ("a2a", buffer grouped by destination, elements per destination, elements per source)
                send, scount, rcount = req[1], [int(x) for x in req[2]], [int(x) for x in req[3]]
                out = torch.empty(sum(rcount), dtype=send.dtype, device=send.device)
                dist.all_to_all_single(out, send, rcount, scount, group=self.group)
                torch.cuda.current_stream(send.device).synchronize()
                reply = out


def run_local(gens):
    """LocalCollective: step the W ranks' generators in turn (one process, one device); every request is a collective, so all ranks
    issue the same kind at the same step.  Returns every rank's result."""
    W = len(gens)
    replies = [None] * W
    results = [None] * W
    live = list(range(W))
    while live:
        reqs = {}
        for r in live:
            try:
                reqs[r] = gens[r].send(replies[r])
            except StopIteration as e:
                results[r] = e.value
        done = [r for r in live if r not in reqs]
        if done and reqs:
            raise RuntimeError("ranks %s finished while ranks %s wait in a collective" % (done, sorted(reqs)))
        live = sorted(reqs)
        if not live:
            break
        kinds = {reqs[r][0] for r in live}
        if len(kinds) != 1:
            raise RuntimeError("ranks issued different collectives: %s" % {r: reqs[r][0] for r in live})
        if kinds == {"gather"}:
            objs = [reqs[r][1] for r in range(W)]
            replies = [list(objs) for _ in range(W)]
        else:
            import torch
            parts = []
            for s_ in range(W):
                cnt = [int(x) for x in reqs[s_][2]]
                parts.append(torch.split(reqs[s_][1], cnt))
            replies = [torch.cat([parts[s_][d] for s_ in range(W)]) for d in range(W)]
    return results


# ---------------------------------------------------------------------------------------------------------------------
# the ingest of one rank
# ---------------------------------------------------------------------------------------------------------------------
class _Front:
    def __init__(self, h):
        self.h = h

    def __del__(self):
        try:
            if self.h:
                native.lib().mmlst_ingest_front_free(self.h)
                self.h = None
        except Exception:  # noqa: BLE001
            pass

    def info(self) -> FrontInfo:
        i = FrontInfo()
        native.check(native.lib().mmlst_ingest_front_info(self.h, C.byref(i)))
        return i


def _key(phase: int, word: int) -> int:
    return (phase << 56) | (word & ((1 << 56) - 1))


def _agree(errs):
    """The refusal every rank raises: the least (phase, index, code) of all ranks; a failure that is not a refusal (CUDA, memory)
    comes after every refusal, the lowest rank's first."""
    best = None
    for r, e in enumerate(errs):
        if e is None:
            continue
        k = (e[0], r) if e[1] is None else (e[0], -1)
        if best is None or k < best[0]:
            best = (k, e)
    if best is None:
        return
    e = best[1]
    if e[1] is None:
        native.check(native.lib().mmlst_ingest_refusal(e[0]))
    raise native.MmlstError(e[1], e[2])


_OTHER = 1 << 63   # sorts after every refusal key (phase <= 4)


def _local(fn):
    """Run fn(); a failure becomes this rank's entry for the next agreement instead of an exception (every rank must reach every
    collective, whatever went wrong on one of them)."""
    try:
        return fn(), None
    except native.MmlstError as e:
        return None, (_OTHER, e.code, str(e).split(": ", 1)[-1])
    except OSError as e:
        return None, (_OTHER, native.E_IO, "%s: %s" % (type(e).__name__, e))
    except MemoryError as e:
        return None, (_OTHER, native.E_NOMEM, "%s: %s" % (type(e).__name__, e))
    except Exception as e:  # noqa: BLE001 -- CUDA / allocator failures from torch among them
        code = native.E_NOMEM if "out of memory" in str(e) else native.E_CUDA
        return None, (_OTHER, code, "%s: %s" % (type(e).__name__, e))


def ingest_steps(path: str, device, rank: int, world: int, locus_of=None, minqual: int = 20, max_depth: Optional[int] = 8000,
                 presorted: bool = False, want_qhash: bool = True, sentinel_nodes: int = 1, check_crc: bool = False, halo_blocks: int = 1,
                 lenient_tags: bool = False):
    """Generator of rank `rank`'s ingest (module text); returns its streams.DeviceStreams."""
    import torch
    from . import bam
    dev = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
    lib = native.lib()
    size = os.path.getsize(path)
    header, err = _local(lambda: read_header(path))
    errs = yield ("gather", err)
    _agree(errs)
    text, names, ref_len, first_record = header
    n_ref = len(names)
    if locus_of is None:
        from . import api
        locus_of = api.AlleleIndex(names).locus_of
    owner = np.ascontiguousarray((np.asarray(locus_of, dtype=np.int64) % world).astype(np.int32))

    # ---- shard plan: contiguous block ranges, verified boundaries
    import time
    secs = {}
    t0 = time.perf_counter()
    fd = os.open(path, os.O_RDONLY)
    try:
        g, err = _local(lambda: 0 if rank == 0 else find_block(fd, size, size * rank // world))
        got = yield ("gather", (g, err))
        _agree([e for _g, e in got])
        starts = [x for x, _e in got]
        for _ in range(world + 1):
            stop = starts[rank + 1] if rank + 1 < world else size
            land, err = _local(lambda: walk_blocks(fd, size, starts[rank], stop) if starts[rank] < stop else starts[rank])
            got = yield ("gather", (land, err))
            _agree([e for _l, e in got])
            lands = [x for x, _e in got]
            msg = plan_refusal(starts, lands)
            if msg is not None:   # every rank saw the same walks: every rank raises the same refusal here
                raise native.MmlstError(native.E_BAM, "mmlst_bam_ingest: " + msg)
            new = next_starts(starts, lands)
            if new == starts:
                break
            starts = new
        else:
            raise native.MmlstError(native.E_BAM, "mmlst_bam_ingest: the BGZF block boundaries of the shards did not converge")
        c0 = starts[rank]
        c1 = max(c0, starts[rank + 1] if rank + 1 < world else size)
        secs["plan"] = time.perf_counter() - t0

        # ---- front half: own blocks + a halo of the next ones
        def halo_end(k):
            p, got = c1, 0
            while got < k and p < size:
                t = block_size_at(fd, p, size)
                if not t:
                    break
                p += t
                got += 1 if block_isize(fd, p - t, t) else 0
            return p

        stream = torch.cuda.current_stream(dev).cuda_stream

        def open_front(end):
            t1 = time.perf_counter()
            buf = torch.empty(max(end - c0, 1), dtype=torch.uint8, pin_memory=True)
            if end > c0:
                with open(path, "rb") as fh:
                    fh.seek(c0)
                    if fh.readinto(memoryview(buf.numpy())[:end - c0]) != end - c0:
                        raise native.MmlstError(native.E_IO, "short read on %s" % path)
            secs["read"] = secs.get("read", 0.0) + time.perf_counter() - t1
            h = C.c_void_p()
            with torch.cuda.device(dev):
                native.check(lib.mmlst_ingest_front_open(dev.index or 0, buf.data_ptr(), end - c0, c1 - c0, ref_len.ctypes.data, n_ref,
                                                          1 if check_crc else 0, stream, C.byref(h)))
            return _Front(h)

        k = halo_blocks
        end = 0
        t0 = time.perf_counter()

        def first_open():
            nonlocal end
            end = halo_end(k)
            return open_front(end)
        front, err = _local(first_open)
        fi = front.info() if front else None
        mine = (int(fi.own_inflated), int(fi.n_own_blocks)) if fi else (0, 0)
        if fi is not None and fi.block_error != BROKEN:
            err = (_key(0, int(fi.block_error)), None, None)   # block index made global below
        got = yield ("gather", (mine, err))
        ubase = [0] * world
        bbase = [0] * world
        for r in range(1, world):
            ubase[r] = ubase[r - 1] + got[r - 1][0][0]
            bbase[r] = bbase[r - 1] + got[r - 1][0][1]
        usize = ubase[-1] + got[-1][0][0]
        errs = []
        for r, (m, e) in enumerate(got):
            if e is not None and e[1] is None:   # buffer block index -> file block index
                w = e[0]
                e = (_key(0, (((w & ((1 << 56) - 1)) >> 8) + bbase[r]) << 8 | (w & 0xFF)), None, None)
            errs.append(e)
        _agree(errs)
        secs["inflate"] = time.perf_counter() - t0
        t0 = time.perf_counter()

        # ---- record entry: rank r starts where rank r-1's chain leaves its range; repeat until nothing changes
        def want_entry(r, exits):
            if r == 0 or first_record >= ubase[r]:
                return first_record
            return exits[r - 1]

        def walk(entry_global):
            """entry_global None = guess it; BROKEN = no record starts here (an earlier shard met a malformed record)"""
            nonlocal front, end, k
            while True:
                if entry_global is None:
                    e = BROKEN
                elif entry_global == BROKEN:
                    e = BROKEN - 1   # past the own range: the chain passes through
                else:
                    e = entry_global - ubase[rank]
                native.check(lib.mmlst_ingest_front_walk(front.h, e))
                fi = front.info()
                if fi.need and ubase[rank] + int(fi.need) <= usize and end < size:   # the last record ends past the halo: a longer one
                    k *= 2
                    end = halo_end(k)
                    front = None          # its buffers go back to the workspace before the longer buffer is inflated
                    front = open_front(end)
                    continue
                ent = BROKEN if fi.entry >= BROKEN - 1 else ubase[rank] + int(fi.entry)
                ex = BROKEN if fi.exit >= BROKEN - 1 else ubase[rank] + int(fi.exit)
                return ent, ex

        entry = first_record if (rank == 0 or first_record >= ubase[rank]) else None
        res, err = _local(lambda: walk(entry))
        for _ in range(world + 1):
            pairs = yield ("gather", (res, err))
            _agree([p[1] for p in pairs])
            exits = [p[0][1] for p in pairs]
            if all(pairs[r][0][0] == want_entry(r, exits) for r in range(world)):
                break
            w = want_entry(rank, exits)
            if res[0] != w:
                res, err = _local(lambda: walk(w))
        else:
            raise native.MmlstError(native.E_BAM, "mmlst_bam_ingest: record chain did not converge")
        secs["chain"] = time.perf_counter() - t0
        t0 = time.perf_counter()

        # ---- partition
        fi, err = _local(lambda: native.check(lib.mmlst_ingest_front_partition(front.h, owner.ctypes.data if n_ref else None, world)) or front.info())
        mine = None
        if fi is not None:
            mine = (int(fi.n_rec), _u64(fi.dest_records, world), _u64(fi.dest_bytes, world), int(fi.unsorted), int(fi.first_key),
                    int(fi.last_key), int(fi.chain_error))
        got = yield ("gather", (mine, err))
        _agree([e for _m, e in got])
    finally:
        os.close(fd)
    base = [0] * world
    for r in range(1, world):
        base[r] = base[r - 1] + got[r - 1][0][0]
    chain_errs = []
    for r, (m, _e) in enumerate(got):
        ce = m[6]
        chain_errs.append(None if ce == BROKEN else (_key(1, ((ce >> 8) + base[r]) << 8 | (ce & 0xFF)), None, None))
    # --presorted: out of order inside a shard, or between the last record of a shard and the first of the next one that has records
    unsorted = any(m[3] for m, _e in got)
    prev = None
    for m, _e in got:
        if m[0]:
            if prev is not None and m[4] < prev:
                unsorted = True
            prev = m[5]
    drec, dbytes = mine[1], mine[2]
    own_blocks, own_inflated = int(fi.n_own_blocks), int(fi.own_inflated)
    n, nbytes = int(fi.n_rec), int(sum(dbytes))
    secs["partition"] = time.perf_counter() - t0
    t0 = time.perf_counter()

    # ---- exchange: the partitioned buffers as they are, one all-to-all each
    recv_rec = [got[s_][0][1][rank] for s_ in range(world)]
    recv_bytes = [got[s_][0][2][rank] for s_ in range(world)]
    recs = yield ("a2a", _dev_tensor(fi.send, nbytes, torch.uint8, dev, front), dbytes, recv_bytes)
    rlen = yield ("a2a", _dev_tensor(fi.send_len, n, torch.int32, dev, front), drec, recv_rec)
    ridx = yield ("a2a", _dev_tensor(fi.send_idx, n, torch.int32, dev, front), drec, recv_rec)
    fi = None
    front = None   # the rank's compressed and inflated shard and its partition go back to the workspace before the back half
    nrec = int(rlen.numel())
    src_base = torch.repeat_interleave(torch.tensor(base, dtype=torch.int64, device=dev), torch.tensor(recv_rec, dtype=torch.int64, device=dev))
    gidx = (ridx.to(torch.int64) + src_base).to(torch.int32).contiguous()
    del ridx, src_base
    secs["exchange"] = time.perf_counter() - t0
    t0 = time.perf_counter()

    # ---- back half
    o = bam.UnpackOpts(int(minqual), int(max_depth or 0), int(sentinel_nodes), 0, 1, 1 if presorted else 0, 1 if want_qhash else 0, 0,
                       1 if lenient_tags else 0)
    names_b = "\n".join(names).encode("latin-1")
    text_b = text.encode("latin-1")
    a = BackArgs(ref_len.ctypes.data if n_ref else None, names_b, text_b, n_ref, 1 if unsorted else 0)
    h = C.c_void_p()
    ew = C.c_uint64(BROKEN)
    with torch.cuda.device(dev):
        rc = lib.mmlst_bam_ingest_back(dev.index or 0, recs.data_ptr() if nrec else None, rlen.data_ptr() if nrec else None,
                                       gidx.data_ptr() if nrec else None, nrec, C.byref(a), C.byref(o), torch.cuda.current_stream(dev).cuda_stream,
                                       C.byref(h), C.byref(ew))
    err = None
    if rc != 0:
        err = (int(ew.value), None, None) if ew.value != BROKEN else (_OTHER, rc, lib.mmlst_last_error().decode(errors="replace"))
    keep = bam._DevHandle(h) if rc == 0 else None
    del recs, rlen, gidx
    # a malformed record found by the front half: a refusal of phase 1 at its file index
    ce = chain_errs[rank]
    if ce is not None and (err is None or ce[0] < err[0]):
        err = ce
    errs = yield ("gather", err)
    _agree(errs)
    secs["back"] = time.perf_counter() - t0
    s = bam._dev_streams(keep, dev, want_qhash, lenient_tags)
    s.ingest_stats.update({"bgzf_blocks": own_blocks, "compressed_bytes": c1 - c0, "inflated_bytes": own_inflated})
    s.shard = {"rank": rank, "world": world, "records_parsed": n, "records_received": nrec, "file_index_base": base[rank],
               "bytes_sent": int(nbytes), "bytes_received": int(sum(recv_bytes)), "seconds": secs}
    return s


def _u64(addr, n):
    if not addr or n == 0:
        return [0] * n
    return [int(x) for x in (C.c_uint64 * n).from_address(addr)]


def _dev_tensor(addr, n, dtype, dev, keep):
    import torch
    from .bam import _DevArray
    if not addr or n == 0:
        return torch.zeros(0, dtype=dtype, device=dev)
    typestr = {torch.uint8: "|u1", torch.int32: "<i4"}[dtype]
    return torch.as_tensor(_DevArray(addr, n, typestr, keep), device=dev)
