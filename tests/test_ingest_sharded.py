"""One BAM ingested by W ranks (bam.ingest_bam_sharded, metamlst_b200/shard.py, csrc/ingest.cu front / back half): every rank's
streams against the host unpacker's whole sample cut by owner (`DeviceStreams.from_soa(mode="loci")`), for W in {2, 3, 5} driven in
one process on one GPU (LocalCollective).  The CPU tests pin the shard plan: the block-header search, its verification, and the
C structs the driver reads."""
import ctypes as C
import glob
import json
import os
import struct

import numpy as np
import pytest

from conftest import GOLDEN
from metamlst_b200 import bam, native, packing, shard, streams
from oracle import bamio

BAMS = sorted(glob.glob(os.path.join(GOLDEN, "*", "sample.bam")))
IDS = [os.path.basename(os.path.dirname(p)) for p in BAMS]


def _reblocked(tmp_path, sizes, src=os.path.join(GOLDEN, "basic", "sample.bam"), name="cut.bam"):
    from test_ingest_core import reblock
    p = str(tmp_path / name)
    open(p, "wb").write(reblock(open(src, "rb").read(), sizes))
    return p


def _block_offsets(raw: bytes):
    out, p = [], 0
    while p < len(raw):
        out.append(p)
        p += struct.unpack_from("<H", raw, p + 16)[0] + 1
    return out


# ---------------------------------------------------------------------------------------------------------------------
# CPU: shard planning
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sizes", [(977,), (4096, 313, 65280), (131,)])
def test_block_search_finds_true_boundaries(tmp_path, sizes):
    p = _reblocked(tmp_path, sizes)
    raw = open(p, "rb").read()
    offs = _block_offsets(raw)
    fd = os.open(p, os.O_RDONLY)
    try:
        for g in range(0, len(raw), max(1, len(raw) // 97)):
            f = shard.find_block(fd, len(raw), g)
            assert f == next((o for o in offs if o >= g), len(raw))
        for a, b in zip(offs, offs[1:]):
            assert shard.block_size_at(fd, a, len(raw)) == b - a
            assert shard.walk_blocks(fd, len(raw), a, b) == b
            assert shard.walk_blocks(fd, len(raw), a, b - 1) == b
    finally:
        os.close(fd)


def test_block_search_false_positive_is_repaired(tmp_path):
    """A payload that contains a valid-looking BGZF header pair: the search takes it, the walk of the previous range does not land on
    it, and the next round moves the boundary to the landing point."""
    fake = b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + struct.pack("<H", 27) + b"\x03\x00" + struct.pack("<II", 0, 0)
    body = fake + fake + b"x" * 50
    import zlib
    co = zlib.compressobj(0, zlib.DEFLATED, -15)   # stored: the fake headers appear verbatim in the payload
    pl = co.compress(body) + co.flush()
    blk = b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + struct.pack("<H", len(pl) + 25) + pl + struct.pack("<II", zlib.crc32(body), len(body))
    raw = blk + blk + bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
    p = str(tmp_path / "fp.bin")
    open(p, "wb").write(raw)
    fd = os.open(p, os.O_RDONLY)
    try:
        g = shard.find_block(fd, len(raw), 1)
        assert 0 < g < len(blk)                         # inside the first block's payload
        starts = [0, g]
        lands = [shard.walk_blocks(fd, len(raw), 0, g), len(raw)]
        assert lands[0] == len(blk)
        starts = shard.next_starts(starts, lands)
        assert starts == [0, len(blk)]
        lands = [shard.walk_blocks(fd, len(raw), 0, starts[1]), len(raw)]
        assert shard.next_starts(starts, lands) == starts
    finally:
        os.close(fd)


def test_next_starts_fixed_point():
    # rank 2's predecessor walk failed: rank 2 keeps its start until rank 1 is repaired
    assert shard.next_starts([0, 10, 20], [12, (15, "bad"), 99]) == [0, 12, 20]
    assert shard.next_starts([0, 12, 20], [12, 25, 99]) == [0, 12, 25]


def test_plan_refusal_only_from_a_verified_range():
    # rank 1's start is not yet verified (rank 0 landed elsewhere): its failed walk may come from a false header
    assert shard.plan_refusal([0, 10, 20], [12, (15, "bad at 15"), 30]) is None
    assert shard.plan_refusal([0, 12, 20], [12, (15, "bad at 15"), 30]) == "bad at 15"
    assert shard.plan_refusal([0, 12], [(3, "bad at 3"), 30]) == "bad at 3"
    assert shard.plan_refusal([0, 12, 25], [12, 25, 40]) is None


def test_block_refusal_texts_are_the_block_tables(tmp_path):
    p = _reblocked(tmp_path, (977,))
    raw = bytearray(open(p, "rb").read())
    offs = _block_offsets(bytes(raw))
    b = offs[5]
    raw[b] = 0x1e
    q = str(tmp_path / "bad.bam")
    open(q, "wb").write(bytes(raw))
    fd = os.open(q, os.O_RDONLY)
    try:
        land = shard.walk_blocks(fd, len(raw), 0, len(raw))
        assert land == (b, "not a BGZF block at byte %d (plain gzip / truncated file?)" % b)
        q2 = str(tmp_path / "trunc.bam")
        open(q2, "wb").write(bytes(open(p, "rb").read())[:offs[7] + 30])
        fd2 = os.open(q2, os.O_RDONLY)
        assert shard.walk_blocks(fd2, offs[7] + 30, 0, offs[7] + 30) == (offs[7], "truncated BGZF block at %d" % offs[7])
        os.close(fd2)
    finally:
        os.close(fd)


@pytest.mark.parametrize("path", BAMS, ids=IDS)
def test_header_matches_the_oracle_reader(path):
    text, names, lens, first = shard.read_header(path)
    h, _recs = bamio.read_bam(path)
    assert names == list(h.ref_names) and list(lens) == list(h.ref_lens)
    import zlib
    from test_ingest_core import bgzf_blocks
    u = b"".join(zlib.decompress(pl, -15) for pl, _ in bgzf_blocks(open(path, "rb").read()))
    assert first == 12 + struct.unpack_from("<i", u, 4)[0] + sum(9 + len(n) for n in names)


def test_local_collective_routes_every_chunk():
    import torch

    def rank(r, W):
        got = yield ("gather", r * 10)
        assert got == [x * 10 for x in range(W)]
        # rank r sends d + 1 elements of value 100 * r + d to destination d
        counts = [d + 1 for d in range(W)]
        buf = torch.cat([torch.full((d + 1,), 100 * r + d) for d in range(W)])
        recv = yield ("a2a", buf, counts, [r + 1] * W)
        return recv.tolist()
    out = shard.run_local([rank(r, 3) for r in range(3)])
    assert out[1] == [1, 1, 101, 101, 201, 201]


def test_struct_layouts_match_the_header():
    assert C.sizeof(shard.FrontInfo) == 11 * 8 + 4 + 4 + 5 * 8 + 8 + 2 * 8 + 3 * 8
    assert shard.FrontInfo.send.offset == 96 and shard.FrontInfo.seconds.offset == 160
    assert C.sizeof(shard.BackArgs) == 32 and shard.BackArgs.unsorted.offset == 28


# ---------------------------------------------------------------------------------------------------------------------
# GPU: every rank against the host-unpacked sample cut by owner
# ---------------------------------------------------------------------------------------------------------------------
def _locus_of(soa):
    from metamlst_b200 import api
    return api.AlleleIndex(soa.ref_names).locus_of


def _check_ranks(path, W, **kw):
    import torch
    soa = bam.unpack_bam(path, pinned=False, minqual=kw.get("minqual", 20), max_depth=kw.get("max_depth", 8000),
                         presorted=kw.get("presorted", False))
    loc = _locus_of(soa)
    ranks = bam.ingest_bam_local(path, W, 0, **kw)
    h = lambda t: t.cpu().numpy()
    owner = np.asarray(loc, dtype=np.int64) % W
    dropped = 0
    for r, st in enumerate(ranks):
        want = streams.DeviceStreams.from_soa(soa, torch.device("cuda", 0), rank=r, world=W, mode="loci", locus_of=loc, want_qhash=True)
        assert list(st.ref_names) == list(soa.ref_names)
        assert np.array_equal(h(st.tid), h(want.tid)) and np.array_equal(h(st.as0), h(want.as0))
        assert np.array_equal(h(st.xm3), h(want.xm3)) and np.array_equal(h(st.qlen), h(want.qlen))
        assert np.array_equal(h(st.orig_idx), h(want.orig_idx))
        if soa.qhash is not None:
            assert np.array_equal(h(st.qhash), h(want.qhash))
        # pileup: every owned contig's records and rows equal the whole sample's (rows rebased), other contigs empty
        cs = st.contig_start.astype(np.int64)
        assert cs.shape[0] == len(soa.ref_names) + 1
        recs = h(st.p_recs).reshape(-1).view(packing.PREC_DTYPE)
        planes = h(st.planes).view(np.uint32)
        for t in range(len(soa.ref_names)):
            a, b = int(cs[t]), int(cs[t + 1])
            wa, wb = int(soa.contig_start[t]), int(soa.contig_start[t + 1])
            if owner[t] != r:
                assert a == b, (r, t)
                continue
            assert b - a == wb - wa, (r, t)
            if b == a:
                continue
            mine, ref = recs[a:b], soa.p_recs[wa:wb]
            for f in ("pos", "reflen", "as_named", "xm_named", "nw"):
                assert np.array_equal(mine[f], ref[f]), (r, t, f)
            for j in range(b - a):
                rw = int(ref["nw"][j]) * 3
                assert np.array_equal(planes[int(mine["row_off"][j]):int(mine["row_off"][j]) + rw],
                                      soa.planes[int(ref["row_off"][j]):int(ref["row_off"][j]) + rw]), (r, t, j)
        dropped += st.n_dropped
    assert dropped == soa.n_dropped_by_cap
    return ranks


@pytest.mark.gpu
@pytest.mark.parametrize("W", [2, 3, 5])
@pytest.mark.parametrize("path", BAMS, ids=IDS)
def test_golden_bams_sharded(path, W):
    man = json.load(open(os.path.join(GOLDEN, "manifest.json")))
    presorted = "--presorted" in man[os.path.basename(os.path.dirname(path))]["args"]
    _check_ranks(path, W, presorted=presorted)


@pytest.mark.gpu
@pytest.mark.parametrize("W", [2, 3, 5])
@pytest.mark.parametrize("sizes", [(977,), (4096, 313, 65280), (131,), (60000, 7)])
def test_shard_boundaries_inside_records(tmp_path, sizes, W):
    _check_ranks(_reblocked(tmp_path, sizes), W)


@pytest.mark.gpu
def test_more_ranks_than_blocks(tmp_path):
    p = _reblocked(tmp_path, (1 << 16,))
    nblk = len(_block_offsets(open(p, "rb").read()))
    ranks = _check_ranks(p, nblk + 3)
    assert sum(int(s.tid.shape[0]) == 0 for s in ranks) >= 3


@pytest.mark.gpu
@pytest.mark.parametrize("W", [2, 3, 5])
@pytest.mark.parametrize("seed,max_depth,minqual", [(1, 8000, 20), (3, 40, 20), (2, 7, 30)])
def test_ragged_reads_and_the_depth_cap(tmp_path, seed, max_depth, minqual, W):
    from test_ragged_reads import _ragged_bam
    p, _recs, _rng = _ragged_bam(tmp_path, seed)
    _check_ranks(p, W, minqual=minqual, max_depth=max_depth)


def _mutated(tmp_path, mutate, sizes=(977,)):
    h, recs = bamio.read_bam(os.path.join(GOLDEN, "basic", "sample.bam"))
    recs = mutate(list(recs))
    p = str(tmp_path / "m.bam")
    bamio.write_bam(p, h.ref_names, h.ref_lens, recs)
    return _reblocked(tmp_path, sizes, src=p, name="m_cut.bam")


def _mutate_at(i, case):
    def mutate(recs):
        r = recs[i]
        if case == "paired":
            recs[i] = r._replace(flag=r.flag | 0x3)
        elif case == "noref":
            recs[i] = r._replace(tid=-1, pos=-1)
        elif case == "no_aux3":
            recs[i] = r._replace(aux=r.aux[:3])
        elif case == "as_range":
            recs[i] = r._replace(aux=(bamio.int_aux("AS", 70000),) + tuple(r.aux[1:]))
        return recs
    return mutate


@pytest.mark.gpu
@pytest.mark.parametrize("case,code", [("paired", -6), ("noref", -4), ("no_aux3", -4), ("as_range", -7)])
def test_refusals_in_a_later_shard(tmp_path, case, code):
    h, recs = bamio.read_bam(os.path.join(GOLDEN, "basic", "sample.bam"))
    k = (3 * len(recs)) // 4
    p = _mutated(tmp_path, _mutate_at(k, case))
    with pytest.raises(native.MmlstError) as e_host:
        bam.unpack_bam(p, pinned=False)
    with pytest.raises(native.MmlstError) as e_dev:
        bam.ingest_bam_local(p, 3, 0)
    assert e_host.value.code == e_dev.value.code == code
    assert "record %d:" % k in str(e_dev.value)
    with pytest.raises(native.MmlstError) as e_one:
        bam.ingest_bam(p, 0)
    assert str(e_one.value) == str(e_dev.value)


@pytest.mark.gpu
def test_first_refusal_in_file_order_wins(tmp_path):
    h, recs = bamio.read_bam(os.path.join(GOLDEN, "basic", "sample.bam"))
    a, b = len(recs) // 3, (4 * len(recs)) // 5

    def mutate(rs):
        rs = _mutate_at(b, "paired")(rs)
        return _mutate_at(a, "as_range")(rs)
    p = _mutated(tmp_path, mutate)
    with pytest.raises(native.MmlstError) as e_one:
        bam.ingest_bam(p, 0)
    for W in (2, 3, 5):
        with pytest.raises(native.MmlstError) as e_dev:
            bam.ingest_bam_local(p, W, 0)
        assert str(e_dev.value) == str(e_one.value) and "record %d:" % a in str(e_dev.value)


@pytest.mark.gpu
def test_bad_crc_in_a_later_shard(tmp_path):
    p = _reblocked(tmp_path, (977,))
    raw = bytearray(open(p, "rb").read())
    offs = _block_offsets(bytes(raw))
    bad = (2 * len(offs)) // 3                                   # inside shard 2 of 3
    end = offs[bad + 1]
    raw[end - 8] ^= 0x5A                                         # the block's CRC32 trailer
    open(p, "wb").write(bytes(raw))
    with pytest.raises(native.MmlstError) as e_one:
        bam.ingest_bam(p, 0, check_crc=True)
    with pytest.raises(native.MmlstError) as e_dev:
        bam.ingest_bam_local(p, 3, 0, check_crc=True)
    assert str(e_dev.value) == str(e_one.value) and "CRC mismatch in BGZF block %d" % bad in str(e_dev.value)
    assert len(bam.ingest_bam_local(p, 3, 0)) == 3                # without check_crc the file is typed


@pytest.mark.gpu
def test_presorted_refusal_is_agreed(tmp_path):
    src = os.path.join(GOLDEN, "presorted", "sample.bam")
    h, recs = bamio.read_bam(src)
    recs = list(recs)
    k = len(recs) // 2
    moved = recs[k:] + recs[:k]   # two sorted halves: out of order only where they meet
    q = str(tmp_path / "u.bam")
    bamio.write_bam(q, h.ref_names, h.ref_lens, moved)
    with pytest.raises(native.MmlstError) as e_one:
        bam.ingest_bam(q, 0, presorted=True)
    assert e_one.value.code == native.E_UNSORTED
    for W in (2, 3):
        with pytest.raises(native.MmlstError) as e_dev:
            bam.ingest_bam_local(q, W, 0, presorted=True)
        assert e_dev.value.code == native.E_UNSORTED and str(e_dev.value) == str(e_one.value)


def _stored_bgzf(u: bytes, B: int) -> bytes:
    """BGZF of the inflated stream u in blocks of B bytes, DEFLATE level 0 (stored): a block's compressed size depends on its length only,
    so the shard plan of the file is the same whatever the order of the records."""
    import zlib
    out = []
    for p in range(0, len(u), B):
        chunk = u[p:p + B]
        co = zlib.compressobj(0, zlib.DEFLATED, -15)
        pl = co.compress(chunk) + co.flush()
        out.append(b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + struct.pack("<H", len(pl) + 25) + pl + struct.pack("<II", zlib.crc32(chunk), len(chunk)))
    out.append(bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000"))
    return b"".join(out)


def _inflated(path):
    import zlib
    from test_ingest_core import bgzf_blocks
    return b"".join(zlib.decompress(pl, -15) for pl, _ in bgzf_blocks(open(path, "rb").read()))


def _plan_inflated_starts(path, W):
    """Inflated offset of every rank's first block under the shard plan (the planner's own functions, run to their fixed point)."""
    raw = open(path, "rb").read()
    fd = os.open(path, os.O_RDONLY)
    try:
        starts = [0] + [shard.find_block(fd, len(raw), len(raw) * r // W) for r in range(1, W)]
        while True:
            lands = [shard.walk_blocks(fd, len(raw), starts[r], starts[r + 1] if r + 1 < W else len(raw)) for r in range(W)]
            new = shard.next_starts(starts, lands)
            if new == starts:
                break
            starts = new
        ustart, u, p = [], 0, 0
        for r in range(W):
            while p < starts[r]:
                t = shard.block_size_at(fd, p, len(raw))
                u += shard.block_isize(fd, p, t)
                p += t
            ustart.append(u)
        return ustart
    finally:
        os.close(fd)


@pytest.mark.gpu
@pytest.mark.parametrize("W", [2, 3])
def test_presorted_file_unsorted_only_across_a_shard_boundary(tmp_path, W):
    """The two sorted halves of the presorted sample, swapped, cut so that the pair out of order is the last record of rank W-1's
    predecessor and the first record of rank W-1: no shard sees it inside its own records."""
    src = os.path.join(GOLDEN, "presorted", "sample.bam")
    h, recs = bamio.read_bam(src)
    recs = list(recs)
    B = 4000
    tmp = str(tmp_path / "tmp.bam")
    bamio.write_bam(tmp, h.ref_names, h.ref_lens, recs)
    u0 = _inflated(tmp)
    _text, _names, _lens, first = shard.read_header(tmp)
    offs, q = [], first                                  # record offsets of the sorted stream
    while q < len(u0):
        offs.append(q)
        q += struct.unpack_from("<i", u0, q)[0] + 4
    lens_b = [b - a for a, b in zip(offs, offs[1:] + [len(u0)])]
    p_stored = str(tmp_path / "layout.bam")
    open(p_stored, "wb").write(_stored_bgzf(u0, B))
    U = _plan_inflated_starts(p_stored, W)[W - 1]     # the same for every order of the records
    key = lambda r: (r.tid, r.pos)
    chosen = None
    for k in range(1, len(recs)):
        J = first + sum(lens_b[k:])                     # inflated offset of recs[k] once recs[k:] + recs[:k]
        if J - lens_b[-1] < U <= J and key(recs[k]) < key(recs[-1]):
            chosen = k
            break
    assert chosen is not None
    moved = recs[chosen:] + recs[:chosen]
    q = str(tmp_path / "u.bam")
    bamio.write_bam(tmp, h.ref_names, h.ref_lens, moved)
    u1 = _inflated(tmp)
    open(q, "wb").write(_stored_bgzf(u1, B))
    assert _plan_inflated_starts(q, W)[W - 1] == U
    J = first + sum(lens_b[chosen:])
    assert struct.unpack_from("<i", u1, J - lens_b[-1])[0] + 4 == lens_b[-1]   # the pair: the record before J starts before U, J at or after it
    assert J - lens_b[-1] < U <= J
    with pytest.raises(native.MmlstError) as e_one:
        bam.ingest_bam(q, 0, presorted=True)
    assert e_one.value.code == native.E_UNSORTED
    with pytest.raises(native.MmlstError) as e_dev:
        bam.ingest_bam_local(q, W, 0, presorted=True)
    assert e_dev.value.code == native.E_UNSORTED and str(e_dev.value) == str(e_one.value)
    assert len(bam.ingest_bam_local(q, W, 0)) == W    # without --presorted the file is typed


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["middle", "last"])
def test_corrupt_block_header_refused_as_the_whole_file(tmp_path, where):
    p = _reblocked(tmp_path, (977,))
    raw = bytearray(open(p, "rb").read())
    offs = _block_offsets(bytes(raw))
    b = offs[len(offs) // 2] if where == "middle" else offs[-3]
    raw[b + 1] = 0x00
    q = str(tmp_path / "bad.bam")
    open(q, "wb").write(bytes(raw))
    with pytest.raises(native.MmlstError) as e_one:
        bam.ingest_bam(q, 0)
    for W in (2, 3):
        with pytest.raises(native.MmlstError) as e_dev:
            bam.ingest_bam_local(q, W, 0)
        assert str(e_dev.value) == str(e_one.value) and "byte %d" % b in str(e_dev.value)


@pytest.mark.gpu
def test_two_ranks_type_every_golden_sample(tmp_path):
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    root = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
    env = dict(os.environ, PYTHONPATH=root)
    import socket
    with socket.socket() as so:   # a port no other job holds
        so.bind(("127.0.0.1", 0))
        port = so.getsockname()[1]
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", str(port), os.path.join(root, "tests", "run_sharded_ingest.py"), str(tmp_path / "out")], env=env,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=900)
    assert p.returncode == 0, p.stdout.decode()[-3000:]
    assert "SHARDED-INGEST-OK" in p.stdout.decode()
