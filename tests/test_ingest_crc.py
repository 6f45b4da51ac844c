"""CRC-32 of the BGZF blocks in the DEVICE ingest (`bam.ingest_bam(check_crc=True)`, csrc/ingest.cu crc_kernel,
csrc/bgzf_crc.cuh).  On the CPU: the kernel's arithmetic compiled by g++ (tests/ingest_emul/crc_emul.cpp) against zlib at every
length and start alignment, and the compiler's report for the kernel.  On the GPU: valid files give the host unpacker's streams
with the check on, and a file whose inflated bytes do not match a trailer CRC is refused by both routes with the same code and
block index -- including a bit flip inside a stored (level 0) DEFLATE block, which the decompression engine and the ISIZE check
cannot see."""
import ctypes as C
import glob
import os
import re
import shutil
import struct
import subprocess
import zlib

import numpy as np
import pytest

from conftest import GOLDEN, ROOT

CSRC = os.path.join(ROOT, "metamlst_b200", "csrc")
EMUL_SRC = os.path.join(ROOT, "tests", "ingest_emul", "crc_emul.cpp")
BAMS = sorted(glob.glob(os.path.join(GOLDEN, "*", "sample.bam")))


# ---- CPU: the kernel's arithmetic on the host ----------------------------------------------------------------------------
@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("crc_emul") / "libcrc_emul.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wall", "-Werror", "-shared", "-fPIC", "-I", CSRC, "-o", so, EMUL_SRC])
    lib = C.CDLL(so)
    for f in ("emul_frame_crc32", "emul_raw", "emul_zeros"):
        getattr(lib, f).restype = C.c_uint32
    lib.emul_frame_crc32.argtypes = [C.c_char_p, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32)]
    lib.emul_check.argtypes = [C.c_char_p, C.c_uint32, C.c_uint32, C.c_uint32]
    lib.emul_raw.argtypes = [C.c_char_p, C.c_uint32]
    lib.emul_zeros.argtypes = [C.c_uint32]
    return lib


def _check_block(lib, m: bytes, mis: int):
    n = len(m)
    z = C.c_uint32()
    got = lib.emul_frame_crc32(m, n, mis, C.byref(z))
    assert z.value == (-(mis + n)) % 16                          # the frame ends at the next 16-byte boundary
    assert got == zlib.crc32(m + bytes(z.value)), (n, mis)        # frame = block || 0^z
    want = zlib.crc32(m)
    assert lib.emul_check(m, n, mis, want) == 1, (n, mis)
    for bit in (0, n % 32, 31):
        assert lib.emul_check(m, n, mis, want ^ (1 << bit)) == 0, (n, mis, bit)


def test_every_length_to_1100_at_every_alignment(emul):
    rng = np.random.default_rng(11)
    data = rng.integers(0, 256, 1100, dtype=np.uint8).tobytes()
    for n in range(0, 1101):
        for mis in range(16):
            _check_block(emul, data[:n], mis)


@pytest.mark.parametrize("n", [4095, 4096, 4097, 65280, 65535, 65536])
@pytest.mark.parametrize("content", ["random", "zeros", "ones"])
def test_long_blocks_at_every_alignment(emul, n, content):
    m = {"random": np.random.default_rng(n).integers(0, 256, n, dtype=np.uint8).tobytes(), "zeros": bytes(n), "ones": b"\xff" * n}[content]
    for mis in range(16):
        _check_block(emul, m, mis)


@pytest.mark.parametrize("n", [0, 1, 3, 4, 255, 256, 1000, 65280, 65536])
def test_the_identities_the_kernel_rests_on(emul, n):
    m = np.random.default_rng(n + 1).integers(0, 256, n, dtype=np.uint8).tobytes()
    raw = emul.emul_raw(m, n)
    assert emul.emul_zeros(n) == zlib.crc32(bytes(n))
    assert raw == zlib.crc32(m) ^ zlib.crc32(bytes(n))           # trailer -> raw value
    for k in (1, 7, 16, 300):
        assert emul.emul_raw(bytes(k) + m, n + k) == raw          # leading zero bytes do not change a raw CRC


def test_crc_kernel_is_built_and_does_not_spill():
    obj, log = os.path.join(CSRC, "ingest.o"), os.path.join(CSRC, "ingest.ptxas.log")
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(obj) or not os.path.exists(log) or not os.path.exists(cuobjdump):
        pytest.skip("needs the objects of build() and cuobjdump")
    sass = subprocess.run([cuobjdump, "-sass", obj], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, timeout=300).stdout.decode(errors="replace")
    body = sass.split("crc_kernel", 1)
    assert len(body) == 2, "crc_kernel not in ingest.o"
    kernel = body[1].split("Function : ", 1)[0]
    assert "LDG.E.128" in kernel and "SHFL.DOWN" in kernel       # 16-byte loads of the inflated stream, shuffle combine
    hits = [m for m in re.finditer(r"Compiling entry function '(\S+)'.*?\n.*?\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads",
                                   open(log).read()) if "crc_kernel" in m.group(1)]
    assert hits, "no ptxas report for crc_kernel"
    for m in hits:
        assert (int(m.group(2)), int(m.group(3)), int(m.group(4))) == (0, 0, 0), m.group(1)


# ---- GPU ------------------------------------------------------------------------------------------------------------------
def _blocks(raw: bytes):
    """[(offset, total, isize)] of every BGZF block."""
    out, p = [], 0
    while p < len(raw):
        xlen = struct.unpack_from("<H", raw, p + 10)[0]
        q, bsize = p + 12, None
        while q + 4 <= p + 12 + xlen:
            if raw[q] == 66 and raw[q + 1] == 67 and struct.unpack_from("<H", raw, q + 2)[0] == 2:
                bsize = struct.unpack_from("<H", raw, q + 4)[0]
            q += 4 + struct.unpack_from("<H", raw, q + 2)[0]
        total = bsize + 1
        out.append((p, total, struct.unpack_from("<I", raw, p + total - 4)[0]))
        p += total
    return out


def _flip_trailer_crc(raw: bytes, k: int) -> bytes:
    """raw with the trailer CRC of non-empty block k flipped."""
    p, total, _ = [b for b in _blocks(raw) if b[2]][k]
    out = bytearray(raw)
    out[p + total - 8] ^= 0x01
    return bytes(out)


def _write(tmp_path, name, raw):
    p = str(tmp_path / name)
    open(p, "wb").write(raw)
    return p


def _expect_crc_refusal(fn, k):
    from metamlst_b200 import native
    with pytest.raises(native.MmlstError) as e:
        fn()
    assert e.value.code == native.E_BAM
    assert "CRC mismatch in BGZF block %d" % k in str(e.value), str(e.value)
    assert "CRC mismatch in BGZF block %d" % (k + 1) not in str(e.value)


def _stored_bam(db, n_reads, seed):
    import torch
    from metamlst_b200 import synth
    core = synth.gen_core(db, n_reads, 150, seed=seed, K=4, device="cuda:0")
    raw = synth.write_bam_fast(db, [core], order="name", align_records=True, level=0)
    del core
    torch.cuda.empty_cache()
    return raw.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("path", BAMS, ids=[os.path.basename(os.path.dirname(p)) for p in BAMS])
@pytest.mark.parametrize("presorted", [False, True])
def test_golden_bams_with_the_check(path, presorted):
    import json
    from metamlst_b200 import bam
    from test_ingest_gpu import same_streams
    man = json.load(open(os.path.join(GOLDEN, "manifest.json")))
    if presorted and "--presorted" not in man[os.path.basename(os.path.dirname(path))]["args"]:
        pytest.skip("file is not coordinate-sorted")
    same_streams(bam.ingest_bam(path, 0, presorted=presorted, check_crc=True), bam.unpack_bam(path, presorted=presorted, pinned=False))


@pytest.mark.gpu
@pytest.mark.parametrize("name,sizes", [("lowcov", (1,)), ("basic", (131,)), ("basic", (4095,)), ("basic", (65536,)),
                                        ("basic", (65536, 1, 4095, 131, 7)), ("lowcov", (1, 2, 3, 5, 8, 13, 21)), ("deep", (65535, 17, 60001, 4097))])
def test_every_block_length_and_alignment(tmp_path, name, sizes):
    from metamlst_b200 import bam
    from test_ingest_core import reblock
    from test_ingest_gpu import same_streams
    raw = reblock(open(os.path.join(GOLDEN, name, "sample.bam"), "rb").read(), sizes)
    p = _write(tmp_path, "cut.bam", raw)
    same_streams(bam.ingest_bam(p, 0, check_crc=True), bam.unpack_bam(p, pinned=False))


@pytest.mark.gpu
@pytest.mark.parametrize("level", [1, 0])
def test_synthetic_sample_of_a_million_records(tmp_path, level):
    import torch
    from metamlst_b200 import bam, synth
    from test_ingest_gpu import same_streams
    db = synth.make_db(("ecoli", "saureus"), alleles_per_locus=64, n_profiles=64, seed=5)
    core = synth.gen_core(db, 250_000, 150, seed=77, K=4, device="cuda:0")
    raw = synth.write_bam_fast(db, [core], order="name", align_records=True, level=level)
    del core
    torch.cuda.empty_cache()
    p = _write(tmp_path, "synth.bam", raw.tobytes())
    st = bam.ingest_bam(p, 0, check_crc=True)
    assert int(st.tid.shape[0]) == 1_000_000
    same_streams(st, bam.unpack_bam(p, pinned=False))


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["first", "middle", "last"])
def test_a_wrong_trailer_crc_is_refused_by_both_routes(tmp_path, where):
    from metamlst_b200 import bam
    from test_ingest_core import reblock
    from test_ingest_gpu import same_streams
    good = reblock(open(os.path.join(GOLDEN, "basic", "sample.bam"), "rb").read(), (4095, 977))
    nb = sum(1 for b in _blocks(good) if b[2])
    k = {"first": 0, "middle": nb // 2, "last": nb - 1}[where]
    p = _write(tmp_path, "bad.bam", _flip_trailer_crc(good, k))
    _expect_crc_refusal(lambda: bam.unpack_bam(p, pinned=False), k)
    _expect_crc_refusal(lambda: bam.ingest_bam(p, 0, check_crc=True), k)
    # without the check the device route still takes the file (the default is unchanged)
    same_streams(bam.ingest_bam(p, 0), bam.unpack_bam(_write(tmp_path, "good.bam", good), pinned=False))


@pytest.mark.gpu
def test_a_flipped_quality_in_a_stored_block(tmp_path):
    import torch
    from metamlst_b200 import bam, synth
    db = synth.make_db(("ecoli",), alleles_per_locus=16, n_profiles=16, seed=9)
    good = _stored_bam(db, 2000, seed=31)
    blocks = [b for b in _blocks(good) if b[2]]
    payloads = [good[p + 12 + struct.unpack_from("<H", good, p + 10)[0]:p + total - 8] for p, total, _ in blocks]
    u = b"".join(zlib.decompress(pl, -15) for pl in payloads)
    uoff = np.cumsum([0] + [b[2] for b in blocks])
    # first record after the header; then the middle quality of the first mapped all-M record with a quality >= 20 there
    r = 12 + struct.unpack_from("<i", u, 4)[0]
    for _ in range(struct.unpack_from("<i", u, r - 4)[0]):
        r += 8 + struct.unpack_from("<i", u, r)[0]
    while True:
        bs, _tid, _pos, l_name, _mq, _bin, n_cig, flag, l_seq = struct.unpack_from("<iiiBBHHHI", u, r)
        mid = r + 36 + l_name + 4 * n_cig + (l_seq + 1) // 2 + l_seq // 2
        if not flag & 4 and u[mid] >= 20 and all(struct.unpack_from("<I", u, r + 36 + l_name + 4 * c)[0] & 15 == 0 for c in range(n_cig)):
            break
        r += 4 + bs
    bi = int(np.searchsorted(uoff, mid, side="right")) - 1
    # offset of that byte in the file: walk block bi's stored DEFLATE blocks (1 header byte, LEN, NLEN, then LEN bytes verbatim)
    p, total, _ = blocks[bi]
    c, left = p + 12 + struct.unpack_from("<H", good, p + 10)[0], mid - int(uoff[bi])
    while True:
        assert good[c] & 0x06 == 0, "not a stored block"
        ln = struct.unpack_from("<H", good, c + 1)[0]
        if left < ln:
            break
        left -= ln
        c += 5 + ln
    assert good[c + 5 + left] == u[mid]
    bad = bytearray(good)
    bad[c + 5 + left] = 2   # quality 2: under minqual, the base leaves the pileup
    pg, pb = _write(tmp_path, "good.bam", good), _write(tmp_path, "bad.bam", bytes(bad))
    _expect_crc_refusal(lambda: bam.unpack_bam(pb, pinned=False), bi)
    _expect_crc_refusal(lambda: bam.ingest_bam(pb, 0, check_crc=True), bi)
    st_bad, st_good = bam.ingest_bam(pb, 0), bam.ingest_bam(pg, 0)
    assert st_bad.planes.shape == st_good.planes.shape
    assert not torch.equal(st_bad.planes, st_good.planes), "the flipped quality did not reach the plane rows"


@pytest.mark.gpu
def test_empty_blocks_with_a_nonzero_crc_field_are_accepted(tmp_path):
    from metamlst_b200 import bam
    from test_ingest_core import reblock
    from test_ingest_gpu import same_streams
    src = open(os.path.join(GOLDEN, "basic", "sample.bam"), "rb").read()
    good = reblock(src, (4095,))
    empty = b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + struct.pack("<H", 2 + 25) + b"\x03\x00" + struct.pack("<II", 0xDEADBEEF, 0)
    blocks = _blocks(good)
    cut = blocks[len(blocks) // 2][0]
    raw = good[:cut] + empty + empty + good[cut:] + empty
    p = _write(tmp_path, "empty.bam", raw)
    soa = bam.unpack_bam(p, pinned=False)
    same_streams(bam.ingest_bam(p, 0, check_crc=True), soa)
    same_streams(bam.ingest_bam(p, 0, check_crc=True), bam.unpack_bam(os.path.join(GOLDEN, "basic", "sample.bam"), pinned=False))


@pytest.mark.gpu
def test_the_check_on_a_second_stream_from_pinned_bytes(tmp_path):
    import torch
    from metamlst_b200 import bam
    from test_ingest_core import reblock
    from test_ingest_gpu import same_streams
    path = os.path.join(GOLDEN, "basic", "sample.bam")
    data = bam.read_pinned(path)
    assert data.is_pinned()
    s2 = torch.cuda.Stream()
    with torch.cuda.stream(s2):
        st = bam.ingest_bam(data, 0, check_crc=True)
    same_streams(st, bam.unpack_bam(path, pinned=False))
    raw = _flip_trailer_crc(reblock(open(path, "rb").read(), (8191,)), 5)
    bad = torch.from_numpy(np.frombuffer(raw, np.uint8).copy()).pin_memory()
    with torch.cuda.stream(s2):
        _expect_crc_refusal(lambda: bam.ingest_bam(bad, 0, check_crc=True), 5)
        st2 = bam.ingest_bam(data, 0, check_crc=True)   # the refusal leaves the stream usable
    torch.cuda.synchronize()
    assert torch.equal(st2.planes, st.planes)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(os.path.basename(os.path.dirname(p)) for p in BAMS))
def test_sample_typer_with_the_check_reproduces_reference_files(name, tmp_path):
    from metamlst_b200 import sample
    from test_sample_driver import _check_against_golden, _params
    d = os.path.join(GOLDEN, name)
    typer = sample.SampleTyper(os.path.join(d, "db.sqlite"), device=0, ingest="device", check_crc=True, **_params(name))
    res = typer.type_bam(os.path.join(d, "sample.bam"), str(tmp_path / "out"), want_stdout=True, timestamp=7)
    _check_against_golden(name, res, str(tmp_path / "out"))
    # a copy whose last non-empty block has a wrong trailer CRC is refused; the same typer without the check types it
    raw = open(os.path.join(d, "sample.bam"), "rb").read()
    k = sum(1 for b in _blocks(raw) if b[2]) - 1
    bad = _write(tmp_path, "sample.bam", _flip_trailer_crc(raw, k))
    _expect_crc_refusal(lambda: typer.type_bam(bad, str(tmp_path / "out2")), k)
    typer.check_crc = False
    typer.type_bam(bad, str(tmp_path / "out3"))
    typer.close()
