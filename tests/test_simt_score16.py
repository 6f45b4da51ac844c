"""Form 7 of the run-length score kernel and the pack kernel of its compact stream, run WITHOUT a GPU on the host emulation of
tests/simt (the kernels' own text, one std::thread per lane): the pack output equals a numpy statement of the format, and the tables
of the compact kernel equal numpy -- across chunk and run boundaries, extreme scores, chunks whose AS span exceeds the 10-bit field,
minscore around a chunk's base (per-chunk fallback to the 3-byte arrays) and max_xm around the 4-bit XM field (per-call fallback)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from metamlst_b200 import packing
from test_simt_score import _np_score, _ptr, _streams

SIMT = os.path.join(ROOT, "tests", "simt")


@pytest.fixture(scope="module")
def simt16():
    so = os.path.join(SIMT, "libsimt_score16.so")
    srcs = [os.path.join(SIMT, "simt_score16.cpp"), os.path.join(SIMT, "simt_score.cpp"), os.path.join(SIMT, "simt_host_emul.h"),
            os.path.join(ROOT, "metamlst_b200", "csrc", "score_runs_kernels.cuh"), os.path.join(ROOT, "metamlst_b200", "csrc", "common.cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-I", SIMT,
                               "-I", os.path.join(ROOT, "metamlst_b200", "csrc"), "-o", so, srcs[0]])
    lib = C.CDLL(so)
    lib.simt_pack16.restype = C.c_int
    lib.simt_pack16.argtypes = [C.c_uint] + [C.c_void_p] * 3 + [C.c_uint64] + [C.c_void_p] * 2
    lib.simt_score16.restype = C.c_int
    lib.simt_score16.argtypes = ([C.c_uint] + [C.c_void_p] * 2 + [C.c_uint32] + [C.c_void_p] * 6 + [C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint32,
                                 C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 4)
    return lib


def np_pack16(as0, xm3, chunk_qlen):
    """The compact stream, stated in numpy: head = u16(top) | len(SEQ) << 16 per chunk, code = 0x8400 | x' << 11 | a per record."""
    n = as0.shape[0]
    nch = (n + 255) // 256
    pad = np.full(nch * 256, -32768, np.int64)
    pad[:n] = as0
    top = pad.reshape(nch, 256).max(1)
    base = np.repeat(top - 1023, 256)[:n]
    a = np.clip(as0.astype(np.int64) - base, 0, 1023)
    x = 15 - np.minimum(xm3.astype(np.int64), 15)
    code = (0x8400 | (x << 11) | a).astype(np.uint16)
    head = ((top & 0xFFFF) | (chunk_qlen.astype(np.int64) << 16)).astype(np.uint32)
    return code, head, top


def fallback_chunks(top, n, minscore):
    """Full chunks the compact kernel reduces from the 3-byte arrays: code 0 ("as0 <= top - 1023") could pass."""
    return int(np.count_nonzero(minscore <= top[: n // 256] - 1023))


_SIZES = [1, 255, 256, 257, 511, 513, 4096, 30011]


@pytest.mark.parametrize("n", _SIZES)
def test_compact_stream_form_matches_numpy(simt16, n):
    rng = np.random.default_rng(7000 + n)
    n_ref = 300
    nch = (n + 255) // 256
    for style in (("mixed", "long", "short", "config2") if n < 20000 else ("mixed", "config2")):
        tid = _streams(n, style, rng, n_ref)
        shift = np.repeat(rng.integers(-400, 400, nch), 256)[:n]  # chunks of different tops, so a minscore puts some chunks on each side
        as0 = np.clip(rng.integers(-50, 301, n) + shift, -32768, 32767).astype(np.int16)
        as0[rng.integers(0, n, max(1, n // 1000))] = 32767   # AS span of the chunk far beyond the 10-bit field
        as0[rng.integers(0, n, max(1, n // 1000))] = -32768
        as0[rng.integers(0, n, max(1, n // 1000))] = -32767
        xm3 = rng.integers(0, 17, n).astype(np.uint8)
        xm3[rng.integers(0, n, max(1, n // 500))] = 255
        qlen = np.repeat(rng.integers(30, 160, nch), 256)[:n].astype(np.uint16)
        allow = np.zeros(n_ref + 8, np.uint8)
        allow[:n_ref] = rng.random(n_ref) < 0.8
        soa = packing.SoaHost([], np.zeros(0, np.int32), tid, as0, xm3, qlen, None, np.zeros(0, packing.PREC_DTYPE), np.zeros(0, np.uint32), 0,
                              np.zeros(1, np.uint64)).build_runs(max_fraction=1.0)
        assert soa.run_tid is not None and soa.chunk_qlen is not None
        code = np.zeros(nch * 256, np.uint16)  # whole chunks, as the pipeline allocates it
        head = np.zeros(nch, np.uint32)
        assert simt16.simt_pack16(2, _ptr(as0), _ptr(xm3), _ptr(soa.chunk_qlen), n, _ptr(code), _ptr(head)) == 0
        want_code, want_head, top = np_pack16(as0, xm3, soa.chunk_qlen)
        assert np.array_equal(code[:n], want_code) and np.array_equal(head, want_head), (n, style)
        b0 = int(top[0]) - 1023  # base of chunk 0
        params = [(100, 5, 50), (-32768, 255, 0), (40000, 5, 50), (100, -1, 50), (100, 5, 70000), (100, 14, 50), (100, 15, 50), (-32768, 5, 0),
                  (b0 + 1, 5, 50), (b0, 5, 50), (b0 - 1, 5, 50), (max(min(b0 + 1000, 32767), -32768), 3, 50)]
        known = np.minimum(tid, n_ref)  # ids >= n_ref behave as a filtered allele
        allow_x = np.concatenate([allow[:n_ref], [0]])
        for grid in (1, 3):
            for k, (minscore, max_xm, min_len) in enumerate(params):
                if k and (grid != 1 or style != "mixed") and not (n < 20000 and k >= 8):
                    continue
                if n >= 20000 and grid != 1:
                    continue
                sum_as = np.zeros(n_ref, np.int64); n_hit = np.zeros(n_ref, np.uint32); first = np.full(n_ref, 0xFFFFFFFF, np.uint32)
                counters = np.zeros(2, np.uint64)
                rc = simt16.simt_score16(grid, _ptr(soa.run_tid), _ptr(soa.run_start), int(soa.run_tid.shape[0]), _ptr(soa.chunk_run),
                                         _ptr(soa.chunk_qlen), _ptr(as0), _ptr(xm3), _ptr(code), _ptr(head), n, 7, _ptr(allow), n_ref,
                                         minscore, max_xm, min_len, _ptr(sum_as), _ptr(n_hit), _ptr(first), _ptr(counters))
                assert rc == 0
                ws, wc, wf, wt, wi = _np_score(known, as0.astype(np.int64), xm3.astype(int), qlen.astype(int), np.arange(n) + 7,
                                               allow_x, n_ref + 1, minscore, max_xm, min_len)
                where = (n, style, grid, minscore, max_xm, min_len, fallback_chunks(top, n, minscore))
                assert np.array_equal(sum_as, ws[:n_ref]), where
                assert np.array_equal(n_hit, wc[:n_ref]) and np.array_equal(first, wf[:n_ref]), where
                assert (int(counters[0]), int(counters[1])) == (wt, wi), where


def test_minscore_around_a_chunk_base_splits_the_chunks():
    """The boundary parameter sets above really put chunks on both sides of the per-chunk rule."""
    rng = np.random.default_rng(5)
    n = 4096
    shift = np.repeat(rng.integers(-400, 400, n // 256), 256)
    as0 = np.clip(rng.integers(-50, 301, n) + shift, -32768, 32767).astype(np.int16)
    _code, _head, top = np_pack16(as0, np.zeros(n, np.uint8), np.zeros(n // 256, np.uint16))
    b0 = int(top[0]) - 1023
    assert fallback_chunks(top, n, b0) >= 1 and fallback_chunks(top, n, b0 - 1) >= 1
    assert fallback_chunks(top, n, b0 + 1) < n // 256 and fallback_chunks(top, n, b0) < n // 256
    assert fallback_chunks(top, n, 100) == 0
