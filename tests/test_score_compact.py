"""Form 7 of the run-length score kernel on the GPU: the compact 2 B / record stream (mmlst_score_pack16_dev) scored by
mmlst_score_runs16_dev gives the tables of form 6 and of numpy, on raw streams and through DevicePipeline; the pipeline derives the
stream again for every sample it is bound to and keeps the 5-byte form for streams without uniform chunks.  Needs a B200."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN
from metamlst_b200 import api, native, packing, pipeline
from test_simt_score import _np_score, _streams
from test_simt_score16 import fallback_chunks, np_pack16

pytestmark = pytest.mark.gpu


@pytest.fixture
def form():
    """Sets the library's score form for one test and restores it."""
    lib = native.lib()
    prev = lib.mmlst_set_score_variant(-1)
    yield lambda v: lib.mmlst_set_score_variant(v)
    lib.mmlst_set_score_variant(prev)


def _raw_score(variant, soa, d, code, head, allow, n_ref, minscore, max_xm, min_len, idx_base=7):
    import torch
    lib = native.lib()
    lib.mmlst_set_score_variant(variant)
    n = int(soa.as0.shape[0])
    sum_as = torch.zeros(n_ref, dtype=torch.int64, device="cuda"); n_hit = torch.zeros(n_ref, dtype=torch.int32, device="cuda")
    first = torch.full((n_ref,), -1, dtype=torch.int32, device="cuda"); cnt = torch.zeros(2, dtype=torch.int64, device="cuda")
    native.check(lib.mmlst_score_runs16_dev(native.ptr(d["run_tid"]), native.ptr(d["run_start"]), int(soa.run_tid.shape[0]), native.ptr(d["chunk_run"]),
                                            native.ptr(d["chunk_qlen"]), native.ptr(d["as0"]), native.ptr(d["xm3"]), native.ptr(code), native.ptr(head), n,
                                            idx_base, native.ptr(allow), n_ref, minscore, max_xm, min_len, native.ptr(sum_as), native.ptr(n_hit),
                                            native.ptr(first), native.ptr(cnt), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return (sum_as.cpu().numpy(), n_hit.cpu().numpy().view(np.uint32), first.cpu().numpy().view(np.uint32), tuple(int(x) for x in cnt.cpu().numpy()))


def _pack(d, n):
    import torch
    nch = (n + 255) // 256
    code = torch.empty(nch * 256, dtype=torch.int16, device="cuda")
    head = torch.empty(nch, dtype=torch.int32, device="cuda")
    native.check(native.lib().mmlst_score_pack16_dev(native.ptr(d["as0"]), native.ptr(d["xm3"]), native.ptr(d["chunk_qlen"]), n, native.ptr(code),
                                                     native.ptr(head), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return code, head


@pytest.mark.parametrize("n", [1, 255, 256, 257, 511, 513, 4096, 30011, 1_000_003])
def test_form7_equals_form6_and_numpy_on_raw_streams(form, n):
    import torch
    rng = np.random.default_rng(8000 + n)
    n_ref = 300
    nch = (n + 255) // 256
    for style in ("mixed", "long", "short", "config2"):
        tid = _streams(n, style, rng, n_ref)
        shift = np.repeat(rng.integers(-400, 400, nch), 256)[:n]
        as0 = np.clip(rng.integers(-50, 301, n) + shift, -32768, 32767).astype(np.int16)
        as0[rng.integers(0, n, max(1, n // 1000))] = 32767
        as0[rng.integers(0, n, max(1, n // 1000))] = -32768
        xm3 = rng.integers(0, 17, n).astype(np.uint8)
        xm3[rng.integers(0, n, max(1, n // 500))] = 255
        qlen = np.repeat(rng.integers(30, 160, nch), 256)[:n].astype(np.uint16)
        allow = np.zeros(n_ref + 8, np.uint8)
        allow[:n_ref] = rng.random(n_ref) < 0.8
        soa = packing.SoaHost([], np.zeros(0, np.int32), tid, as0, xm3, qlen, None, np.zeros(0, packing.PREC_DTYPE), np.zeros(0, np.uint32), 0,
                              np.zeros(1, np.uint64)).build_runs(max_fraction=1.0)
        up = lambda a: torch.from_numpy(np.ascontiguousarray(a).view({1: np.uint8, 2: np.int16, 4: np.int32}[a.dtype.itemsize])).cuda()
        d = {k: up(getattr(soa, k)) for k in ("run_tid", "run_start", "chunk_run", "chunk_qlen", "as0", "xm3")}
        code, head = _pack(d, n)
        want_code, want_head, top = np_pack16(as0, xm3, soa.chunk_qlen)
        assert np.array_equal(code.cpu().numpy().view(np.uint16)[:n], want_code) and np.array_equal(head.cpu().numpy().view(np.uint32), want_head)
        allow_d = up(allow)
        known = np.minimum(tid, n_ref)
        allow_x = np.concatenate([allow[:n_ref], [0]])
        b0 = int(top[0]) - 1023
        for minscore, max_xm, min_len in ((100, 5, 50), (80, 5, 50), (-32768, 255, 0), (40000, 5, 50), (100, -1, 50), (100, 5, 70000),
                                          (100, 14, 50), (100, 15, 50), (b0 + 1, 5, 50), (b0, 5, 50), (b0 - 1, 5, 50)):
            ws, wc, wf, wt, wi = _np_score(known, as0.astype(np.int64), xm3.astype(int), qlen.astype(int), np.arange(n) + 7, allow_x, n_ref + 1,
                                           minscore, max_xm, min_len)
            want = (ws[:n_ref], wc[:n_ref], wf[:n_ref], (wt, wi))
            for v in (7, 6):
                got = _raw_score(v, soa, d, code, head, allow_d, n_ref, minscore, max_xm, min_len)
                where = (n, style, v, minscore, max_xm, min_len, fallback_chunks(top, n, minscore))
                assert all(np.array_equal(a, b) for a, b in zip(got[:3], want[:3])) and got[3] == want[3], where


def _synthetic(n_reads, seed, db=None):
    from metamlst_b200 import devpack, synth
    db = db or synth.make_db(("ecoli", "saureus"), alleles_per_locus=16, n_profiles=20, seed=seed)
    core = synth.gen_core(db, n_reads, read_len=150, seed=seed, K=4, sub_err=0.005, device="cuda:0")   # configs[1]: L = 150, K = 4
    return db, devpack.pack_cores(db, [core], 20, 8000)


def test_pipeline_form7_equals_form6_step_graph_and_rebind(form):
    db, st = _synthetic(200_000, 41)
    _db, st2 = _synthetic(150_000, 42, db)  # a second sample of the same cohort
    assert st.chunk_qlen is not None and getattr(st, "orig_idx", None) is None
    index = api.AlleleIndex(db.ref_names())
    pipe = pipeline.DevicePipeline(st, index, db.row_seq, minscore=80, max_xM=5, min_read_len=50, penalty=100)
    assert pipe.code16 is not None and pipe.compact_fallback_chunks() == 0
    soa = st.to_host(pinned=False)
    n_ref = len(index.ref_names)
    tid = np.repeat(soa.run_tid, np.diff(soa.run_start.astype(np.int64)))
    ws, wc, wf, wt, wi = _np_score(tid, soa.as0.astype(np.int64), soa.xm3.astype(int), np.repeat(soa.chunk_qlen, 256)[: soa.n_rec].astype(int),
                                   np.arange(soa.n_rec), index.allow_mask(None), n_ref, 80, 5, 50)
    res = {}
    for v in (7, 6):
        form(v)
        pipe.want_tables = True
        r = pipe.step()
        tabs = [x.copy() for x in pipe.tables()]
        assert np.array_equal(tabs[0], ws) and np.array_equal(tabs[1], wc) and np.array_equal(tabs[2], wf), v
        assert (pipe.total_reads, pipe.ignored_reads) == (wt, wi)
        pipe.want_tables = False
        pipe.capture()
        assert pipe.step_graph() == r
        res[v] = (r, pipe.total_reads, pipe.ignored_reads)
    assert res[7] == res[6]
    # another sample bound to the same pipeline: its own compact stream, and the same results as a pipeline built for it
    form(7)
    pipe.rebind(st2)
    assert pipe.code16.shape[0] == (int(st2.as0.shape[0]) + 255) // 256 * 256
    got = pipe.step()
    assert got == pipeline.DevicePipeline(st2, index, db.row_seq, minscore=80, max_xM=5, min_read_len=50, penalty=100).step()
    form(6)
    assert pipe.step() == got
    form(7)
    # max_xM outside the 4-bit XM field: the 3-byte call, same results
    wide = pipeline.DevicePipeline(st2, index, db.row_seq, minscore=80, max_xM=15, min_read_len=50, penalty=100)
    r15 = wide.step()
    form(6)
    assert wide.step() == r15


def test_stream_without_uniform_chunks_keeps_the_five_byte_form(form):
    db, st = _synthetic(20_000, 43)
    index = api.AlleleIndex(db.ref_names())
    want = pipeline.DevicePipeline(st, index, db.row_seq).step()
    st.chunk_qlen = None  # what a sample of mixed read lengths in one chunk looks like to the pipeline
    pipe = pipeline.DevicePipeline(st, index, db.row_seq)
    assert not pipe.use_qc and pipe.code16 is None and pipe.compact_fallback_chunks() == -1
    form(7)
    assert pipe.step() == want


def test_fallback_counts_on_the_golden_bams(form):
    """Chunks form 7 reduces from the 3-byte arrays at minscore 80, on every golden BAM that gets a compact stream (coordinate-sorted
    files: the name-ordered ones carry a file-order index and keep the 3-byte form); each one is scored equal to form 6."""
    from metamlst_b200 import bam
    man = json.load(open(os.path.join(GOLDEN, "manifest.json")))
    seen = {}
    for name in sorted(man):
        path = os.path.join(GOLDEN, name, "sample.bam")
        if not os.path.exists(path):
            continue
        try:
            st = bam.ingest_bam(path, 0, presorted=man[name].get("order") == "coord")
        except native.MmlstError:
            continue  # a scenario whose BAM the reference refuses too
        index = api.AlleleIndex(list(st.ref_names))
        pipe = pipeline.DevicePipeline(st, index, lambda t: "A" * int(st.ref_lens[t]), minscore=80, max_xM=5, min_read_len=50)
        seen[name] = (int(st.as0.shape[0]), pipe.compact_fallback_chunks())
        if pipe.code16 is None:
            continue
        form(7)
        pipe.want_tables = True
        r7 = (pipe.step(), [x.copy() for x in pipe.tables()], pipe.total_reads, pipe.ignored_reads)
        form(6)
        r6 = (pipe.step(), [x.copy() for x in pipe.tables()], pipe.total_reads, pipe.ignored_reads)
        assert r7[0] == r6[0] and all(np.array_equal(a, b) for a, b in zip(r7[1], r6[1])) and r7[2:] == r6[2:], name
    print("golden BAMs (records, chunks reduced from the 3-byte form at minscore 80; -1 = no compact stream):", seen)
    assert any(c >= 0 for _n, c in seen.values())
