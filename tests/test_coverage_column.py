"""Coverage column of stage 1 (H7, csrc/coverage.cu) against the reference's `sequenceBank`.

metamlst.py:127 stores `sequenceBank[species_gene][QNAME] = len(SEQ)` and :228 sums the dict, so for every (locus, QNAME) the
LAST passing record in FILE order decides the length.  The cases here give the records of one name different lengths (SEQ `*`,
which counts as length 1, trimmed reads, a second record of the name on another allele of the locus later in the file), so that
"last in file order" differs from "last in the coordinate-sorted stream" and from "any record of the name".

CPU: the plain dict restatement used below equals the oracle's `stage1` bank on every rewritten BAM; a numpy restatement of the
sharded coverage (insert -> exchange of table entries -> merge -> sum) adds up to the whole sample for every shard mode and world.
GPU (`-m gpu`): the kernel's edges through `mmlst_coverage_dev`, every upload form of `mmlst_coverage`, `DevicePipeline` on
host-unpacked, device-ingested and sliced streams, shards driven step by step on one device, the driver's stdout, and two real
ranks (skipped below two GPUs).
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT
from helpers import small_case, table_to_records
from metamlst_b200 import api, bam, native, packing, streams
from oracle import bamio, mlst_oracle as orc

gpu = pytest.mark.gpu
GOLDEN_RATIO = 0x9E3779B97F4A7C15   # csrc/coverage.cu: key.hi ^= (locus + 1) * this (one name set per locus)


@pytest.fixture(scope="module")
def ctx():
    c = native.Context(0)
    yield c
    c.close()


# ------------------------------------------------------------------------------------------------ references
def _bank_sums(bank):
    return {k: sum(v.values()) for k, v in bank.items()}


def _dict_bank(h, recs, minscore, max_xm, min_len, species_filter=None):
    """metamlst.py:115,127,228 restated on the records in file order: last[(locus, QNAME)] = len(SEQ), then the sum per locus."""
    keep = species_filter.split(",") if species_filter else None
    last = {}
    for r in recs:
        sp, g, _a = h.ref_names[r.tid].split("_")
        if keep is not None and sp not in keep:
            continue
        ql = len(r.seq) or 1   # SEQ '*' prints as one character
        if int(r.aux[0][2]) >= minscore and ql >= min_len and int(r.aux[3][2]) <= max_xm:
            last[(sp + "_" + g, r.qname)] = ql
    out = {}
    for (locus, _q), v in last.items():
        out[locus] = out.get(locus, 0) + v
    return out


def _dict_coverage(tid, as0, xm3, qlen, idx, key, allow, locus_of, minscore, max_xm, min_len):
    """The same on raw arrays: passing records in ascending file index overwrite last[(locus, key)]; {locus: sum}."""
    n_ref = allow.shape[0]
    t = tid.astype(np.int64)
    inside = t < n_ref
    ok = np.zeros(tid.shape[0], bool)
    ok[inside] = (allow[t[inside]] != 0) & (as0[inside].astype(np.int64) >= minscore) & (qlen[inside].astype(np.int64) >= min_len) & \
        (xm3[inside].astype(np.int64) <= max_xm)
    last = {}
    for i in np.nonzero(ok)[0][np.argsort(np.asarray(idx)[ok], kind="stable")].tolist():
        last[(int(locus_of[t[i]]), int(key[i, 0]), int(key[i, 1]))] = int(qlen[i])
    out = {}
    for (l, _a, _b), v in last.items():
        out[l] = out.get(l, 0) + v
    return out


# ------------------------------------------------------------------------------------------------ mixed-length BAMs
def _trim(r, t):
    """Drop the last t bases: SEQ, QUAL and the last CIGAR op together, so that the CIGAR query length stays l_seq."""
    op, ln = r.cigar[-1]
    if op not in (0, 1, 4, 7, 8) or ln < 2:
        return r
    t = min(t, ln - 1, len(r.seq) - 1)
    if t <= 0:
        return r
    return r._replace(cigar=r.cigar[:-1] + ((op, ln - t),), seq=r.seq[:-t], qual=r.qual[:-t] if r.qual else b"")


def _star(r):
    return r._replace(seq="", qual=b"")   # SEQ '*': l_seq == 0 is accepted with any CIGAR


def _rewrite(h, recs, seed, L):
    """Every record kept, about 10 % printed with SEQ '*', 35 % trimmed (some below 50 bases), and for 12 % of the records a
    second record of the same QNAME on another allele of the same locus with another length, a few records later in the file."""
    rng = np.random.default_rng(seed)
    alleles = {}
    for t, name in enumerate(h.ref_names):
        alleles.setdefault(name.rsplit("_", 1)[0], []).append(t)
    out, pending = [], []
    for orig in recs:
        u = rng.random()
        r = _star(orig) if u < 0.10 else (_trim(orig, int(rng.integers(1, L - 5))) if u < 0.45 else orig)
        out.append(r)
        others = [t for t in alleles[h.ref_names[r.tid].rsplit("_", 1)[0]] if t != r.tid]
        if others and rng.random() < 0.12:
            alt = int(rng.choice(others))
            m = _trim(orig, int(rng.integers(1, L // 2)))
            m = m._replace(tid=alt, pos=max(0, min(r.pos, int(h.ref_lens[alt]) - m.ref_len())))
            pending.append((len(out) + int(rng.integers(1, 40)), m))
        while pending and pending[0][0] <= len(out):
            out.append(pending.pop(0)[1])
    out.extend(m for _d, m in pending)
    return out


def _write(path, h, recs, coord):
    if coord:
        recs = sorted(recs, key=lambda r: (r.tid, r.pos))
    bamio.write_bam(path, h.ref_names, h.ref_lens, recs, sort_order="coordinate" if coord else "unknown")
    return recs


# name -> (golden directory or None, seed); every case is written name-ordered ("unsorted") and coordinate-sorted
SOURCES = {"basic": ("basic", 11), "two_org": ("two_org", 12), "synth": (None, 13)}
MIN_LENS = (0, 1, 50)


@pytest.fixture(scope="module")
def bams(tmp_path_factory):
    return _make_bams(tmp_path_factory.mktemp("cov_bams"))


def _make_bams(d):
    """{(name, order): (path, header, records in file order, db path or None)}, order in ('name', 'coord')."""
    out = {}
    for name, (gold, seed) in SOURCES.items():
        if gold:
            h, recs = bamio.read_bam(os.path.join(GOLDEN, gold, "sample.bam"))
            db = os.path.join(GOLDEN, gold, "db.sqlite")
        else:
            _db, tab = small_case(seed=seed, n_reads=1500, L=100, K=4, orgs=("ecoli", "saureus"), apl=5)
            h, recs = table_to_records(tab)
            db = None
        mixed = _rewrite(h, recs, seed, 100)
        for order in ("name", "coord"):
            p = str(d / ("%s_%s.bam" % (name, order)))
            written = _write(p, h, mixed, order == "coord")
            h2, back = bamio.read_bam(p)
            assert back == written
            out[(name, order)] = (p, h2, back, db)
    return out


CASES = [(n, o) for n in SOURCES for o in ("name", "coord")]


def _unpack(path, order):
    return bam.unpack_bam(path, presorted=(order == "coord"), want_qhash=True)


# ================================================================================================ CPU
@pytest.mark.parametrize("case", CASES, ids=lambda c: "%s-%s" % c)
def test_dict_restatement_is_the_oracle_sequence_bank(bams, case):
    """The reference every GPU test below compares with: pinned to the oracle's stage 1 on every rewritten BAM."""
    _p, h, recs, _db = bams[case]
    lens = [len(r.seq) or 1 for r in recs]
    assert 1 in lens and min(l for l in lens if l > 1) < 50 and max(lens) == 100   # SEQ '*', short and full reads are all there
    names = {}
    for r in recs:
        names.setdefault((h.ref_names[r.tid].rsplit("_", 1)[0], r.qname), set()).add(len(r.seq) or 1)
    assert sum(len(v) > 1 for v in names.values()) > 20   # many (locus, QNAME) with records of different lengths
    for min_len in MIN_LENS:
        for filt in (None, "saureus"):
            _cel, bank, _t, _i = orc.stage1(h, recs, 80, 5, min_len, filt, 100)
            assert _dict_bank(h, recs, 80, 5, min_len, filt) == _bank_sums(bank), (min_len, filt)
    # the order matters on these files: taking the last record in (tid, pos) order instead gives other sums
    if case[1] == "name":
        srt = sorted(recs, key=lambda r: (r.tid, r.pos))
        assert _dict_bank(h, srt, 80, 5, 0) != _dict_bank(h, recs, 80, 5, 0)


def _np_shard_coverage(shards, allow, locus_of, minscore, max_xm, min_len, merge):
    """numpy / dict restatement of the sharded coverage: per shard insert (max value word per key), every shard merges the
    others' entries into the keys it holds (if `merge`), then every shard's sum pass; returns the sum over shards {locus: bases}."""
    tables, recs = [], []
    for st in shards:
        tid = st.tid.numpy().view(np.uint32).astype(np.int64)
        n = tid.shape[0]
        idx = st.orig_idx.numpy().view(np.uint32).astype(np.int64) if st.orig_idx is not None else st.idx_base + np.arange(n)
        qlen = st.qlen.numpy().view(np.uint16).astype(np.int64)
        ok = (tid < allow.shape[0])
        ok[ok] = (allow[tid[ok]] != 0)
        ok &= (st.as0.numpy().astype(np.int64) >= minscore) & (qlen >= min_len) & (st.xm3.numpy().astype(np.int64) <= max_xm)
        qh = st.qhash.numpy().view(np.uint64)
        rows = [((int(locus_of[tid[i]]), int(qh[i, 0]), int(qh[i, 1])), ((int(idx[i]) + 1) << 16) | int(qlen[i]), int(qlen[i]))
                for i in np.nonzero(ok)[0].tolist()]
        t = {}
        for k, v, _q in rows:
            t[k] = max(t.get(k, 0), v)
        tables.append(t)
        recs.append(rows)
    if merge:
        entries = [dict(t) for t in tables]   # what every shard exports before anyone merges
        for r, t in enumerate(tables):
            for s, e in enumerate(entries):
                if s != r:
                    for k in t:
                        if k in e:
                            t[k] = max(t[k], e[k])
    out = {}
    for t, rows in zip(tables, recs):
        for k, v, q in rows:
            if t[k] == v:
                out[k[0]] = out.get(k[0], 0) + q
    return out


@pytest.mark.parametrize("world", [2, 3, 4])
@pytest.mark.parametrize("mode", ["ranges", "loci"])
def test_sharded_coverage_restatement_adds_up(bams, mode, world):
    """The exchange the device pipeline runs on record shards, restated: merged shards add up to the whole sample, for both
    shard modes; without the merge, "ranges" shards count names whose records straddle a cut once per rank."""
    path, h, recs, _db = bams[("synth", "name")]
    soa = _unpack(path, "name")
    index = api.AlleleIndex(soa.ref_names)
    allow = index.allow_mask(None)
    for min_len in (1, 50):
        want = _dict_bank(h, recs, 80, 5, min_len)
        shards = [streams.DeviceStreams.from_soa(soa, "cpu", rank=r, world=world, mode=mode, locus_of=index.locus_of, want_qhash=True)
                  for r in range(world)]
        got = _np_shard_coverage(shards, allow, index.locus_of, 80, 5, min_len, merge=True)
        assert {"%s_%s" % index.locus_names[l]: v for l, v in got.items()} == want
        naive = _np_shard_coverage(shards, allow, index.locus_of, 80, 5, min_len, merge=False)
        if mode == "loci":
            assert naive == got   # whole loci per rank: nothing to merge
        else:
            assert naive != got and all(naive[l] >= got[l] for l in got)


# ================================================================================================ GPU: kernel edges
def _kernel_coverage(tid, as0, xm3, qlen, oidx, key, allow, locus_of, n_loci, minscore=100, max_xm=5, min_len=0, idx_base=0,
                     slots=None):
    """mmlst_coverage_dev on torch tensors -> ({locus: bases}, table_slots)."""
    lib = native.lib()
    d = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a).view(dt)).cuda()
    n = int(tid.shape[0])
    slots = int(slots or lib.mmlst_coverage_table_slots(n))
    t = [d(tid.astype(np.uint32), np.int32), d(as0.astype(np.int16), np.int16), d(xm3.astype(np.uint8), np.uint8),
         d(qlen.astype(np.uint16), np.int16), None if oidx is None else d(oidx.astype(np.uint32), np.int32),
         d(key.astype(np.uint64), np.int64), d(allow.astype(np.uint8), np.uint8), d(locus_of.astype(np.uint32), np.int32)]
    table = torch.zeros(slots * 3, dtype=torch.int64, device="cuda")
    cov = torch.zeros(n_loci + 1, dtype=torch.int64, device="cuda")
    native.check(lib.mmlst_coverage_dev(native.ptr(t[0]), native.ptr(t[1]), native.ptr(t[2]), native.ptr(t[3]), native.ptr(t[4]),
                                        native.ptr(t[5]), n, idx_base, native.ptr(t[6]), native.ptr(t[7]), int(allow.shape[0]), minscore,
                                        max_xm, min_len, native.ptr(table), slots, native.ptr(cov), torch.cuda.current_stream().cuda_stream))
    c = cov.cpu().numpy()
    assert c[n_loci] == 0
    return {l: int(v) for l, v in enumerate(c[:n_loci]) if v}


def _check(tid, as0, xm3, qlen, oidx, key, allow, locus_of, n_loci, idx_base=0, slots=None, **prm):
    idx = (idx_base + np.arange(tid.shape[0])) if oidx is None else oidx.astype(np.int64)
    p = dict(minscore=100, max_xm=5, min_len=0)
    p.update(prm)
    want = _dict_coverage(tid, as0, xm3, qlen, idx, key, allow, locus_of, p["minscore"], p["max_xm"], p["min_len"])
    got = _kernel_coverage(tid, as0, xm3, qlen, oidx, key, allow, locus_of, n_loci, p["minscore"], p["max_xm"], p["min_len"], idx_base, slots)
    assert got == want
    return want


def _records(rng, n, n_ref, lens=(1, 200)):
    tid = rng.integers(0, n_ref, n).astype(np.uint32)
    as0 = rng.integers(100, 200, n).astype(np.int16)
    xm3 = rng.integers(0, 6, n).astype(np.uint8)
    qlen = rng.integers(lens[0], lens[1], n).astype(np.uint16)
    return tid, as0, xm3, qlen


@gpu
@pytest.mark.parametrize("slots", [2, 4, 1024])
def test_full_table_with_probe_chains_that_wrap(slots):
    """Exactly table_slots distinct (locus, name) keys in a table of that many slots: every slot ends up taken and the probe
    chains run past the last slot back to slot 0, in the insert and in the sum pass."""
    for seed in range(4):
        rng = np.random.default_rng(1000 * slots + seed)
        n_loci = 3
        locus_of = np.arange(2 * n_loci, dtype=np.uint32) // 2     # two alleles per locus
        allow = np.ones(2 * n_loci, np.uint8)
        pairs = set()
        while len(pairs) < slots:
            pairs.add((int(rng.integers(0, n_loci)), int(rng.integers(1, 1 << 62)), int(rng.integers(0, 1 << 62))))
        pairs = sorted(pairs)
        per = rng.integers(1, 4, slots)                               # 1..3 records per key, of different lengths
        owner = np.repeat(np.arange(slots), per)
        n = owner.shape[0]
        tid = np.array([2 * pairs[k][0] + int(rng.integers(0, 2)) for k in owner], np.uint32)
        key = np.array([[pairs[k][1], pairs[k][2]] for k in owner], np.uint64)
        as0 = rng.integers(100, 200, n).astype(np.int16)
        xm3 = np.zeros(n, np.uint8)
        qlen = rng.integers(1, 300, n).astype(np.uint16)
        oidx = rng.permutation(n).astype(np.uint32)
        _check(tid, as0, xm3, qlen, oidx, key, allow, locus_of, n_loci, slots=slots)
        _check(tid, as0, xm3, qlen, None, key, allow, locus_of, n_loci, slots=slots)


@gpu
def test_empty_slot_sentinel_and_one_name_on_many_loci():
    """Hashes {0,0} and {0,1}; on every 7th locus the hash that the locus fold turns into the empty-slot key {0,0}, which the
    kernel remaps.  The remap once sent that name to {1,0} on every locus, so these names of different loci merged into one
    slot and all but one locus lost their length.  Also one name present on every locus."""
    rng = np.random.default_rng(7)
    n_loci = 200
    locus_of = np.arange(2 * n_loci, dtype=np.uint32) // 2
    allow = np.ones(2 * n_loci, np.uint8)
    rows = []
    for l in range(0, n_loci, 7):
        fold = ((l + 1) * GOLDEN_RATIO) & 0xFFFFFFFFFFFFFFFF
        for k in ((0, 0), (0, 1), (0, fold), (5, 5)):
            for _ in range(3):
                rows.append((2 * l + int(rng.integers(0, 2)), k))
    # one name on every locus, 1..4 records each
    for l in range(n_loci):
        for _ in range(int(rng.integers(1, 5))):
            rows.append((2 * l + int(rng.integers(0, 2)), (0xDEADBEEF, 0x1234)))
    order = rng.permutation(len(rows))
    rows = [rows[i] for i in order]
    n = len(rows)
    tid = np.array([r[0] for r in rows], np.uint32)
    key = np.array([r[1] for r in rows], np.uint64)
    as0 = rng.integers(100, 200, n).astype(np.int16)
    xm3 = np.zeros(n, np.uint8)
    qlen = rng.integers(1, 500, n).astype(np.uint16)
    for oidx in (None, rng.permutation(n).astype(np.uint32)):
        want = _check(tid, as0, xm3, qlen, oidx, key, allow, locus_of, n_loci)
        assert len(want) == n_loci


@gpu
def test_grid_stride_rounds_in_both_passes():
    """More records than one grid covers (16 CTAs of 256 threads per SM): every thread runs several rounds of both passes."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = max(2_500_000, 3 * 16 * sms * 256 + 77)
    rng = np.random.default_rng(3)
    n_ref, n_loci = 120, 40
    locus_of = (np.arange(n_ref) // 3).astype(np.uint32)
    allow = (rng.random(n_ref) < 0.9).astype(np.uint8)
    tid, as0, xm3, qlen = _records(rng, n, n_ref)
    as0 = rng.integers(80, 200, n).astype(np.int16)
    key = np.zeros((n, 2), np.uint64)
    key[:, 0] = rng.integers(1, n // 4, n).astype(np.uint64)
    key[:, 1] = rng.integers(0, 3, n).astype(np.uint64)
    _check(tid, as0, xm3, qlen, rng.permutation(n).astype(np.uint32), key, allow, locus_of, n_loci, min_len=50)
    _check(np.sort(tid), as0, xm3, qlen, None, key, allow, locus_of, n_loci, idx_base=12345)


@gpu
def test_warp_aggregated_add_on_one_locus_many_loci_and_mixed_lanes():
    """Warps of 32 records all on one locus (one REDUX + one atomic), on 32 loci, with failing lanes, and a partial last warp."""
    rng = np.random.default_rng(11)
    n_loci = 64
    locus_of = np.arange(n_loci, dtype=np.uint32)
    allow = np.ones(n_loci, np.uint8)
    allow[5] = 0
    blocks = []
    for w in range(600):
        kind = w % 4
        if kind == 0:
            t = np.full(32, w % n_loci)
        elif kind == 1:
            t = rng.permutation(n_loci)[:32]
        elif kind == 2:
            t = np.full(32, (w * 7) % n_loci)
            t[rng.random(32) < 0.5] = rng.integers(0, n_loci)
        else:
            t = rng.integers(0, 2, 32) + (w % (n_loci - 1))
        blocks.append(t)
    tid = np.concatenate(blocks)[: 600 * 32 - 13].astype(np.uint32)  # the last warp has lanes past n_rec
    n = tid.shape[0]
    as0 = rng.integers(100, 200, n).astype(np.int16)
    as0[rng.random(n) < 0.2] = 10          # failing lanes
    xm3 = rng.integers(0, 7, n).astype(np.uint8)
    qlen = rng.integers(1, 65536, n).astype(np.uint16)
    key = np.zeros((n, 2), np.uint64)
    key[:, 0] = np.arange(n) // 2           # names shared by neighbouring lanes
    key[:, 1] = 9
    _check(tid, as0, xm3, qlen, None, key, allow, locus_of, n_loci)
    key[:, 0] = np.arange(n)                # every record its own name: every passing lane adds
    _check(tid, as0, xm3, qlen, rng.permutation(n).astype(np.uint32), key, allow, locus_of, n_loci)


@gpu
def test_file_index_at_the_top_of_the_value_word_and_extreme_lengths():
    """(index + 1) << 16 | len(SEQ) with orig_idx up to 0xFFFFFFFF and idx_base past 2^32 up to the last index the 48 bits
    hold; len(SEQ) of 1 and 65535; an idx_base past the last one is refused."""
    rng = np.random.default_rng(13)
    n, n_loci = 20000, 10
    locus_of = np.arange(n_loci, dtype=np.uint32)
    allow = np.ones(n_loci, np.uint8)
    tid = rng.integers(0, n_loci, n).astype(np.uint32)
    as0 = rng.integers(100, 200, n).astype(np.int16)
    xm3 = np.zeros(n, np.uint8)
    qlen = rng.choice(np.array([1, 2, 65534, 65535], np.uint16), n)
    key = np.zeros((n, 2), np.uint64)
    key[:, 0] = rng.integers(1, 3000, n).astype(np.uint64)
    top = (0xFFFFFFFF - rng.permutation(n)).astype(np.uint32)       # distinct file indices up to 0xFFFFFFFF
    _check(tid, as0, xm3, qlen, top, key, allow, locus_of, n_loci)
    for base in (1 << 32, (1 << 32) + 12345, (1 << 48) - 1 - n):
        _check(np.sort(tid), as0, xm3, qlen, None, key, allow, locus_of, n_loci, idx_base=base)
    with pytest.raises(native.MmlstError) as e:
        _kernel_coverage(tid, as0, xm3, qlen, None, key, allow, locus_of, n_loci, idx_base=(1 << 48) - n)
    assert e.value.code == native.E_RANGE


@gpu
def test_records_outside_the_index_or_filtered_out():
    """tid >= n_ref (the kernel reads nothing for them), alleles with allow = 0, and every threshold at its edge."""
    rng = np.random.default_rng(17)
    n, n_ref = 30000, 50
    locus_of = (np.arange(n_ref) // 5).astype(np.uint32)
    allow = (rng.random(n_ref) < 0.6).astype(np.uint8)
    tid = rng.integers(0, n_ref, n).astype(np.uint32)
    tid[rng.random(n) < 0.1] = rng.choice(np.array([n_ref, n_ref + 1, 0xFFFFFFFF], np.uint32))
    as0 = rng.integers(98, 103, n).astype(np.int16)
    xm3 = rng.integers(3, 7, n).astype(np.uint8)
    qlen = rng.integers(48, 53, n).astype(np.uint16)
    key = np.zeros((n, 2), np.uint64)
    key[:, 0] = rng.integers(1, 2000, n).astype(np.uint64)
    for oidx in (None, rng.permutation(n).astype(np.uint32)):
        _check(tid, as0, xm3, qlen, oidx, key, allow, locus_of, 10, minscore=100, max_xm=5, min_len=50)
    none = _kernel_coverage(tid, as0, xm3, qlen, None, key, np.zeros(n_ref, np.uint8), locus_of, 10)
    assert none == {}


# ================================================================================================ GPU: the C-ABI's upload forms
@gpu
@pytest.mark.parametrize("n", [1, 255, 256, 257, "past-grid-cap"])
def test_expand_chunk_qlen_gives_back_qlen(n):
    """mmlst_expand_chunk_qlen_dev at chunk edges and past the grid cap (16 CTAs of 256 threads per SM: grid-stride rounds)."""
    if n == "past-grid-cap":
        n = 2 * 16 * torch.cuda.get_device_properties(0).multi_processor_count * 256 + 99
    rng = np.random.default_rng(n)
    chunk = rng.integers(0, 65536, (n + 255) // 256).astype(np.uint16)
    want = np.repeat(chunk, 256)[:n]
    cq = torch.from_numpy(chunk.view(np.int16)).cuda()
    out = torch.full((n + 3,), -1, dtype=torch.int16, device="cuda")
    native.check(native.lib().mmlst_expand_chunk_qlen_dev(native.ptr(cq), n, native.ptr(out), torch.cuda.current_stream().cuda_stream))
    got = out.cpu().numpy().view(np.uint16)
    assert np.array_equal(got[:n], want) and np.all(got[n:] == 0xFFFF)   # nothing written past n_rec


def _forms(soa):
    """(form, SoaHost) for every upload form of the score stream mmlst_coverage takes."""
    yield "tid", _clone(soa, runs=False)
    yield "runs", _clone(soa, runs=True)
    qc = _clone(soa, runs=False)
    rng = np.random.default_rng(5)
    qc.qlen = np.repeat(rng.integers(1, 160, (qc.n_rec + 255) // 256), 256)[: qc.n_rec].astype(np.uint16)   # one len(SEQ) per chunk
    qc.build_runs(max_fraction=1.0)
    assert qc.chunk_qlen is not None
    yield "qc", qc
    for cover, coeff in ((1.0, 3), (0.5, 0), (0.5, 2)):
        z = _clone(soa, runs=True)
        z.deflate(block=4096, cover=cover, as_xm_coeff=coeff)
        assert z.z_bytes is not None
        yield "deflate-%g-%d" % (cover, coeff), z


def _clone(soa, runs):
    c = packing.SoaHost(soa.ref_names, soa.ref_lens, soa.tid.copy(), soa.as0.copy(), soa.xm3.copy(), soa.qlen.copy(),
                        None if soa.orig_idx is None else soa.orig_idx.copy(), soa.p_recs, soa.planes, soa.max_row_words, soa.contig_start)
    c.qhash = soa.qhash.copy()
    if runs:
        c.build_runs(max_fraction=1.0)
        c.chunk_qlen = None
        assert c.run_tid is not None
    return c


@gpu
@pytest.mark.parametrize("case", CASES, ids=lambda c: "%s-%s" % c)
def test_every_upload_form_of_the_c_abi(ctx, bams, case):
    """api.coverage_sums after an explicit-tid, a run-length (expanded by mmlst_expand_runs_dev), a per-chunk len(SEQ) (expanded
    by mmlst_expand_chunk_qlen_dev) and a DEFLATE upload, fresh and resident right after api.score_soa on the same context."""
    path, h, recs, _db = bams[case]
    base = _unpack(path, case[1])
    assert (base.orig_idx is None) == (case[1] == "coord")
    index = api.AlleleIndex(base.ref_names)
    allow = index.allow_mask(None)
    for form, soa in _forms(base):
        for min_len in MIN_LENS:
            if form == "qc":
                idx = np.arange(soa.n_rec) if soa.orig_idx is None else soa.orig_idx.astype(np.int64)
                want = {"%s_%s" % index.locus_names[l]: v for l, v in _dict_coverage(soa.tid, soa.as0, soa.xm3, soa.qlen, idx, soa.qhash, allow,
                                                                                     index.locus_of, 80, 5, min_len).items()}
            else:
                want = _bank_sums(orc.stage1(h, recs, 80, 5, min_len, None, 100)[1])
            assert api.coverage_sums(ctx, soa, index, 80, 5, min_len) == want, (form, min_len)
            api.score_soa(ctx, soa, index, 80, 5, min_len, None, 100)
            assert api.coverage_sums(ctx, soa, index, 80, 5, min_len, stream_resident=True) == want, (form, min_len, "resident")


# ================================================================================================ GPU: device pipeline
def _pipe(st, index, min_len, **kw):
    from metamlst_b200 import pipeline
    lens = np.asarray(st.ref_lens)
    return pipeline.DevicePipeline(st, index, lambda t: "A" * int(lens[t]), minscore=80, max_xM=5, min_read_len=min_len, **kw)


@gpu
@pytest.mark.parametrize("case", CASES, ids=lambda c: "%s-%s" % c)
def test_device_pipeline_coverage_in_file_order(bams, case):
    """DevicePipeline.run_coverage on host-unpacked streams (orig_idx when the file was not sorted) and on device-ingested
    streams of the same file."""
    path, h, recs, _db = bams[case]
    soa = _unpack(path, case[1])
    index = api.AlleleIndex(soa.ref_names)
    host = streams.DeviceStreams.from_soa(soa, "cuda:0", want_qhash=True)
    assert (host.orig_idx is None) == (case[1] == "coord")
    dev = bam.ingest_bam(path, 0, presorted=(case[1] == "coord"), want_qhash=True)
    for min_len in MIN_LENS:
        want = _bank_sums(orc.stage1(h, recs, 80, 5, min_len, None, 100)[1])
        assert _pipe(host, index, min_len).run_coverage() == want, ("host", min_len)
        assert _pipe(dev, index, min_len).run_coverage() == want, ("device ingest", min_len)


def _shards(case, bams, mode, world):
    path, h, recs, _db = bams[case]
    soa = _unpack(path, case[1])
    index = api.AlleleIndex(soa.ref_names)
    if mode == "slice":   # a device-ingested sample cut after packing
        whole = bam.ingest_bam(path, 0, presorted=(case[1] == "coord"), want_qhash=True)
        return h, recs, index, [whole.slice_ranges(r, world) for r in range(world)]
    return h, recs, index, [streams.DeviceStreams.from_soa(soa, "cuda:0", rank=r, world=world, mode=mode, locus_of=index.locus_of,
                                                           want_qhash=True) for r in range(world)]


@gpu
@pytest.mark.parametrize("world", [1, 2, 3, 4])
@pytest.mark.parametrize("mode", ["ranges", "loci", "slice"])
@pytest.mark.parametrize("case", [("synth", "name"), ("two_org", "name"), ("two_org", "coord")], ids=lambda c: "%s-%s" % c)
def test_shards_add_up_to_the_whole_sample(bams, case, mode, world):
    """The sharded coverage of run_coverage, driven step by step over shard pipelines on one device: insert on every shard,
    every record shard merges the other shards' table entries (owner-mode "loci" shards do not), sum pass; the per-shard sums
    add up -- what the all-reduce does -- to the whole sample."""
    h, recs, index, shards = _shards(case, bams, mode, world)
    for min_len in (1, 50):
        want = _bank_sums(orc.stage1(h, recs, 80, 5, min_len, None, 100)[1])
        pipes = [_pipe(st, index, min_len) for st in shards]
        for p in pipes:
            p.coverage_insert()
        if mode != "loci":
            entries = [p.coverage_entries() for p in pipes]
            for r, p in enumerate(pipes):
                for s, e in enumerate(entries):
                    if s != r:
                        p.coverage_merge(e)
        tot = sum(p.coverage_sum().cpu().numpy().astype(np.int64) for p in pipes)
        assert {"%s_%s" % index.locus_names[l]: int(v) for l, v in enumerate(tot) if v} == want, min_len
        if world == 1:
            assert _pipe(shards[0], index, min_len).run_coverage() == want


@gpu
def test_merge_skips_padding_and_absent_keys():
    """mmlst_coverage_merge_dev: rows of zeros (the padding of the all-gather) and keys the table does not hold change nothing;
    a present key takes the larger value word only."""
    lib = native.lib()
    slots = 1024
    table = torch.zeros(slots * 3, dtype=torch.int64, device="cuda")
    tid = np.zeros(50, np.uint32)
    key = np.stack([np.arange(1, 51), np.arange(50)], 1).astype(np.uint64)
    d = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a).view(dt)).cuda()
    args = [d(tid, np.int32), d(np.full(50, 150, np.int16), np.int16), d(np.zeros(50, np.uint8), np.uint8), d(np.full(50, 70, np.uint16), np.int16),
            None, d(key, np.int64)]
    allow, locus_of = d(np.ones(1, np.uint8), np.uint8), d(np.zeros(1, np.uint32), np.int32)
    cov = torch.zeros(2, dtype=torch.int64, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    native.check(lib.mmlst_coverage_insert_dev(*[native.ptr(a) for a in args], 50, 0, native.ptr(allow), native.ptr(locus_of), 1, 100, 5, 0,
                                               native.ptr(table), slots, 0, stream))
    before = table.clone()
    keys = table[: 2 * slots].view(slots, 2)
    occ = (keys != 0).any(1)
    assert int(occ.sum()) == 50
    mine_k, mine_v = keys[occ].clone(), table[2 * slots:][occ].clone()
    foreign_k = torch.cat([torch.zeros((7, 2), dtype=torch.int64, device="cuda"), mine_k + 12345, mine_k[:10]])
    foreign_v = torch.cat([torch.full((7,), 1 << 60, dtype=torch.int64, device="cuda"), torch.full((50,), 1 << 60, dtype=torch.int64, device="cuda"),
                           mine_v[:5] + (1 << 20), mine_v[5:10] - 1])
    native.check(lib.mmlst_coverage_merge_dev(native.ptr(foreign_k.contiguous()), native.ptr(foreign_v), int(foreign_k.shape[0]), native.ptr(table),
                                              slots, stream))
    after = table.clone()
    assert torch.equal(after[: 2 * slots], before[: 2 * slots])          # keys untouched, nothing inserted
    vals_after = after[2 * slots:][occ]
    assert torch.equal(vals_after[:5], mine_v[:5] + (1 << 20)) and torch.equal(vals_after[5:], mine_v[5:])
    native.check(lib.mmlst_coverage_sum_dev(*[native.ptr(a) for a in args], 50, 0, native.ptr(allow), native.ptr(locus_of), 1, 100, 5, 0,
                                            native.ptr(table), slots, native.ptr(cov), stream))
    assert int(cov[0]) == 45 * 70   # the five names whose maximum now lies elsewhere are added by nobody here


# ================================================================================================ GPU: the driver's stdout
def _captured_coverage(monkeypatch):
    """Every coverage dict the driver renders into its allele table, with the text it rendered."""
    from metamlst_b200 import sample
    seen = []
    real = sample._screen_allele_table

    def spy(call, genes, coverage, longest):
        text = real(call, genes, coverage, longest)
        seen.append((call, genes, dict(coverage), longest, text))
        return text
    monkeypatch.setattr(sample, "_screen_allele_table", spy)
    return seen, real


@gpu
@pytest.mark.parametrize("min_len", [1, 50])
@pytest.mark.parametrize("engine,ingest", [("device", "host"), ("device", "device"), ("onecall", "host")])   # device ingest feeds the device engine only
@pytest.mark.parametrize("name", ["basic", "two_org"])
def test_driver_prints_the_reference_coverage(bams, monkeypatch, tmp_path, name, ingest, engine, min_len):
    """SampleTyper.type_bam(want_stdout=True) on a rewritten name-ordered BAM: the coverage behind every printed allele table
    is the oracle's sequenceBank sum, and the printed table is the one those sums give."""
    from metamlst_b200 import sample
    path, h, recs, db = bams[(name, "name")]
    seen, real = _captured_coverage(monkeypatch)
    typer = sample.SampleTyper(db, device=0, engine=engine, ingest=ingest, min_read_len=min_len)
    res = typer.type_bam(path, str(tmp_path / "out"), want_stdout=True)
    cel, bank, _t, _i = orc.stage1(h, recs, 80, 5, min_len, None, 100)
    want = _bank_sums(bank)
    assert seen, "no allele table was printed"
    for call, genes, cov, longest, text in seen:
        for g in genes:
            k = call.species + "_" + g
            assert cov[k] == want[k], k
        assert text == real(call, cel[call.species], want, longest)
        assert text in res.stdout
    typer.close()


# ================================================================================================ GPU: two real ranks
@gpu
def test_two_ranks_print_the_reference_coverage(bams, tmp_path):
    """torchrun x 2 (NCCL): a rewritten name-ordered BAM typed by two ranks, each scoring a contiguous range of the sorted stream
    (names of a locus fall on both sides of the cut); rank 0's coverage equals the oracle's."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    path, h, recs, db = bams[("two_org", "name")]
    want = _bank_sums(orc.stage1(h, recs, 80, 5, 1, None, 100)[1])
    out = str(tmp_path / "cov.json")
    env = dict(os.environ, PYTHONPATH=ROOT)
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29873", os.path.join(ROOT, "tests", "run_sharded_coverage.py"), path, db, "1", out], env=env,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=600)
    assert p.returncode == 0, p.stdout.decode()[-3000:]
    got = json.load(open(out))
    assert got and all(got[k] == want[k] for k in got), (got, want)
