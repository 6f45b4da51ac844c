"""Whole-BAM methods of seam S2' (metamlst_b200/cmseq_api.py: BamFile.base_stats_all / base_stats_arrays / reference_free_consensus_all /
polymorphism_rate_all / breadth_and_depth_of_coverage_all, csrc/contig_stats.cu).  Each must return, for every contig, exactly what the
per-contig method returns: same values, same types at every leaf, same key order.

CPU: the bulk seam (`cmseq_api._bulk_stats`) is answered by the oracle's counts and a numpy restatement of the device's column rule, the
per-contig seam by the oracle as in test_cmseq_api.py.  GPU (`-m gpu`): the real path on the golden BAMs and on a seeded BAM of several
thousand contigs."""
import ctypes as C
import gzip
import json
import math
import os
import re

import numpy as np
import pytest

from conftest import GOLDEN, ROOT
from helpers import records_to_table
from metamlst_b200 import cmseq_api, native
from oracle import bamio, corc

GOLD = json.loads(gzip.open(os.path.join(GOLDEN, "cmseq_api.json.gz")).read())
CSRC = os.path.join(ROOT, "metamlst_b200", "csrc")
BULK = {"get_base_stats": "base_stats_all", "get_all_base_values": "base_stats_all", "reference_free_consensus": "reference_free_consensus_all",
        "polymorphism_rate": "polymorphism_rate_all", "breadth_and_depth_of_coverage": "breadth_and_depth_of_coverage_all",
        "depth_of_coverage": "breadth_and_depth_of_coverage_all", "breadth_of_coverage": "breadth_and_depth_of_coverage_all"}


# ---- comparison ---------------------------------------------------------------------------------------------------------------
def _same(a, b, path=""):
    """Exact equality, NaN equal to NaN, and the same type at every leaf and container."""
    assert type(a) is type(b), (path, type(a), type(b))
    if isinstance(a, dict):
        assert list(a.keys()) == list(b.keys()), (path, list(a.keys())[:5], list(b.keys())[:5])
        for k in a:
            _same(a[k], b[k], path + "/" + str(k))
    elif isinstance(a, (list, tuple)) or type(a).__name__ == "dict_values":
        a, b = list(a), list(b)
        assert len(a) == len(b), (path, len(a), len(b))
        for i, (x, y) in enumerate(zip(a, b)):
            _same(x, y, path + "[%d]" % i)
    elif isinstance(a, (float, np.floating)) and math.isnan(a):
        assert math.isnan(b), (path, a, b)
    else:
        assert a == b, (path, a, b)


def _plain(x):
    if isinstance(x, dict):
        return {str(k): _plain(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)) or type(x).__name__ in ("dict_values", "dict_keys"):
        return [_plain(v) for v in x]
    if isinstance(x, np.generic):
        return x.item()
    return x


def _same_json(a, b, path=""):
    """test_cmseq_api's comparison against the golden JSON: ints and floats distinguished only by value."""
    if isinstance(a, dict) and isinstance(b, dict):
        assert list(a.keys()) == list(b.keys()), path
        for k in a:
            _same_json(a[k], b[k], path + "/" + str(k))
    elif isinstance(a, list) and isinstance(b, list):
        assert len(a) == len(b), path
        for i, (x, y) in enumerate(zip(a, b)):
            _same_json(x, y, path + "[%d]" % i)
    elif isinstance(a, float) and isinstance(b, float) and math.isnan(a) and math.isnan(b):
        pass
    else:
        assert a == b, (path, a, b)


def _kwargs(case):
    kw = dict(case["kwargs"])
    if "BAM_tagFilter" in kw:
        kw["BAM_tagFilter"] = [tuple(e) for e in kw["BAM_tagFilter"]]
    if "consensus_rule" in kw:
        kw["consensus_rule"] = getattr(cmseq_api.BamContig, kw["consensus_rule"])
    return kw


def _per_contig(contig, method, kw):
    kw = dict(kw)
    if method == "get_all_base_values":
        return contig.get_all_base_values(kw.pop("stats_value"), **kw)
    return getattr(contig, method)(**kw)


def _from_bulk(all_result, name, method, kw):
    """What the per-contig method returns, read from the whole-BAM result (the derived methods are the reference's one-liners)."""
    r = all_result[name]
    if method == "get_all_base_values":
        return [r[k].get(kw["stats_value"], 'NaN') for k in r]
    if method == "depth_of_coverage":
        return r[1]
    if method == "breadth_of_coverage":
        return r[0]
    return r


def _bulk_call(bf, method, kw, **extra):
    kw = {k: v for k, v in kw.items() if k != "stats_value"}
    return getattr(bf, BULK[method])(**kw, **extra)


def _check_equal_to_per_contig(bf, cases, golden=None, **extra):
    """Every distinct (method, kwargs) of `cases` over every kept contig: bulk == per-contig; golden results too where given."""
    seen = set()
    for case in cases:
        key = (case["method"], json.dumps(case["kwargs"], sort_keys=True))
        if key in seen:
            continue
        seen.add(key)
        kw = _kwargs(case)
        got = _bulk_call(bf, case["method"], kw, **extra)
        assert list(got) == list(bf.contigs), key
        for name in bf.contigs:
            want = _per_contig(bf.get_contig_by_label(name), case["method"], kw)
            _same(_from_bulk(got, name, case["method"], kw), want, "%s:%s" % (key, name))
    for case in golden or ():
        kw = _kwargs(case)
        got = _bulk_call(bf, case["method"], kw, **extra)
        _same_json(_plain(_from_bulk(got, case["contig"], case["method"], kw)), case["result"], "%s:%s" % (case["method"], case["contig"]))


# ---- numpy restatement of mmlst_contig_stats (the CPU answer of the bulk seam) ---------------------------------------------------
def restate_stats(counts_of, tids, col_off, prm, want_cons):
    """mmlst_contig_stats_dev restated: counts_of(tid) -> u32[len][5]."""
    width = cmseq_api._WIDTH[prm.mode]
    n = len(tids)
    sel_off, low_off, depth_off = np.zeros(n + 1, np.uint32), np.zeros(n + 1, np.uint32), np.zeros(n + 1, np.uint64)
    cols, vals, cons = [], [], []
    for i, t in enumerate(tids):
        c = np.asarray(counts_of(t), dtype=np.uint32)
        ln = int(col_off[i + 1] - col_off[i])
        assert c.shape == (ln, 5)
        acgt = c[:, :4].astype(np.int64)
        depth, bmax = acgt.sum(axis=1), acgt.max(axis=1)
        local = np.arange(ln)
        win = (local >= prm.trunc) & (local < ln - prm.trunc) if ln > 2 * prm.trunc else np.ones(ln, bool)
        sel = win & (depth >= prm.mincov)
        low = sel.copy()
        low[sel] = bmax[sel].astype(np.float64) / depth[sel].astype(np.float64) < prm.dominant_frq_thrsh
        sel_off[i + 1] = sel_off[i] + sel.sum()
        low_off[i + 1] = low_off[i] + low.sum()
        depth_off[i + 1] = depth_off[i] + np.uint64(depth[sel].sum())
        pick = low if prm.mode == native.STATS_LOWDOM else sel
        cols.append(local[pick])
        vals.append({native.STATS_COLUMNS: c[pick], native.STATS_DEPTH: depth[pick][:, None],
                     native.STATS_LOWDOM: np.stack([bmax[pick], depth[pick]], axis=1)}[prm.mode].astype(np.uint32))
        if want_cons:
            order = c[:, [0, 1, 2, 4, 3]]                    # A, C, G, N, T: argmax keeps the first maximum (H8)
            call = np.frombuffer(b"ACGNT", np.uint8)[np.argmax(order, axis=1)]
            cons.append(np.where(sel, call, np.uint8(prm.none_char)).astype(np.uint8))
    return cmseq_api._BatchStats(sel_off, low_off, depth_off,
                                 np.concatenate(cols).astype(np.uint32) if cols else np.zeros(0, np.uint32),
                                 np.concatenate(vals) if vals else np.zeros((0, width), np.uint32),
                                 (np.concatenate(cons) if cons else np.zeros(0, np.uint8)) if want_cons else None)


class _Oracle:
    """Both seams answered from the committed BAM by the C oracle; records the batches the bulk seam saw."""

    def __init__(self, bam):
        h, recs = bamio.read_bam(bam)
        self.tab = records_to_table(h, recs).sorted_by_coord()
        self.batches = []

    def counts(self, soa, tid, minscore, max_xm):
        return corc.contig_counts(self.tab, tid, soa.minqual, minscore, max_xm, 8000)[0]

    def contig_counts(self, ctx, soa, tid, minscore, max_xm):
        return self.counts(soa, tid, minscore, max_xm)

    def bulk_stats(self, ctx, soa, tids, col_off, minscore, max_xm, prm, want_cons):
        self.batches.append((list(tids), int(col_off[-1])))
        return restate_stats(lambda t: self.counts(soa, t, minscore, max_xm), tids, col_off, prm, want_cons)


@pytest.fixture
def oracle_seams(monkeypatch):
    def make(bam):
        o = _Oracle(bam)
        monkeypatch.setattr(cmseq_api, "_contig_counts", o.contig_counts)
        monkeypatch.setattr(cmseq_api, "_bulk_stats", o.bulk_stats)
        return o
    return make


# ---- CPU --------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("scen", sorted(GOLD))
def test_bulk_host_logic_equals_the_per_contig_methods(scen, oracle_seams):
    bam = os.path.join(GOLDEN, scen, "sample.bam")
    oracle_seams(bam)
    bf = cmseq_api.BamFile(bam, ctx=object())
    _check_equal_to_per_contig(bf, GOLD[scen]["cases"], GOLD[scen]["cases"])


def test_vectorised_p_values_equal_the_scalar_calls():
    from scipy import stats
    rng = np.random.default_rng(5)
    s = rng.integers(1, 20000, 4000)
    m = np.minimum(s, (s * rng.uniform(0.2, 1.0, s.size)).astype(np.int64) + 1)
    for err in (0.001, 0.01, 0.2):
        got = cmseq_api._pvalues(m, s, err)
        for i in range(s.size):
            want = stats.binom.cdf(float(m[i]), int(s[i]), 1.0 - err)
            assert type(got[i]) is type(want) and got[i] == want, (m[i], s[i], err)


def test_bulk_refuses_what_the_per_contig_methods_refuse(oracle_seams, tmp_path):
    bam = os.path.join(GOLDEN, "basic", "sample.bam")
    oracle_seams(bam)
    bf = cmseq_api.BamFile(bam, ctx=object())
    with pytest.raises(NotImplementedError):
        bf.base_stats_all(trimReads=(5, 5))
    with pytest.raises(NotImplementedError):
        bf.reference_free_consensus_all(trimReads=(5, 5))
    with pytest.raises(NotImplementedError):
        bf.base_stats_arrays(BAM_tagFilter=[("NM", "loc_lte", 3)])
    with pytest.raises(ValueError):
        bf.base_stats_all(min_read_depth=0)
    for f in (bf.polymorphism_rate_all, bf.breadth_and_depth_of_coverage_all, bf.reference_free_consensus_all):
        with pytest.raises(ValueError):
            f(mincov=0)
    with pytest.raises(NotImplementedError, match="majority_rule_polymorphicLoci"):
        bf.reference_free_consensus_all(consensus_rule=lambda col: "A")
    with pytest.raises(KeyError):
        bf.base_stats_all(contigs=["no_such_contig"])
    next(bf.get_contigs_obj()).set_stepper("all")
    for f in (bf.base_stats_all, bf.polymorphism_rate_all, bf.breadth_and_depth_of_coverage_all):
        with pytest.raises(NotImplementedError):
            f()
    # a tag filter on a file with untagged pileup records
    h, recs = bamio.read_bam(bam)
    lean = str(tmp_path / "lean.bam")
    bamio.write_bam(lean, h.ref_names, h.ref_lens, [r._replace(aux=[a for a in r.aux if a[0] == "AS"]) for r in recs])
    lb = cmseq_api.BamFile(lean, ctx=object())
    for f in (lb.base_stats_all, lb.reference_free_consensus_all):
        with pytest.raises(KeyError, match="cmseq/cmseq.py:545"):
            f(BAM_tagFilter=[("AS", "loc_gte", 50), ("XM", "loc_lte", 5)])
    full = cmseq_api.BamFile(bam, ctx=object())
    _same(lb.base_stats_all(), full.base_stats_all())


@pytest.mark.parametrize("scen", ["basic", "deep"])
def test_batching_does_not_change_results(scen, oracle_seams):
    bam = os.path.join(GOLDEN, scen, "sample.bam")
    o = oracle_seams(bam)
    bf = cmseq_api.BamFile(bam, ctx=object())
    lens = [c.length for c in bf.contigs.values()]
    one = max(lens)
    runs = {}
    for budget in (1, one, cmseq_api.DEFAULT_COL_BUDGET):
        o.batches.clear()
        runs[budget] = tuple(getattr(bf, m)(col_budget=budget, **kw) for m, kw in
                             (("base_stats_all", {"min_read_depth": 2}), ("reference_free_consensus_all", {"noneCharacter": "."}),
                              ("polymorphism_rate_all", {"pvalue": 0.9, "dominant_frq_thrsh": 0.99}),
                              ("breadth_and_depth_of_coverage_all", {"mincov": 1, "trunc": 10})))
        for tids, cols in o.batches:
            assert cols <= budget or len(tids) == 1, (budget, tids, cols)   # a contig longer than the budget runs alone
            assert tids == sorted(tids)
        if budget == 1:
            assert all(len(t) == 1 for t, _c in o.batches)
    for budget in (one, cmseq_api.DEFAULT_COL_BUDGET):
        _same(runs[budget], runs[1])


def test_subset_and_gates_select_the_same_contigs(oracle_seams):
    bam = os.path.join(GOLDEN, "two_org", "sample.bam")
    oracle_seams(bam)
    for kw in ({}, {"minimumReadsAligning": 50, "minlen": 100}, {"filterInputList": list(GOLD["two_org"]["contigs"])}):
        bf = cmseq_api.BamFile(bam, ctx=object(), **kw)
        got = bf.breadth_and_depth_of_coverage_all(mincov=1)
        assert list(got) == list(bf.contigs)
        sub = list(bf.contigs)[::3][::-1]
        part = bf.polymorphism_rate_all(contigs=sub)
        assert list(part) == [c for c in bf.contigs if c in set(sub)]   # header order
        for name in sub:
            _same(part[name], bf.get_contig_by_label(name).polymorphism_rate())


def test_a_batch_past_the_index_bound_is_refused():
    lib = native.lib()
    prm = native.ContigStatsParams(native.STATS_COLUMNS, 1, 0, ord("-"), 0.8)
    big = native.CONTIG_STATS_MAX_COLS + 1
    rc = lib.mmlst_contig_stats_dev(None, None, 1, big, C.byref(prm), None, 0, None, None, None, None, None, None, 0, None)
    assert rc == native.E_RANGE and "at most 858993459" in lib.mmlst_last_error().decode()
    col_off = np.array([0, big], np.uint32)
    tid = np.zeros(1, np.uint32)
    z = np.zeros(2, np.uint64)
    out = native.ContigStatsOut(native.ptr(z), native.ptr(z), native.ptr(z), None, None, None, 0, 0)
    soa = native.Soa()
    assert lib.mmlst_contig_stats(None, C.byref(soa), native.ptr(tid), 1, native.ptr(col_off), 0, 255, C.byref(prm), C.byref(out)) == native.E_RANGE
    # the driver keeps multi-contig batches under the bound and hands a longer contig to the library alone
    assert native.CONTIG_STATS_MAX_COLS == (2 ** 32 - 1) // 5


def test_ctypes_mirrors_match_the_header(tmp_path):
    import subprocess
    inc = os.path.join(ROOT, "include")
    pairs = [("mmlst_contig_stats_params", native.ContigStatsParams), ("mmlst_contig_stats_out", native.ContigStatsOut)]
    body = ""
    for cname, mirror in pairs:
        body += 'printf(" %%zu", sizeof(%s));' % cname
        for f, _t in mirror._fields_:
            body += 'printf(" %%zu", offsetof(%s, %s));' % (cname, f)
    body += 'printf(" %u %u %u %u", MMLST_STATS_COLUMNS, MMLST_STATS_DEPTH, MMLST_STATS_LOWDOM, MMLST_CONTIG_STATS_MAX_COLS);'
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "mmlst.h"\nint main(void){' + body + 'return 0;}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", inc, str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    i = 0
    for cname, mirror in pairs:
        assert got[i] == C.sizeof(mirror), cname
        offs = [getattr(mirror, f).offset for f, _t in mirror._fields_]
        assert got[i + 1:i + 1 + len(offs)] == offs, cname
        i += 1 + len(offs)
    assert got[i:] == [native.STATS_COLUMNS, native.STATS_DEPTH, native.STATS_LOWDOM, native.CONTIG_STATS_MAX_COLS]


def test_contig_stats_kernels_have_no_stack_frame_and_no_spills():
    log = os.path.join(CSRC, "contig_stats.ptxas.log")
    if not os.path.exists(log):
        pytest.skip("needs the ptxas logs of build()")
    hits = [m for m in re.finditer(r"Compiling entry function '(\S+)'.*?\n.*?\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads",
                                   open(log).read()) if "contig_stats" in m.group(1)]
    assert {k for k in ("cs_tile_kernel", "cs_scan_kernel", "cs_emit_kernel") if any(k in m.group(1) for m in hits)} == \
        {"cs_tile_kernel", "cs_scan_kernel", "cs_emit_kernel"}
    for m in hits:
        assert (int(m.group(2)), int(m.group(3)), int(m.group(4))) == (0, 0, 0), m.group(1)


# ---- a seeded BAM of many contigs ------------------------------------------------------------------------------------------------
def write_many_contig_bam(path, n_contigs=3000, seed=23, big=3_000_000, reads_per_kb=12.0):
    """Seeded coordinate-sorted BAM: contigs of 1 column to > 2^16 columns and one of `big` columns; contigs without reads, with only N
    bases, with only reads that fail the tag filter AS >= 80 / XM <= 5; a column of ratio exactly 0.8 (4 A, 1 C: contig `tie`), a
    position where more than 8000 reads start (depth cap), a read spanning 60000 skipped columns (rows too wide for the bit-sliced
    kernel's shared memory).  Returns {contig name: role}."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(1, 3000, n_contigs)
    lens[:20] = 1
    lens[20:40] = rng.integers(2, 40, 20)
    lens[40:44] = [65535, 65536, 65537, 131072 + 17]
    names = ["c%05d" % i for i in range(n_contigs)]
    roles = {}
    names += ["big", "tie", "capped", "onlyN", "filtered", "wide"]
    lens = list(int(x) for x in lens) + [big, 40, 500, 300, 300, 70000]
    ref = {i: rng.integers(0, 4, ln).astype(np.uint8) for i, ln in enumerate(lens)}
    recs = []
    k = 0

    def add(tid, pos, seq, qual, cigar=None, as_=90, xm=1):
        nonlocal k
        recs.append(bamio.BamRecord("r%d" % k, 0, tid, int(pos), 42, cigar or ((0, len(seq)),), seq, bytes(qual),
                                    (bamio.int_aux("AS", as_), bamio.int_aux("XS", 0), bamio.int_aux("XM", xm))))
        k += 1

    acgt = np.frombuffer(b"ACGT", np.uint8)
    for tid, ln in enumerate(lens):
        name = names[tid]
        if name in ("tie", "capped", "onlyN", "filtered", "wide"):
            continue
        if tid % 7 == 3 and name != "big":
            roles[name] = "no reads"
            continue
        n_reads = max(1, int(ln * reads_per_kb / 1000 * rng.uniform(0.2, 3.0)))
        for _ in range(n_reads):
            rl = int(min(ln, rng.integers(30, 151)))
            pos = int(rng.integers(0, ln - rl + 1))
            b = ref[tid][pos:pos + rl].copy()
            mut = rng.random(rl) < 0.03
            b[mut] = rng.integers(0, 4, int(mut.sum()))
            seq = acgt[b].tobytes().decode()
            if rng.random() < 0.02:
                seq = seq[:rl // 2] + "N" + seq[rl // 2 + 1:]
            add(tid, pos, seq, rng.integers(2, 41, rl).astype(np.uint8), as_=int(rng.integers(40, 120)), xm=int(rng.integers(0, 9)))
    t = names.index("tie")
    for i in range(5):
        add(t, 0, ("A" * 10) + ("C" if i == 4 else "A") + ("A" * 19), [35] * 30)
    roles["tie"] = "column 10: 4 A + 1 C, ratio 0.8"
    t = names.index("capped")
    for i in range(8200):
        add(t, 5, "ACGT" * 10, [35] * 40)
    roles["capped"] = "8200 reads start at column 5"
    t = names.index("onlyN")
    for i in range(20):
        add(t, 10 * i, "N" * 50, [35] * 50)
    roles["onlyN"] = "only N bases"
    t = names.index("filtered")
    for i in range(20):
        add(t, 10 * i, "ACGT" * 12, [35] * 48, as_=10, xm=8)
    roles["filtered"] = "every read fails AS >= 80 / XM <= 5"
    t = names.index("wide")
    add(t, 100, "ACGT" * 25, [35] * 100, cigar=((0, 50), (3, 60000), (0, 50)))
    add(t, 200, "ACGT" * 25, [35] * 100)
    roles["wide"] = "a read spans 60000 skipped columns"
    recs.sort(key=lambda r: (r.tid, r.pos))
    bamio.write_bam(path, names, lens, recs, sort_order="coordinate")
    return roles


@pytest.fixture(scope="module")
def many_bam(tmp_path_factory):
    path = str(tmp_path_factory.mktemp("many") / "many.bam")
    roles = write_many_contig_bam(path)
    return path, roles


# ---- GPU --------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("scen", sorted(GOLD))
def test_bulk_on_the_gpu_equals_the_per_contig_methods_and_the_reference(scen):
    bam = os.path.join(GOLDEN, scen, "sample.bam")
    bf = cmseq_api.BamFile(bam)
    try:
        _check_equal_to_per_contig(bf, GOLD[scen]["cases"], GOLD[scen]["cases"])
        _check_equal_to_per_contig(bf, GOLD[scen]["cases"][:20], None, col_budget=1)
    finally:
        bf.close()


def _device_flags_match_the_counts(bf, mode, minqual, tagf, mincov, trunc, thr, col_budget):
    """Full mode: every prefix, compacted column and consensus byte the device returned, re-derived on the host from the counts the
    per-contig seam returns for the same contigs."""
    seen = []
    real = cmseq_api._bulk_stats

    def spy(ctx, soa, tids, col_off, minscore, max_xm, prm, want_cons):
        r = real(ctx, soa, tids, col_off, minscore, max_xm, prm, want_cons)
        seen.append((soa, list(tids), col_off.copy(), minscore, max_xm, r))
        return r

    cmseq_api._bulk_stats = spy
    try:
        list(bf._bulk(None, minqual, tagf, mode, mincov, trunc, thr, ord("-"), True, col_budget))
    finally:
        cmseq_api._bulk_stats = real
    assert seen
    for soa, tids, col_off, minscore, max_xm, r in seen:
        prm = native.ContigStatsParams(mode, int(mincov), int(trunc), ord("-"), float(thr))
        want = restate_stats(lambda t: cmseq_api._contig_counts(bf.ctx, soa, t, minscore, max_xm), tids, col_off, prm, True)
        for f in want._fields:
            assert np.array_equal(getattr(r, f), getattr(want, f)), (f, tids[:3])
    return seen


@pytest.mark.gpu
def test_many_contigs_full_mode(many_bam):
    path, roles = many_bam
    bf = cmseq_api.BamFile(path)
    try:
        names = list(bf.contigs)
        assert len(names) > 3000 and max(c.length for c in bf.contigs.values()) >= 3_000_000
        tie = bf.get_contig_by_label("tie")
        tagf = [("AS", "loc_gte", 80), ("XM", "loc_lte", 5)]
        # ratio exactly at the threshold is not flagged; one ulp above it is
        at = bf.polymorphism_rate_all(mincov=5, pvalue=1.1, dominant_frq_thrsh=0.8, contigs=["tie"])["tie"]
        above = bf.polymorphism_rate_all(mincov=5, pvalue=1.1, dominant_frq_thrsh=float(np.nextafter(0.8, 1.0)), contigs=["tie"])["tie"]
        assert at["total_polymorphic_bases"] == 0 and above["total_polymorphic_bases"] == 1 and above["ratios"] == [0.8]
        # mincov at and one above the column's coverage
        assert bf.breadth_and_depth_of_coverage_all(mincov=5, minqual=30, contigs=["tie"])["tie"][0] == 30 / 40
        assert math.isnan(bf.breadth_and_depth_of_coverage_all(mincov=6, minqual=30, contigs=["tie"])["tie"][0])
        _same(bf.polymorphism_rate_all(mincov=5, dominant_frq_thrsh=float(np.nextafter(0.8, 1.0)))["tie"],
              tie.polymorphism_rate(mincov=5, dominant_frq_thrsh=float(np.nextafter(0.8, 1.0))))
        # contigs with no reads, only N bases, only filtered reads: the empty forms
        filt = bf.base_stats_all(BAM_tagFilter=tagf, contigs=["filtered", "onlyN", "c00003"])
        assert all(type(v) is type(cmseq_api.defaultdict(dict)) and len(v) == 0 for v in filt.values())
        cons = bf.reference_free_consensus_all(BAM_tagFilter=tagf, contigs=["filtered", "onlyN", "c00003"], noneCharacter="~")
        assert cons == {n: "~" * bf.get_contig_by_label(n).length for n in ("c00003", "onlyN", "filtered")}
        # full mode: device flags and counts against the counts, at a forced tiny and the default budget
        for budget in (1000, cmseq_api.DEFAULT_COL_BUDGET):
            for mode, minqual, tagf_, mincov, trunc, thr in ((native.STATS_COLUMNS, 30, None, 1, 0, 0.8),
                                                             (native.STATS_LOWDOM, 20, tagf, 2, 0, 0.95),
                                                             (native.STATS_DEPTH, 30, None, 3, 20, 0.0)):
                _device_flags_match_the_counts(bf, mode, minqual, tagf_, mincov, trunc, thr, budget)
        # every method equals the per-contig loop, trunc below, at and above len / 2
        for budget in (1000, cmseq_api.DEFAULT_COL_BUDGET):
            for method, kw in (("breadth_and_depth_of_coverage", {"mincov": 1, "minqual": 30, "trunc": 10}),
                               ("breadth_and_depth_of_coverage", {"mincov": 2, "minqual": 5, "trunc": 1500}),
                               ("polymorphism_rate", {"mincov": 2, "minqual": 20, "pvalue": 0.9, "dominant_frq_thrsh": 0.99}),
                               ("reference_free_consensus", {"consensus_rule": cmseq_api.BamContig.majority_rule_polymorphicLoci,
                                                             "mincov": 2, "minqual": 20, "dominant_frq_thrsh": 0.99}),
                               ("reference_free_consensus", {"BAM_tagFilter": tagf, "noneCharacter": "N"})):
                got = getattr(bf, BULK[method])(col_budget=budget, **kw)
                assert list(got) == names
                for name in names:
                    _same(got[name], getattr(bf.get_contig_by_label(name), method)(**kw), "%s:%s" % (method, name))
        # trunc with len <= 2 trunc, = 2 trunc + 1 and larger (contig lengths 1..3000 cover all three at trunc 1500 and 20)
        lens = {c.length for c in bf.contigs.values()}
        assert 3000 - 1 in lens or any(l <= 3000 for l in lens)
        t = next(c for c in bf.contigs.values() if c.length % 2 == 1 and c.length > 3)
        got = bf.breadth_and_depth_of_coverage_all(mincov=1, minqual=5, trunc=t.length // 2, contigs=[t.name])[t.name]
        _same(got, t.breadth_and_depth_of_coverage(mincov=1, minqual=5, trunc=t.length // 2))
        a = bf.base_stats_arrays(min_read_depth=1, BAM_tagFilter=tagf)
        full = bf.base_stats_all(min_read_depth=1, BAM_tagFilter=tagf)
        assert a.names == names and int(a.offsets[-1]) == sum(len(v) for v in full.values())
        for name in ("big", "wide", "capped", "c00041", "c00042"):
            _same(full[name], bf.get_contig_by_label(name).get_base_stats(min_read_depth=1, BAM_tagFilter=tagf), name)
    finally:
        bf.close()


@pytest.mark.gpu
def test_contig_selection_matches_the_per_contig_loop(many_bam):
    path, _roles = many_bam
    for kw in ({"filterInputList": ["big", "tie", "c00007", "c00100"]}, {"minlen": 2000}, {"minimumReadsAligning": 30}):
        bf = cmseq_api.BamFile(path, **kw)
        try:
            got = bf.polymorphism_rate_all(mincov=2)
            assert list(got) == list(bf.contigs)
            for name in bf.contigs:
                _same(got[name], bf.get_contig_by_label(name).polymorphism_rate(mincov=2))
            sub = list(bf.contigs)[1::2]
            assert list(bf.breadth_and_depth_of_coverage_all(contigs=sub)) == sub
        finally:
            bf.close()


@pytest.mark.gpu
def test_untagged_file_on_the_gpu(tmp_path):
    src = os.path.join(GOLDEN, "basic", "sample.bam")
    h, recs = bamio.read_bam(src)
    lean = str(tmp_path / "lean.bam")
    bamio.write_bam(lean, h.ref_names, h.ref_lens, [r._replace(aux=[a for a in r.aux if a[0] == "AS"]) for r in recs])
    bf, full = cmseq_api.BamFile(lean), cmseq_api.BamFile(src)
    try:
        _same(bf.base_stats_all(), full.base_stats_all())
        _same(bf.reference_free_consensus_all(), full.reference_free_consensus_all())
        with pytest.raises(KeyError, match="cmseq/cmseq.py:545"):
            bf.base_stats_all(BAM_tagFilter=[("AS", "loc_gte", 50), ("XM", "loc_lte", 5)])
    finally:
        bf.close()
        full.close()


@pytest.mark.gpu
def test_contig_stats_dev_consume_leaves_zero_counts():
    """mmlst_contig_stats_dev with MMLST_CONSENSUS_CONSUME zeroes every count it read, and a second call on fresh counts gives the same."""
    import torch
    lib = native.lib()
    rng = np.random.default_rng(3)
    lens = [1, 5000, 0, 4096, 4097, 13, 0]
    col_off = np.zeros(len(lens) + 1, np.uint32)
    col_off[1:] = np.cumsum(lens)
    total = int(col_off[-1])
    counts = rng.integers(0, 6, (total, 5)).astype(np.uint32)
    prm = native.ContigStatsParams(native.STATS_COLUMNS, 2, 0, ord("-"), 0.7)
    dev = "cuda:0"
    d_counts = torch.from_numpy(counts.view(np.int32)).to(dev)
    d_off = torch.from_numpy(col_off.view(np.int32)).to(dev)
    scratch = torch.zeros(int(lib.mmlst_contig_stats_scratch_bytes(total)), dtype=torch.uint8, device=dev)
    n = len(lens)
    sel = torch.zeros(n + 1, dtype=torch.int32, device=dev)
    low = torch.zeros(n + 1, dtype=torch.int32, device=dev)
    dep = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    oc = torch.zeros(total, dtype=torch.int32, device=dev)
    ov = torch.zeros(total * 5, dtype=torch.int32, device=dev)
    cons = torch.zeros(total, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    native.check(lib.mmlst_contig_stats_dev(native.ptr(d_counts), native.ptr(d_off), n, total, C.byref(prm), native.ptr(scratch), scratch.numel(),
                                            native.ptr(sel), native.ptr(low), native.ptr(dep), native.ptr(oc), native.ptr(ov), native.ptr(cons),
                                            native.CONSENSUS_CONSUME, st))
    torch.cuda.synchronize()
    want = restate_stats(lambda i: counts[col_off[i]:col_off[i + 1]], list(range(n)), col_off, prm, True)
    k = int(want.sel_off[-1])
    assert np.array_equal(sel.cpu().numpy().view(np.uint32), want.sel_off) and np.array_equal(low.cpu().numpy().view(np.uint32), want.low_off)
    assert np.array_equal(dep.cpu().numpy().view(np.uint64), want.depth_off)
    assert np.array_equal(oc.cpu().numpy().view(np.uint32)[:k], want.cols)
    assert np.array_equal(ov.cpu().numpy().view(np.uint32)[:5 * k].reshape(k, 5), want.vals)
    assert np.array_equal(cons.cpu().numpy(), want.cons)
    assert int(d_counts.abs().sum()) == 0
