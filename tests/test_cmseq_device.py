"""cmseq's BamFile over the device ingest (metamlst_b200/cmseq_api.py: BamFile(ingest="device"), contig-sharded with a group) and what it
stands on: `lenient_tags` in the device ingest (csrc/ingest_core.cuh, csrc/ingest.cu) and `mmlst_contig_stats_resident` (csrc/api.cu).

CPU: the lenient per-record text compiled for the host (tests/ingest_emul/ingest_lenient_emul.cpp) against `unpack_bam(lenient_tags=True)`,
the ctypes mirror of mmlst_dev_bam_info_t, the owner map, `merge_rank_results`, and the device route's host logic with its two seams
answered by the oracle.  GPU: the lenient ingest (one GPU and sharded) against the host unpacker, and every BamFile method of the device
route, on one GPU and sharded over W = 2, 3 and 5 ranks in one process, against the host route and the golden JSON."""
import ctypes as C
import functools
import glob
import os
import subprocess
import types
from fractions import Fraction

import numpy as np
import pytest

from conftest import GOLDEN, ROOT
from metamlst_b200 import bam, cmseq_api, native
from oracle import bamio
from test_cmseq_bulk import GOLD, BULK, _Oracle, _check_equal_to_per_contig, _kwargs, _same, write_many_contig_bam
from test_ingest_core import check as check_emulated, emulate

BAMS = sorted(glob.glob(os.path.join(GOLDEN, "*", "sample.bam")))
IDS = [os.path.basename(os.path.dirname(p)) for p in BAMS]
TAGF = [("AS", "loc_gte", 80), ("XM", "loc_lte", 5)]


# ---- inputs ----------------------------------------------------------------------------------------------------------------------
def write_lenient_bams(d):
    """The BAMs of test_bam_unpack's lenient test (fully tagged; BWA-like lean: AS and NM only, every 5th record without aux; positional
    fields present but no AS / XM by name) and one whose 1st fields leave int16 and whose 4th fields go negative on some records."""
    import helpers
    _db, tab = helpers.small_case(seed=23, n_reads=300, L=100, K=2, orgs=("ecoli",), apl=4)
    recs = list(bamio.table_records(tab.sorted_by_coord()))
    names, lens = list(tab.ref_names), [int(x) for x in tab.ref_lens]
    lean = [r._replace(aux=[] if i % 5 == 0 else [a for a in r.aux if a[0] == "AS"] + [bamio.int_aux("NM", 1)]) for i, r in enumerate(recs)]
    named = [r._replace(aux=[bamio.int_aux("NM", 3), bamio.int_aux("X0", 1), bamio.int_aux("X1", 0), bamio.int_aux("XO", 2)]) for r in recs]
    firsts, fourths = (40000, -40000, 32767, -32768, 90), (-3, 0, 300, 7)
    ranged = [r._replace(aux=[bamio.int_aux("AS", firsts[i % 5]), bamio.int_aux("XS", 0), bamio.int_aux("XN", 0), bamio.int_aux("XM", fourths[i % 4])])
              for i, r in enumerate(recs)]
    out = {}
    for name, rs in (("full", recs), ("lean", lean), ("named", named), ("ranged", ranged)):
        out[name] = os.path.join(str(d), name + ".bam")
        bamio.write_bam(out[name], names, lens, rs, sort_order="coordinate")
    return out


@pytest.fixture(scope="module")
def lenient_bams(tmp_path_factory):
    return write_lenient_bams(tmp_path_factory.mktemp("lenient"))


LENIENT = ["full", "lean", "named", "ranged"]


# ---- CPU: the lenient per-record text on the host --------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def emul_lenient(tmp_path_factory):
    emul = os.path.join(ROOT, "tests", "ingest_emul")
    so = str(tmp_path_factory.mktemp("emul") / "libingest_lenient_emul.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", emul, "-I", os.path.join(ROOT, "metamlst_b200", "csrc"), "-o", so,
                           os.path.join(emul, "ingest_lenient_emul.cpp")])
    lib = C.CDLL(so)
    for f in ("emul_parse_lenient", "emul_pack_lenient", "emul_untagged"):
        getattr(lib, f).restype = C.c_uint64
    lib.emul_chain.restype = C.c_longlong
    # test_ingest_core.emulate drives emul_parse / emul_pack: here they are the lenient forms
    return types.SimpleNamespace(emul_chain=lib.emul_chain, emul_parse=lib.emul_parse_lenient, emul_pack=lib.emul_pack_lenient,
                                 emul_pack_columns=lib.emul_pack_columns, untagged=lib.emul_untagged)


def _emulated_equals_host(lib, path):
    soa = bam.unpack_bam(path, pinned=False, lenient_tags=True)
    check_emulated(emulate(lib, open(path, "rb").read()), soa)
    assert int(lib.untagged()) == soa.n_untagged
    return soa


@pytest.mark.parametrize("name", LENIENT)
def test_lenient_parse_and_pack_equal_the_host_unpacker(emul_lenient, lenient_bams, name):
    soa = _emulated_equals_host(emul_lenient, lenient_bams[name])
    if name == "ranged":   # the rule's both sides are exercised: kept fields, replaced fields, untagged records
        assert {-32768, 32767}.issubset(set(soa.as0.tolist())) and 255 in soa.xm3.tolist() and 0 < soa.n_untagged < soa.n_prec
    if name in ("lean", "named"):
        assert soa.n_untagged == soa.n_prec > 0


@pytest.mark.parametrize("path", BAMS, ids=IDS)
def test_lenient_parse_and_pack_on_golden_bams(emul_lenient, path):
    assert _emulated_equals_host(emul_lenient, path).n_untagged == 0


def test_dev_bam_info_mirror_matches_the_header(tmp_path):
    body = 'printf(" %zu", sizeof(mmlst_dev_bam_info_t));'
    for f, _t in bam.DevBamInfo._fields_:
        body += 'printf(" %%zu", offsetof(mmlst_dev_bam_info_t, %s));' % f
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "mmlst.h"\nint main(void){' + body + 'return 0;}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert got == [C.sizeof(bam.DevBamInfo)] + [getattr(bam.DevBamInfo, f).offset for f, _t in bam.DevBamInfo._fields_]
    assert bam.DevBamInfo._fields_[-1][0] == "n_untagged"


# ---- CPU: ownership and the merge ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [1, 2, 3, 5, 8, 64])
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_owner_map_is_contiguous_covering_and_balanced(world, seed):
    rng = np.random.default_rng(seed)
    lens = rng.integers(1, [10, 5000, 3_000_000][seed], int(rng.integers(1, 40)))
    own = cmseq_api.owner_map(lens, world)
    assert own.shape == lens.shape and own.dtype == np.int32
    assert (np.diff(own) >= 0).all() and own.min() >= 0 and own.max() < world   # contiguous header ranges, every contig owned
    total, start = int(lens.sum()), 0
    for t, ln in enumerate(lens.tolist()):   # the rule, in exact arithmetic
        r = int(own[t])
        assert Fraction(r * total, world) <= start < Fraction((r + 1) * total, world)
        start += ln
    share = np.bincount(own, weights=lens, minlength=world)
    assert (share <= total / world + lens.max()).all()   # a rank holds its 1/W of the columns plus at most one contig
    if world > len(lens):
        assert (share == 0).any()


def test_owner_map_edges():
    assert cmseq_api.owner_map([7], 5).tolist() == [0]
    assert cmseq_api.owner_map([1] * 6, 3).tolist() == [0, 0, 1, 1, 2, 2]
    assert cmseq_api.owner_map([1, 1, 100], 4).tolist() == [0, 0, 0]
    assert cmseq_api.owner_map([], 3).tolist() == []


def test_merge_rank_results_is_the_union_in_header_order():
    refs = ["c%d" % i for i in range(9)]
    whole = {n: {"v": i, "l": [i] * i} for i, n in enumerate(refs) if i != 4}
    parts = [{n: whole[n] for n in ("c6", "c0", "c2")}, {}, {n: whole[n] for n in ("c8", "c1", "c3", "c5", "c7")}]
    got = cmseq_api.merge_rank_results(parts, refs)
    assert list(got) == list(whole) and got == whole
    with pytest.raises(ValueError):
        cmseq_api.merge_rank_results([{"c1": 1}, {"c1": 1}], refs)
    with pytest.raises(KeyError):
        cmseq_api.merge_rank_results([{"nope": 1}], refs)


def test_group_needs_the_device_route():
    with pytest.raises(ValueError, match="ingest='device'"):
        cmseq_api.BamFile(BAMS[0], ctx=object(), group=cmseq_api._LocalRank(cmseq_api._LocalGroup(2), 0))
    with pytest.raises(ValueError):
        cmseq_api.BamFile(BAMS[0], ctx=object(), ingest="gpu")


# ---- CPU: the device route's host logic, its seams answered by the oracle --------------------------------------------------------
@pytest.fixture
def device_route_on_the_oracle(monkeypatch):
    """BamFile(ingest="device") with the ingest answered by the host unpacker and both resident seams by the oracle."""
    def make(path):
        o = _Oracle(path)
        monkeypatch.setattr(cmseq_api, "_resident_counts", o.contig_counts)
        monkeypatch.setattr(cmseq_api, "_resident_stats", o.bulk_stats)
        monkeypatch.setattr(cmseq_api, "_contig_counts", None)   # the host route's seams must not be reached
        monkeypatch.setattr(cmseq_api, "_bulk_stats", None)
        calls = []

        def ingest(p, device, minqual, want_qhash, lenient_tags, check_crc):
            assert (want_qhash, lenient_tags, check_crc) == (False, True, True)
            calls.append(minqual)
            return bam.unpack_bam(p, minqual=minqual, want_qhash=False, lenient_tags=True, pinned=False)
        monkeypatch.setattr(cmseq_api.bam_mod, "ingest_bam", ingest)
        return calls
    return make


@pytest.mark.parametrize("scen", sorted(GOLD))
def test_device_route_host_logic_matches_the_reference(scen, device_route_on_the_oracle):
    path = os.path.join(GOLDEN, scen, "sample.bam")
    calls = device_route_on_the_oracle(path)
    bf = cmseq_api.BamFile(path, ctx=object(), ingest="device")
    _check_equal_to_per_contig(bf, GOLD[scen]["cases"], GOLD[scen]["cases"])
    assert len(calls) == len(set(calls))   # one ingest per threshold
    g = GOLD[scen]
    assert sorted(cmseq_api.BamFile(path, minimumReadsAligning=50, minlen=100, ctx=object(), ingest="device").contigs) == g["kept_minreads_50"]


def test_device_route_untagged_rule_on_the_oracle(device_route_on_the_oracle, tmp_path):
    src = os.path.join(GOLDEN, "basic", "sample.bam")
    h, recs = bamio.read_bam(src)
    lean = str(tmp_path / "lean.bam")
    bamio.write_bam(lean, h.ref_names, h.ref_lens, [r._replace(aux=[a for a in r.aux if a[0] == "AS"]) for r in recs])
    device_route_on_the_oracle(lean)
    bf = cmseq_api.BamFile(lean, ctx=object(), ingest="device")
    with pytest.raises(KeyError, match="cmseq/cmseq.py:545"):
        bf.base_stats_all(BAM_tagFilter=TAGF)
    with pytest.raises(KeyError, match="cmseq/cmseq.py:545"):
        next(bf.get_contigs_obj()).get_base_stats(BAM_tagFilter=TAGF)
    bf.base_stats_all()


# ---- GPU: the lenient device ingest ----------------------------------------------------------------------------------------------
def _all_bams(lenient_bams):
    return [(n, lenient_bams[n]) for n in LENIENT] + list(zip(IDS, BAMS))


@pytest.mark.gpu
def test_lenient_ingest_equals_the_host_unpacker(lenient_bams):
    from test_ingest_gpu import same_streams
    for name, path in _all_bams(lenient_bams):
        for minqual in (20, 30):
            soa = bam.unpack_bam(path, pinned=False, lenient_tags=True, minqual=minqual)
            st = bam.ingest_bam(path, 0, lenient_tags=True, check_crc=True, minqual=minqual)
            same_streams(st, soa)
            assert st.lenient and st.n_untagged == soa.n_untagged, (name, minqual)
        with pytest.raises(native.MmlstError) if name in ("lean", "named", "ranged") else _nothing():
            bam.ingest_bam(path, 0)   # the strict ingest still refuses what the strict unpacker refuses


class _nothing:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


@pytest.mark.gpu
@pytest.mark.parametrize("W", [2, 3, 5])
def test_lenient_sharded_ingest_equals_the_host_stream_cut_by_owner(lenient_bams, W, monkeypatch):
    from test_ingest_sharded import _check_ranks
    monkeypatch.setattr(bam, "unpack_bam", functools.partial(bam.unpack_bam, lenient_tags=True))
    for name, path in _all_bams(lenient_bams):
        soa = bam.unpack_bam(path, pinned=False)
        ranks = _check_ranks(path, W, lenient_tags=True)
        assert all(s.lenient for s in ranks) and sum(s.n_untagged for s in ranks) == soa.n_untagged, (name, W)


@pytest.mark.gpu
def test_proper_pairs_stay_refused_and_lenient_streams_are_not_scored(lenient_bams, tmp_path):
    from metamlst_b200 import api, pipeline
    h, recs = bamio.read_bam(lenient_bams["lean"])
    pp = str(tmp_path / "paired.bam")
    bamio.write_bam(pp, h.ref_names, h.ref_lens, [r._replace(flag=r.flag | 0x3) for r in recs[:10]], sort_order="coordinate")
    with pytest.raises(native.MmlstError, match="proper-pair"):
        bam.ingest_bam(pp, 0, lenient_tags=True)
    with pytest.raises(native.MmlstError, match="proper-pair"):
        bam.ingest_bam_local(pp, 2, 0, lenient_tags=True)
    st = bam.ingest_bam(lenient_bams["full"], 0, lenient_tags=True)
    index = api.AlleleIndex(st.ref_names)
    with pytest.raises(ValueError, match="lenient_tags"):
        pipeline.DevicePipeline(st, index, lambda t: "A" * int(st.ref_lens[t]))
    strict = bam.ingest_bam(lenient_bams["full"], 0)
    pipe = pipeline.DevicePipeline(strict, index, lambda t: "A" * int(st.ref_lens[t]))
    with pytest.raises(ValueError, match="lenient_tags"):
        pipe.rebind(st)


# ---- GPU: BamFile(ingest="device") -----------------------------------------------------------------------------------------------
def _distinct(cases):
    seen, out = set(), []
    for c in cases:
        k = (c["method"], repr(sorted(c["kwargs"].items())))
        if k not in seen:
            seen.add(k)
            out.append(c)
    return out


def _bulk(bf, case, **extra):
    kw = {k: v for k, v in _kwargs(case).items() if k != "stats_value"}
    return getattr(bf, BULK[case["method"]])(**kw, **extra)


@pytest.mark.gpu
@pytest.mark.parametrize("scen", sorted(GOLD))
def test_device_route_equals_the_host_route_and_the_reference(scen):
    path = os.path.join(GOLDEN, scen, "sample.bam")
    dev, host = cmseq_api.BamFile(path, ingest="device"), cmseq_api.BamFile(path)
    try:
        assert dev.references == host.references and dev.lengths == host.lengths and list(dev.contigs) == list(host.contigs)
        _check_equal_to_per_contig(dev, GOLD[scen]["cases"], GOLD[scen]["cases"])
        _check_equal_to_per_contig(dev, GOLD[scen]["cases"][:20], None, col_budget=1)
        for case in _distinct(GOLD[scen]["cases"]):
            for budget in (1, cmseq_api.DEFAULT_COL_BUDGET):
                _same(_bulk(dev, case, col_budget=budget), _bulk(host, case), case["method"])
        assert sorted(cmseq_api.BamFile(path, ingest="device", minimumReadsAligning=50, minlen=100).contigs) == GOLD[scen]["kept_minreads_50"]
    finally:
        dev.close()
        host.close()


@pytest.fixture(scope="module")
def many_bam(tmp_path_factory):
    path = str(tmp_path_factory.mktemp("many") / "many.bam")
    write_many_contig_bam(path)
    return path


MANY_CALLS = [("polymorphism_rate_all", {"mincov": 5, "pvalue": 1.1, "dominant_frq_thrsh": 0.8}),
              ("polymorphism_rate_all", {"mincov": 5, "pvalue": 1.1, "dominant_frq_thrsh": float(np.nextafter(0.8, 1.0))}),
              ("breadth_and_depth_of_coverage_all", {"mincov": 5, "minqual": 30}),
              ("breadth_and_depth_of_coverage_all", {"mincov": 2, "minqual": 5, "trunc": 1500}),
              ("base_stats_all", {"BAM_tagFilter": TAGF}),
              ("reference_free_consensus_all", {"consensus_rule": cmseq_api.BamContig.majority_rule_polymorphicLoci, "mincov": 2, "minqual": 20,
                                                "dominant_frq_thrsh": 0.99}),
              ("reference_free_consensus_all", {"BAM_tagFilter": TAGF, "noneCharacter": "N"})]


@pytest.mark.gpu
def test_device_route_on_many_contigs(many_bam):
    dev, host = cmseq_api.BamFile(many_bam, ingest="device"), cmseq_api.BamFile(many_bam)
    try:
        assert list(dev.contigs) == list(host.contigs) and len(dev.contigs) > 3000
        for budget in (1000, cmseq_api.DEFAULT_COL_BUDGET):
            for method, kw in MANY_CALLS:
                _same(getattr(dev, method)(col_budget=budget, **kw), getattr(host, method)(**kw), "%s:%s" % (method, budget))
        sub = list(host.contigs)[1::7][::-1] + ["tie", "big", "wide", "capped"]
        _same(dev.polymorphism_rate_all(mincov=2, contigs=sub), host.polymorphism_rate_all(mincov=2, contigs=sub))
        for name in ("tie", "big", "wide", "capped", "onlyN", "filtered", "c00041", "c00003"):
            a, b = dev.get_contig_by_label(name), host.get_contig_by_label(name)
            _same(a.get_base_stats(min_read_depth=1, BAM_tagFilter=TAGF), b.get_base_stats(min_read_depth=1, BAM_tagFilter=TAGF), name)
            _same(a.breadth_and_depth_of_coverage(mincov=1, minqual=30, trunc=10), b.breadth_and_depth_of_coverage(mincov=1, minqual=30, trunc=10))
            assert a.reference_free_consensus(mincov=2) == b.reference_free_consensus(mincov=2)
    finally:
        dev.close()
        host.close()
    for kw in ({"filterInputList": ["big", "tie", "c00007", "c00100"]}, {"minlen": 2000}, {"minimumReadsAligning": 30}):
        dev, host = cmseq_api.BamFile(many_bam, ingest="device", **kw), cmseq_api.BamFile(many_bam, **kw)
        try:
            assert list(dev.contigs) == list(host.contigs), kw
            _same(dev.polymorphism_rate_all(mincov=2), host.polymorphism_rate_all(mincov=2))
        finally:
            dev.close()
            host.close()


def _lean(tmp_path):
    src = os.path.join(GOLDEN, "basic", "sample.bam")
    h, recs = bamio.read_bam(src)
    lean = str(tmp_path / "lean.bam")
    bamio.write_bam(lean, h.ref_names, h.ref_lens, [r._replace(aux=[a for a in r.aux if a[0] == "AS"]) for r in recs])
    return src, lean


@pytest.mark.gpu
def test_device_route_untagged_file(tmp_path):
    src, lean = _lean(tmp_path)
    bf, full = cmseq_api.BamFile(lean, ingest="device"), cmseq_api.BamFile(src)
    try:
        _same(bf.base_stats_all(), full.base_stats_all())
        _same(bf.reference_free_consensus_all(), full.reference_free_consensus_all())
        with pytest.raises(KeyError, match="cmseq/cmseq.py:545"):
            bf.base_stats_all(BAM_tagFilter=TAGF)
        with pytest.raises(KeyError, match="cmseq/cmseq.py:545"):
            next(bf.get_contigs_obj()).get_base_stats(BAM_tagFilter=TAGF)
    finally:
        bf.close()
        full.close()


# ---- GPU: contig-sharded, W ranks in one process -------------------------------------------------------------------------------
def _check_sharded(path, W, calls, **kw):
    host = cmseq_api.BamFile(path, **kw)
    ranks = cmseq_api.open_local(path, W, **kw)
    try:
        own = cmseq_api.owner_map(host.lengths, W)
        for r, h in enumerate(ranks):
            assert (h.rank, h.world) == (r, W) and h.references == host.references and h.lengths == host.lengths
            assert list(h.contigs) == [c for c in host.contigs if own[host._tid[c]] == r], r
            assert all(h.owner_of(c) == own[host._tid[c]] for c in host.references)
        for method, ckw in calls:
            want = getattr(host, method)(**ckw)
            got = cmseq_api.merge_rank_results([getattr(h, method)(**ckw) for h in ranks], host.references)
            _same(got, want, "%s:W=%d" % (method, W))
    finally:
        host.close()
        for h in ranks:
            h.close()


def _golden_calls(scen):
    out = []
    for case in _distinct(GOLD[scen]["cases"]):
        kw = {k: v for k, v in _kwargs(case).items() if k != "stats_value"}
        out.append((BULK[case["method"]], kw))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("W", [2, 3, 5])
@pytest.mark.parametrize("scen", sorted(GOLD))
def test_sharded_route_equals_the_host_route(scen, W):
    path = os.path.join(GOLDEN, scen, "sample.bam")
    calls = _golden_calls(scen)
    _check_sharded(path, W, calls)
    _check_sharded(path, W, calls[:3], minimumReadsAligning=50, minlen=100)


@pytest.mark.gpu
@pytest.mark.parametrize("W", [2, 3, 5])
def test_sharded_route_on_many_contigs(many_bam, W):
    _check_sharded(many_bam, W, MANY_CALLS + [("polymorphism_rate_all", {"mincov": 2, "contigs": ["tie", "big", "c00007", "c02000"]}),
                                              ("breadth_and_depth_of_coverage_all", {"col_budget": 1000})])
    _check_sharded(many_bam, W, MANY_CALLS[:2], minimumReadsAligning=30)


@pytest.mark.gpu
@pytest.mark.parametrize("W", [2, 3, 5])
def test_sharded_route_thresholds_and_the_untagged_rule(tmp_path, W):
    src, lean = _lean(tmp_path)
    ranks = cmseq_api.open_local(lean, W)
    host = cmseq_api.BamFile(lean)
    try:
        for h in ranks:
            with pytest.raises(KeyError, match="cmseq/cmseq.py:545"):
                h.base_stats_all(BAM_tagFilter=TAGF)
        owner = next(h for h in ranks if h.contigs)
        c = next(iter(owner.contigs.values()))
        with pytest.raises(RuntimeError, match="prepare"):
            c.get_base_stats(min_base_quality=17)
        for h in ranks:
            h.prepare(17)
        _same(c.get_base_stats(min_base_quality=17), host.get_contig_by_label(c.name).get_base_stats(min_base_quality=17))
        got = cmseq_api.merge_rank_results([h.base_stats_all(min_base_quality=17) for h in ranks], host.references)
        _same(got, host.base_stats_all(min_base_quality=17))
    finally:
        host.close()
        for h in ranks:
            h.close()


@pytest.mark.gpu
def test_two_ranks_gather_over_nccl(tmp_path):
    import socket
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    env = dict(os.environ, PYTHONPATH=ROOT)
    with socket.socket() as so:   # a port no other job holds
        so.bind(("127.0.0.1", 0))
        port = so.getsockname()[1]
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", str(port), os.path.join(ROOT, "tests", "run_cmseq_sharded.py")], env=env,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=900)
    assert p.returncode == 0, p.stdout.decode()[-3000:]
    assert "CMSEQ-SHARDED-OK" in p.stdout.decode()
