"""Edges of the stage-2 pileup kernels (csrc/pileup_bitsliced.cu, csrc/pileup_atomic.cu) against the C port over unpacked records
(`corc.contig_counts`, which shares nothing with the packer) and `corc.consensus`: every counter width of the bit-sliced flush, chunks
longer than the 63 tiles its counters hold, arbitrary chunk partitions and plane offsets, both shared-memory regimes and the atomic
fallback, wide records, the library's own chunk rule beyond one tile, the device-driven pass at chosen chunk lengths, and exact ties /
coverage thresholds at depth.  Counts are compared exactly, not only the consensus they lead to.  Needs a B200: `pytest -m gpu`."""
import numpy as np
import pytest

from metamlst_b200 import api, native, packing, synth
from oracle import corc

pytestmark = pytest.mark.gpu

TILE = 512            # records per tile of the bit-sliced kernel
LANE_PER_TILE = 16    # records a lane takes from one tile (TILE / 32)
MINQUAL = 20
MINSCORE, MAX_XM = 50, 3
ALPHABET = np.frombuffer(b"ACGTNacgtRY", np.uint8)   # lower case counts as its upper-case letter, R / Y / N in bin N
M, I, D, N, S = 0, 1, 2, 3, 4


@pytest.fixture(scope="module")
def ctx():
    c = native.Context(0)
    yield c
    c.close()


# ------------------------------------------------------------------------------------------------ mirrors of the kernel's arithmetic
def smem_regime(max_row_words):
    """Mirror of mmlst_pileup_bitsliced_fits and launch_pileup_bitsliced (csrc/pileup_bitsliced.cu): the bit-sliced kernel's dynamic
    shared memory for a stream whose largest row has max_row_words words -> "2cta" (two CTAs per SM), "1cta", or "atomic" (the
    launch falls back to the atomic kernel)."""
    stage_words = (TILE * max_row_words + 8 + 31) & ~31
    stage_bytes = stage_words * 4 + TILE * 16
    smem = 2 * stage_bytes + 2 * TILE * 16 + 2 * 8 + 16
    if max_row_words < 3 or smem > 220 * 1024:
        return "atomic"
    return "2cta" if smem <= 113 * 1024 else "1cta"


def flush_planes(tiles):
    """Mirror of flush_word (csrc/pileup_bitsliced.cu): bit-planes reduced at a flush after `tiles` tiles on one word."""
    return 6 if tiles <= 3 else 8 if tiles <= 15 else 10


# per-lane records that the next narrower flush could not hold: a case claiming a branch must reach this
BRANCH_THRESHOLD = {6: 1, 8: 1 << 6, 10: 1 << 8}


def row_words_of(nw):
    return 3 * nw + (1 if nw and (3 * nw) % 2 == 0 else 0)


# ------------------------------------------------------------------------------------------------ inputs
def make_table(ref_lens, tid, pos, cigars, seq, qual, AS, XM, names=None):
    """AlnTable of crafted records (flag 0, XS present so the 4th aux field is XM).  cigars: one [(op, len)] for every record or a
    list of them."""
    n = len(tid)
    if cigars and isinstance(cigars[0], tuple):
        cigars = [cigars] * n
    ncig = np.fromiter((len(c) for c in cigars), np.int64, n)
    cig_off = np.zeros(n + 1, np.int64)
    cig_off[1:] = np.cumsum(ncig)
    ops = np.fromiter(((ln << 4) | op for c in cigars for op, ln in c), np.uint32, int(cig_off[-1]))
    names = names or ["o_g%d_1" % i for i in range(len(ref_lens))]
    z = np.zeros(n, np.int32)
    AS = np.asarray(AS, np.int32)
    XM = np.asarray(XM, np.int32)
    return synth.AlnTable(names, np.asarray(ref_lens, np.int32), np.asarray(tid, np.int32), np.asarray(pos, np.int32), np.zeros(n, np.uint16),
                          np.arange(n, dtype=np.int64), cig_off, ops, seq.shape[1], np.ascontiguousarray(seq), np.ascontiguousarray(qual),
                          AS, AS.copy(), np.ones(n, bool), z, XM, z, z, XM.copy())


def letters(rng, ref_col, pair):
    """Bases and qualities of records given the reference column of every read base ([n, L], -1 = not on the reference).  Random letters
    of ALPHABET and qualities on both sides of MINQUAL, except in columns of fixed shape (col % 8): 7 = one letter of ACGTN for every
    record (quality 40), so that every record is counted there; 1, 3, 5, 6 = exact ties between the records of a pair (pair = 0 / 1):
    A = N, A = C, G = T, N = T."""
    n, L = ref_col.shape
    seq = ALPHABET[rng.integers(0, ALPHABET.shape[0], (n, L))]
    qual = np.where(rng.random((n, L)) < 0.3, rng.choice(np.array([2, 19], np.uint8), (n, L)),
                    rng.choice(np.array([20, 21, 35, 40], np.uint8), (n, L))).astype(np.uint8)
    m = ref_col % 8
    second = pair[:, None] == 1
    for k, (a, b) in {1: "AN", 3: "AC", 5: "GT", 6: "NT"}.items():
        sel = (m == k) & (ref_col >= 0)
        seq = np.where(sel, np.where(second, ord(b), ord(a)), seq).astype(np.uint8)
        qual = np.where(sel, 40, qual).astype(np.uint8)
    fixed = (m == 7) & (ref_col >= 0)
    seq = np.where(fixed, np.frombuffer(b"ACGTN", np.uint8)[(ref_col // 8) % 5], seq).astype(np.uint8)
    qual = np.where(fixed, 40, qual).astype(np.uint8)
    return seq, qual


def tags(rng, n_pairs, p_fail):
    """AS / XM per record, equal within a pair; about p_fail of the pairs fail the tag filter (AS < MINSCORE or XM > MAX_XM)."""
    AS = rng.integers(MINSCORE, MINSCORE + 20, n_pairs)
    XM = rng.integers(0, MAX_XM + 1, n_pairs)
    fail = rng.random(n_pairs) < p_fail
    low = fail & (rng.random(n_pairs) < 0.5)
    AS[low] = MINSCORE - rng.integers(1, 10, int(low.sum()))
    XM[fail & ~low] = MAX_XM + rng.integers(1, 4, int((fail & ~low).sum()))
    return np.repeat(AS, 2), np.repeat(XM, 2)


def ref_columns(pos, cigar, L):
    """[n, L] reference column of every read base of records with one CIGAR (-1: inserted / clipped)."""
    col = np.full(L, -1, np.int64)
    q = r = 0
    for op, ln in cigar:
        if op in (M, 7, 8):
            col[q:q + ln] = r + np.arange(ln)
        if op in (M, I, S, 7, 8):
            q += ln
        if op in (M, D, N, 7, 8):
            r += ln
    return np.where(col >= 0, pos[:, None].astype(np.int64) + col, -1)


def stacked_table(seed, n_rec, p_fail=0.15, contig_len=64, names=None, extra=None):
    """n_rec reads of 32 bases stacked on contig word 0: 3/4 at position 0, 1/4 at 31, which straddle words 0 and 1.  Every record
    touches word 0, so every lane of the warp owning it takes 16 records from every tile; column 31 is covered by every record
    (fixed letter, quality 40).  extra: (tid, n) records on another contig of the same length (lower AS), for the selection."""
    rng = np.random.default_rng(seed)
    n_pairs = n_rec // 2
    pos = np.repeat(np.where(np.arange(n_pairs) < (3 * n_pairs) // 4, 0, 31), 2)
    cig = [(M, 32)]
    seq, qual = letters(rng, ref_columns(pos, cig, 32), np.arange(2 * n_pairs) & 1)
    AS, XM = tags(rng, n_pairs, p_fail)
    tid = np.zeros(2 * n_pairs, np.int32)
    n_ref = 1
    if extra is not None:
        t2, n2 = extra
        n_ref = t2 + 1
        p2 = np.repeat(rng.integers(0, contig_len - 32, n2 // 2), 2)
        s2, q2 = letters(rng, ref_columns(p2, cig, 32), np.arange(n2) & 1)
        tid = np.concatenate([tid, np.full(n2, t2, np.int32)])
        pos = np.concatenate([pos, p2])
        seq, qual = np.concatenate([seq, s2]), np.concatenate([qual, q2])
        AS = np.concatenate([AS, np.full(n2, MINSCORE + 1)])
        XM = np.concatenate([XM, np.zeros(n2, np.int64)])
    return make_table([contig_len] * n_ref, tid, pos, cig, seq, qual, AS, XM, names)


def wide_table(seed, kind, n_rec=12000, contig_len=1013):
    """Reads whose rows touch up to `kind` contig words, on a contig whose length is not a multiple of 32; some reads end in its last,
    partial word.  6 / 7 / 8 / 9 words from the read length (170 / 250 bases and where a read starts inside its first word), 15 / 16
    from long D and N operations (100 bases over up to 480 reference columns)."""
    rng = np.random.default_rng(seed)
    n_pairs = n_rec // 2
    if kind in (6, 7, 8, 9):
        L = 170 if kind in (6, 7) else 250
        shapes = [[(M, L)], [(S, 7), (M, L - 14), (I, 2), (M, 5)]]
    else:
        L = 100
        shapes = [[(M, L)], [(M, 40), (D, 260), (M, 60)], [(M, 30), (N, 350), (M, 70)], [(S, 5), (M, 25), (N, 380), (M, 70)]]
    reflen = np.asarray([sum(ln for op, ln in c if op in (M, D, N)) for c in shapes])
    sh = rng.integers(0, len(shapes), n_pairs)
    sh[:16] = np.arange(16) % len(shapes)
    span = reflen[sh]
    limit = np.minimum(31, 32 * kind - span)          # largest offset inside the first word that keeps nw <= kind
    assert np.all(limit >= 0)
    start = rng.integers(0, contig_len - span + 1)
    end_at = contig_len - span                         # ending in the last, partial word (where the offset allows it)
    start = np.where((np.arange(n_pairs) < 16) & ((end_at & 31) <= limit), end_at, start)
    in_word = start & 31
    start = np.where(in_word > limit, start - (in_word - limit), start)
    lg = int(np.argmax(reflen))                        # and reaching exactly `kind` words: the longest shape at its largest offset
    sh[16:18] = lg
    start[16:18] = 64 + min(31, 32 * kind - int(reflen[lg]))
    pos = np.repeat(start, 2)
    cigars = [shapes[k] for k in np.repeat(sh, 2)]
    cols = np.concatenate([ref_columns(pos[i:i + 1], cigars[i], L) for i in range(pos.shape[0])])
    seq, qual = letters(rng, cols, np.arange(2 * n_pairs) & 1)
    AS, XM = tags(rng, n_pairs, 0.15)
    order = np.argsort(pos, kind="stable")
    return make_table([contig_len], np.zeros(2 * n_pairs, np.int32)[order], pos[order], [cigars[i] for i in order], seq[order], qual[order],
                      AS[order], XM[order])


# ------------------------------------------------------------------------------------------------ direct calls
def run_pileup(soa, chunks, impl, total_cols, plane_shift=0, row_bias=0, minscore=MINSCORE, max_xm=MAX_XM):
    """mmlst_pileup_dev on device copies of the packed stream with the test's chunk list [(rec_begin, rec_end, col_base, contig_len)].
    The plane rows are uploaded `plane_shift` words into the buffer and every record's row_off is stored `row_bias` higher (mod 2^32),
    so the chunks carry plane_delta = plane_shift - row_bias (mod 2^32).  Returns u32 counts [total_cols][5]."""
    import torch
    recs = soa.p_recs.copy()
    recs["row_off"] = ((recs["row_off"].astype(np.int64) + row_bias) & 0xFFFFFFFF).astype(np.uint32)
    planes = np.zeros(plane_shift + soa.planes.shape[0], np.uint32)
    planes[plane_shift:] = soa.planes
    delta = (plane_shift - row_bias) & 0xFFFFFFFF
    ck = np.asarray([(b, e, cb, cl, delta, 0, 0, 0) for b, e, cb, cl in chunks], np.uint32).reshape(-1, 8)
    dev = "cuda:0"
    recs_d = torch.from_numpy(recs.view(np.int32).reshape(-1, 4).copy()).to(dev)
    planes_d = torch.from_numpy(planes.view(np.int32)).to(dev)
    chunks_d = torch.from_numpy(ck.view(np.int32)).to(dev)
    counts = torch.zeros(total_cols * 5, dtype=torch.int32, device=dev)
    native.check(native.lib().mmlst_pileup_dev(native.ptr(recs_d), native.ptr(planes_d), native.ptr(chunks_d), int(ck.shape[0]), int(soa.max_row_words),
                                               int(minscore), int(max_xm), native.ptr(counts), int(total_cols), int(impl),
                                               torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return counts.cpu().numpy().view(np.uint32).reshape(total_cols, 5)


def reference(tab, tid=0, minscore=MINSCORE, max_xm=MAX_XM):
    want, _ = corc.contig_counts(tab.sorted_by_coord(), tid, MINQUAL, minscore, max_xm, None)
    return want


def contig_range(soa, tid=0):
    return int(soa.contig_start[tid]), int(soa.contig_start[tid + 1])


# ------------------------------------------------------------------------------------------------ 1, 2: counter widths, chunks > 63 tiles
@pytest.mark.parametrize("impl", [1, 2])
@pytest.mark.parametrize("tiles", [1, 3, 4, 15, 16, 62, 63, 64, 100, 127])
def test_counter_widths_and_chunks_past_63_tiles(tiles, impl):
    """One chunk of `tiles` tiles whose every record touches word 0: each lane of the warp owning it counts exactly 16 records per tile,
    so the flush at the chunk end reduces 6, 8 or 10 planes (1-3, 4-15, 16-63 tiles).  Past 63 tiles a lane holds >= 1024 records of
    word 0 -- more than 10 planes hold -- and the kernel must flush on its own while the word stays the same.  All five bins are
    populated: A/C/G/T, non-ACGT letters, qualities on both sides of minqual, tag-filter failures counted as N; column 31 is counted
    for every record."""
    tab = stacked_table(1000 + tiles, tiles * TILE)
    soa = packing.pack_table(tab, MINQUAL, max_depth=None)
    r0, r1 = contig_range(soa)
    assert (r0, r1) == (0, tiles * TILE) and (r1 - r0 + TILE - 1) // TILE == tiles
    assert np.all((soa.p_pos[r0:r1] >> 5) == 0) and np.all(soa.p_recs["nw"][r0:r1] >= 1)   # every record touches word 0
    per_lane = LANE_PER_TILE * tiles
    target = flush_planes(min(tiles, 63))
    assert per_lane >= BRANCH_THRESHOLD[target]
    assert (tiles > 63) == (per_lane >= 1 << 10)
    assert smem_regime(soa.max_row_words) == "2cta"
    want = reference(tab)
    assert int(want[31].sum()) == tiles * TILE and want[31, 3] > 0 and want[31, 4] > 0   # column 31: every record, T or (failing) N
    assert np.all(want.sum(axis=0) > 0)
    got = run_pileup(soa, [(r0, r1, 0, int(soa.ref_lens[0]))], impl, int(soa.ref_lens[0]))
    assert np.array_equal(got, want), np.argwhere(got != want)[:5]


# ------------------------------------------------------------------------------------------------ 3: arbitrary partitions, offsets
def _partition(rng, r0, r1):
    lens = [1, 31, 511, 512, 513]
    while r0 + sum(lens) < r1:
        lens.append(int(rng.integers(1, 70 * TILE)))
    cuts = np.minimum(r0 + np.cumsum([0] + lens), r1)
    return [(int(a), int(b)) for a, b in zip(cuts[:-1], cuts[1:]) if b > a]


@pytest.mark.parametrize("impl", [1, 2])
def test_arbitrary_partitions_col_base_and_plane_delta(impl):
    """One contig's records split into chunks of 1, 31, 511, 512, 513 records and random lengths (up to 70 tiles), starting mid-tile
    and mixed with the chunks of a second contig; the counts summed over the chunks equal the reference.  The columns live at
    col_base > 0 of a larger tensor (the columns around them stay zero), and the plane rows are uploaded at an offset so that
    plane_delta != 0, including a delta that wraps mod 2^32."""
    db = synth.make_db(("ecoli",), alleles_per_locus=2, n_profiles=4, seed=61, schemes={"ecoli": [("adk", 517), ("fumC", 333)]})
    tab = synth.make_sample(db, 40000, 100, seed=61, K=1, sub_err=0.02, n_frac=0.05, frac_clip=0.2, frac_indel=0.2)
    soa = packing.pack_table(tab, MINQUAL, max_depth=None)
    minscore, max_xm = 2 * tab.read_len - 24, 3
    tids = [t for t in range(len(tab.ref_names)) if contig_range(soa, t)[1] > contig_range(soa, t)[0]]
    assert len(tids) == 2
    rng = np.random.default_rng(61)
    base = [37, 37 + int(soa.ref_lens[tids[0]]) + 5]
    total = base[1] + int(soa.ref_lens[tids[1]]) + 3
    chunks = []
    for t, cb in zip(tids, base):
        r0, r1 = contig_range(soa, t)
        parts = _partition(rng, r0 + 100, r1)           # the first chunk starts mid-tile
        parts = [(r0, r0 + 100)] + parts
        assert sum(b - a for a, b in parts) == r1 - r0 and any((a - r0) % TILE for a, _ in parts)
        chunks += [(a, b, cb, int(soa.ref_lens[t])) for a, b in parts]
    rng.shuffle(chunks)
    wants = [reference(tab, t, minscore, max_xm) for t in tids]
    for shift, bias in ((0, 0), (4093, 0), (3, 256), (6, 0xFFFFFF00)):   # delta 2^32 - 253 wraps; with 2^32 - 256 the stored row_off wraps
        got = run_pileup(soa, chunks, impl, total, plane_shift=shift, row_bias=bias, minscore=minscore, max_xm=max_xm)
        for t, cb, want in zip(tids, base, wants):
            assert np.array_equal(got[cb:cb + want.shape[0]], want), (shift, bias, t)
        assert not got[:base[0]].any() and not got[base[0] + wants[0].shape[0]:base[1]].any() and not got[base[1] + wants[1].shape[0]:].any()


# ------------------------------------------------------------------------------------------------ 4: shared-memory regimes, wide records
@pytest.mark.parametrize("impl", [1, 2])
@pytest.mark.parametrize("kind,regime", [(6, "2cta"), (7, "1cta"), (8, "1cta"), (9, "1cta"), (15, "1cta"), (16, "atomic")])
def test_shared_memory_regimes_and_wide_records(kind, regime, impl):
    """Rows touching up to 6 and 7 words (two CTAs per SM -> one), 8 and 9 (a record wider than the 8-word window feeds several windows
    of one tile), 15 and 16 (the largest stage that fits -> the atomic fallback of impl=2), from read length and from long D / N
    operations, on a contig of 1013 columns with reads ending in its last, partial word; chunks of 1, 7 and all tiles."""
    tab = wide_table(2000 + kind, kind)
    soa = packing.pack_table(tab, MINQUAL, max_depth=None)
    nw = soa.p_recs["nw"]
    assert int(nw.max()) == kind and soa.max_row_words == row_words_of(kind)
    assert smem_regime(soa.max_row_words) == regime
    clen = int(soa.ref_lens[0])
    assert clen % 32 and np.any(soa.p_pos.astype(np.int64) + soa.p_reflen == clen)
    want = reference(tab)
    assert want[clen - 1].sum() > 0
    r0, r1 = contig_range(soa)
    for tiles in (1, 7, (r1 - r0 + TILE - 1) // TILE):
        cr = tiles * TILE
        chunks = [(b, min(r1, b + cr), 0, clen) for b in range(r0, r1, cr)]
        got = run_pileup(soa, chunks, impl, clen)
        assert np.array_equal(got, want), (tiles, np.argwhere(got != want)[:5])


# ------------------------------------------------------------------------------------------------ 5: the library's chunk rule beyond one tile
def test_library_chunk_rule_beyond_one_tile(ctx):
    """api.pileup_consensus (mmlst_pileup_consensus, chunk length by mmlst_chunk_records) over an uncapped sample with ~1.1 M records
    on the chosen contigs: chunks of more than 3 tiles, i.e. the 8-plane flush, through the product path."""
    db = synth.make_db(("ecoli",), alleles_per_locus=2, n_profiles=4, seed=71)
    tab = synth.make_sample(db, 1_100_000, 64, seed=71, K=1, sub_err=0.02, device="cuda:0")
    soa = packing.pack_table(tab, MINQUAL, max_depth=None)
    tids = sorted(set(int(t) for t in tab.tid))
    n = sum(contig_range(soa, t)[1] - contig_range(soa, t)[0] for t in tids)
    tiles = int(native.lib().mmlst_chunk_records(n)) // TILE
    assert n >= 1_000_000 and tiles >= 4 and flush_planes(tiles) >= 8 and LANE_PER_TILE * tiles >= BRANCH_THRESHOLD[8]
    assert smem_regime(soa.max_row_words) == "2cta"
    minscore, max_xm = 2 * tab.read_len - 24, 3
    dbs = [db.row_seq(t) for t in tids]
    st = tab.sorted_by_coord()
    wants = [corc.contig_counts(st, t, MINQUAL, minscore, max_xm, None)[0] for t in tids]
    for impl in (1, 2):
        seqs, holes, snps, counts, col_off = api.pileup_consensus(ctx, soa, tids, dbs, minscore, max_xm, 1, impl, want_counts=True)
        for i, want in enumerate(wants):
            assert np.array_equal(counts[col_off[i]:col_off[i + 1]], want), (impl, tids[i])
            assert (seqs[i], int(holes[i]), int(snps[i])) == corc.consensus(want, dbs[i].encode(), 1)


# ------------------------------------------------------------------------------------------------ 6: the device-driven pass
def _pipeline_case(tab, names, db_seqs, impl=0):
    from metamlst_b200 import pipeline, streams
    soa = packing.pack_table(tab, MINQUAL, max_depth=None)
    st = streams.DeviceStreams.from_soa(soa, "cuda:0")
    index = api.AlleleIndex(names)
    pipe = pipeline.DevicePipeline(st, index, lambda t: db_seqs[t], minscore=MINSCORE, max_xM=MAX_XM, min_read_len=30, impl=impl)
    want, _ = corc.contig_counts(tab.sorted_by_coord(), 0, MINQUAL, MINSCORE, MAX_XM, None)
    return soa, pipe, {"o": [(names[0],) + corc.consensus(want, db_seqs[0].encode(), 1)]}


@pytest.mark.parametrize("impl", [1, 2])
@pytest.mark.parametrize("tiles", [1, 4, 16, 63, 64])
def test_device_pass_at_chosen_chunk_lengths(monkeypatch, tiles, impl):
    """DevicePipeline (score -> mmlst_select_dev -> pileup -> consensus on the device) with MMLST_CHUNK_RECORDS = tiles x 512 over 64
    tiles of reads stacked on the allele the selection chooses (one allele with the most hits and the top AS): step(), the fused
    pileup + consensus launch and a captured graph all equal the reference."""
    rng = np.random.default_rng(tiles)
    names = ["o_g_1", "o_g_2"]
    db_seqs = ["".join(rng.choice(list("ACGT"), 64)) for _ in names]
    tab = stacked_table(3000 + tiles, 64 * TILE, p_fail=0.1, names=names, extra=(1, 64))
    monkeypatch.setenv("MMLST_CHUNK_RECORDS", str(tiles * TILE))
    soa, pipe, want = _pipeline_case(tab, names, db_seqs, impl)
    assert smem_regime(soa.max_row_words) == "2cta" and LANE_PER_TILE * min(tiles, 63) >= BRANCH_THRESHOLD[flush_planes(min(tiles, 63))]
    assert pipe.step() == want
    hdr = pipe.small_h.numpy()[:16]
    assert int(hdr[4]) == tiles * TILE and int(hdr[1]) == -(-64 // tiles)   # records per chunk, chunks of the chosen contig
    pipe.fused_tail = True    # one launch for pileup + consensus (impl=2; impl=1 keeps the two launches)
    assert pipe.step() == want
    pipe.capture()
    assert pipe.step_graph() == want and pipe.step_graph() == want
    pipe.fused_tail = False
    pipe.graph = None
    assert pipe.step() == want


def test_fused_device_pass_falls_back_for_rows_of_16_words():
    """The fused pileup + consensus launch over rows too wide for the bit-sliced kernel's shared memory (16 words): the atomic kernel and
    the separate consensus launch take over, with the same results."""
    names = ["o_g_1"]
    tab = wide_table(4016, 16, n_rec=4000)
    tab.ref_names = names
    rng = np.random.default_rng(16)
    db_seqs = ["".join(rng.choice(list("ACGT"), int(tab.ref_lens[0])))]
    soa, pipe, want = _pipeline_case(tab, names, db_seqs, impl=2)
    assert smem_regime(soa.max_row_words) == "atomic"
    pipe.fused_tail = True
    assert pipe.step() == want and pipe.step() == want
    pipe.fused_tail = False
    assert pipe.step() == want


# ------------------------------------------------------------------------------------------------ 7: consensus at depth
@pytest.mark.parametrize("impl", [1, 2])
def test_consensus_ties_and_mincov_at_depth(ctx, impl):
    """40 000 reads stacked on one word, no tag failures: exact ties at ~10^4 counts in the columns of fixed shape (A = N, A = C, G = T,
    N = T: the first maximum in the order A, C, G, N, T wins), mincov 1, equal to the A+C+G+T of column 3 and one above it."""
    tab = stacked_table(7000, 40000, p_fail=0.0)
    soa = packing.pack_table(tab, MINQUAL, max_depth=None)
    want = reference(tab)
    assert want[3, 0] == want[3, 1] >= 10000 and want[1, 0] == want[1, 4] and want[5, 2] == want[5, 3] and want[6, 4] == want[6, 3] > 0
    cov = int(want[3, :4].sum())
    rng = np.random.default_rng(7)
    dbs = ["".join(rng.choice(list("ACGT"), int(soa.ref_lens[0])))]
    for mincov in (1, cov, cov + 1):
        seqs, holes, snps, counts, _ = api.pileup_consensus(ctx, soa, [0], dbs, MINSCORE, MAX_XM, mincov, impl, want_counts=True)
        assert np.array_equal(counts, want)
        w = corc.consensus(want, dbs[0].encode(), mincov)
        assert (seqs[0], int(holes[0]), int(snps[0])) == w, mincov
        assert (w[0][3] == "A") == (mincov <= cov)
