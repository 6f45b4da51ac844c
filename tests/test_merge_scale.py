"""The cohort merge's three device look-ups (metamlst_b200/merge.py) at the shape of a real MLST scheme: two organisms of 800-2500
alleles per locus and 12000 STs each, hazard rows appended in interleaved gene and organism order, thousands of queries and lists
per call, and a synthetic cohort of 700 samples.  Every device answer is compared with a plain restatement of the same operation:

  exact match      HammingIndex.exact_first (csrc/st_match.cu exact_clean_kernel / exact_flagged_kernel)
                   vs a {sequence: first row} dict built from the table in rowid order, and the verbatim sequenceLocate SQL;
  closest allele   HammingIndex.search (csrc/hamming.cu hamming_min_kernel, csrc/hamming_exact.cu)
                   vs the oracle's C stringDiff scan (oracle/corc.py hamming_min) on every query;
  ST assignment    ProfileIndex.define_profiles (csrc/st_match.cu st_count_kernel / st_emit_kernel)
                   vs an inverted-index count (allele -> profiles, set semantics) on every list, and the verbatim defineProfile SQL.

The merge itself runs on the GPU and on the CPU path (SQL look-ups, stringDiff from the C oracle); both must write the same files,
and the oracle's merge_bacterium must agree on a subset."""
import os
import random
import shutil
import sqlite3
from collections import Counter, defaultdict

import numpy as np
import pytest

from metamlst_b200 import api, merge, synth
from oracle import corc
from oracle import mlst_oracle as orc

ORGS = ("ecoli", "kpneumoniae")                 # 24- and 16-word planes (longest rows 536 + extensions and 501 + extensions)
PLANE_W = {"ecoli": 24, "kpneumoniae": 16}
APL = (2500, 800, 1733, 1024, 1297, 2049, 911, 1900, 803, 1202, 2222, 1031, 1555, 999)   # alleles per locus, scheme order
N_PROFILES = 12000
SHARED_N = (1, 64, 65, 255, 256, 257, 1100)    # the first locus of each organism has one allele in exactly this many STs
PAIR_N = 700                                   # ... and (that 1100-ST allele, allele 1 of the second locus) share 700 STs
N_HAZARDS = 240                                # hazard rows appended per organism
NO = api.NO_IDX
IUPAC = "RYKMSWBDHV"


def _sub(rng, ch):
    return rng.choice([c for c in "ACGT" if c != ch])


def _add_hazards(conn, rng):
    """Appends, in interleaved organism and gene order: the same sequence under another gene (or twice under one gene), prefixes and
    extensions of existing rows, and rows with N, IUPAC codes and lower case.  Every 97th original row also gets an N in place, so
    flagged rows sit in every part of the resident tiles."""
    rows = conn.execute("SELECT recID, bacterium, gene, alleleVariant, sequence FROM alleles ORDER BY recID").fetchall()
    by_gene = defaultdict(list)
    for r in rows:
        by_gene[(r[1], r[2])].append(r)
    upd = []
    for r in rows[::97]:
        p = rng.randrange(len(r[4]))
        upd.append((r[4][:p] + "N" + r[4][p + 1:], r[0]))
    conn.executemany("UPDATE alleles SET sequence = ? WHERE recID = ?", upd)
    nxt = defaultdict(lambda: 5001)              # above every variant the generator made
    flagged = {o: [] for o in ORGS}
    extra = []
    for k in range(N_HAZARDS):
        for o in ORGS:
            genes = [g for g, _l in synth.SCHEMES[o]]
            g = genes[k % 7]
            s = rng.choice(by_gene[(o, g)])[4]
            kind = (k // 7) % 8
            if kind == 0:                        # the sequence of a row of another gene (sometimes the same gene: a duplicate)
                s = rng.choice(by_gene[(o, genes[(k + k // 7) % 7])])[4]
            elif kind == 1:
                s = s[:-rng.randint(1, 40)]
            elif kind == 2:
                s = s + "".join(rng.choice("ACGT") for _ in range(rng.randint(1, min(40, PLANE_W[o] * 32 - len(s)))))
            elif kind == 3:
                p = rng.randrange(len(s))
                s = s[:p] + "N" + s[p + 1:]
            elif kind == 4:
                for p in rng.sample(range(len(s)), rng.randint(1, 3)):
                    s = s[:p] + rng.choice(IUPAC) + s[p + 1:]
            elif kind == 5:
                s = s.lower()
            elif kind == 6:
                p = rng.randrange(len(s) - 20)
                s = s[:p] + s[p:p + 20].lower() + s[p + 20:]
            elif kind == 7 and flagged[o]:       # a flagged sequence under a second gene
                s = rng.choice(flagged[o])
            if s != s.upper() or any(c not in "ACGT" for c in s):
                flagged[o].append(s)
            extra.append((g, o, nxt[(o, g)], s))
            nxt[(o, g)] += 1
    conn.executemany("INSERT INTO alleles (gene, bacterium, alleleVariant, sequence) VALUES (?,?,?,?)", extra)
    conn.commit()
    return extra


class Scale:
    def __init__(self, db, path, shared, hazards):
        self.db, self.path, self.shared, self.hazards = db, path, shared, hazards
        conn = sqlite3.connect(path)
        self.rows = {o: [(g, v, s) for g, v, s in conn.execute(
            "SELECT gene, alleleVariant, sequence FROM alleles WHERE bacterium = ? ORDER BY rowid", (o,))] for o in ORGS}
        conn.close()


@pytest.fixture(scope="module")
def scale(tmp_path_factory):
    db = synth.make_db(ORGS, alleles_per_locus=APL, n_profiles=N_PROFILES, seed=2024)
    nrng = np.random.default_rng(2024)
    shared = {}
    li0 = 0
    for o in ORGS:
        p = db.profiles[o]
        g0, g1 = db.loci[o][0][0], db.loci[o][1][0]
        res = APL[li0] - len(SHARED_N) + 1      # the top variants of the first locus are the shared ones
        bad = p[:, 0] >= res
        p[bad, 0] = nrng.integers(1, res, size=int(bad.sum()))
        perm = nrng.permutation(p.shape[0])
        k = 0
        for i, n in enumerate(SHARED_N):
            p[perm[k:k + n], 0] = res + i
            shared[(o, n)] = "%s_%s_%d" % (o, g0, res + i)
            k += n
        p[perm[k - SHARED_N[-1]:k - SHARED_N[-1] + PAIR_N], 1] = 1
        shared[(o, "pair")] = [shared[(o, SHARED_N[-1])], "%s_%s_1" % (o, g1)]
        li0 += len(db.loci[o])
    path = str(tmp_path_factory.mktemp("merge_scale") / "db.sqlite")
    db.write_sqlite(path)
    conn = sqlite3.connect(path)
    hazards = _add_hazards(conn, random.Random(2024))
    conn.close()
    return Scale(db, path, shared, hazards)


@pytest.fixture(scope="module")
def ctx():
    from metamlst_b200 import native
    c = native.Context(0)
    yield c
    c.close()


def _first_diff(got, want, what):
    for i, (g, w) in enumerate(zip(got, want)):
        if g != w:
            return "%s %d: got %r, want %r" % (what, i, g, w)
    return None if len(got) == len(want) else "%s: %d answers for %d" % (what, len(got), len(want))


# ---------------------------------------------------------------------------------------------------------------- references
def define_profile_ref(conn):
    """defineProfile restated without SQL: labels resolve to the first recID holding them; for the SET of resolved recIDs, count the
    `profiles` rows per profileCode; keep the codes reaching the maximum, in descending code order (what the statement's
    `ORDER BY T DESC` returns in SQLite 3.x); percentage over the number of resolved labels; [(0, 0)] when the last label is unknown."""
    rec_of = {}
    for rec, b, g, v in conn.execute("SELECT recID, bacterium, gene, alleleVariant FROM alleles ORDER BY recID"):
        rec_of.setdefault("%s_%s_%s" % (b, g, v), rec)
    inv = defaultdict(list)
    for code, allele in conn.execute("SELECT profileCode, alleleCode FROM profiles"):
        inv[allele].append(code)

    def define(labels):
        if labels[-1] not in rec_of:
            return [(0, 0)]
        recs = [rec_of[l] for l in labels if l in rec_of]
        cnt = Counter()
        for a in set(recs):
            cnt.update(inv.get(a, ()))
        if not cnt:
            return []
        top = max(cnt.values())
        return [(c, int((float(top) / float(len(recs))) * 100)) for c in sorted((c for c, n in cnt.items() if n == top), reverse=True)]
    return define


def corc_closest(path):
    """merge's Closest from the C oracle's stringDiff scan over the rows of each (organism, gene)."""
    conn = sqlite3.connect(path)
    tabs = {}
    for o in ORGS:
        seqs, rng_of = [], {}
        for g, s in conn.execute("SELECT gene, sequence FROM alleles WHERE bacterium = ? ORDER BY gene, rowid", (o,)):
            lo, _hi = rng_of.get(g, (len(seqs), 0))
            seqs.append(s.encode("latin-1"))
            rng_of[g] = (lo, len(seqs))
        off = np.zeros(len(seqs) + 1, np.int64)
        off[1:] = np.cumsum([len(s) for s in seqs])
        tabs[o] = (np.frombuffer(b"".join(seqs), np.uint8), off, rng_of)
    conn.close()

    def closest(bacterium, items):
        flat, off, rng_of = tabs[bacterium]
        have = [i for i, (g, _s) in enumerate(items) if g in rng_of]
        out = [1 << 30] * len(items)
        d, _a = corc.hamming_min([items[i][1].encode("latin-1") for i in have], flat, off, [rng_of[items[i][0]] for i in have])
        for i, x in zip(have, d):
            out[i] = int(x)
        return out
    return closest


# ---------------------------------------------------------------------------------------------------------------- CPU
def _tie_lists(conn, rng, organisms):
    genes = {o: [g for g, _l in synth.SCHEMES[o]] for o in organisms}
    prof = defaultdict(dict)
    for code, b, g, v in conn.execute("SELECT profileCode, alleles.bacterium, gene, alleleVariant FROM profiles, alleles "
                                      "WHERE alleleCode = alleles.recID"):
        prof[(b, code)][g] = v
    keys = sorted(prof)
    lists = []
    for _ in range(300):
        b, code = rng.choice(keys)
        labels = ["%s_%s_%s" % (b, g, prof[(b, code)][g]) for g in genes[b] if g in prof[(b, code)]]
        k = rng.randrange(6)
        if k == 0:
            labels = rng.sample(labels, rng.randint(1, 3))          # partial: many STs tie
        elif k == 1:
            labels.insert(3, "%s_nogene_1" % b)                     # unknown in the middle: dropped, denominator shrinks
        elif k == 2:
            labels[-1] = "%s_%s_99999" % (b, genes[b][-1])           # unknown last: [(0, 0)]
        elif k == 3:
            labels = labels[:2] + [labels[0]]                        # a label twice: a set test, counted twice in the denominator
        elif k == 4:
            o2 = rng.choice(organisms)
            labels = labels[:1] + ["%s_%s_%d" % (o2, genes[o2][1], rng.randint(1, 5))]   # possibly another organism's allele
        lists.append(labels)
    return lists


def test_oracle_define_profile_is_the_reference_statement(tmp_path):
    """OracleDB.define_profile, api.define_profile (the reference's statement run by sqlite3) and the plain count agree, ties in the
    order the statement returns them: the oracle merge takes the first tied ST of a partial line at 100 %."""
    path = str(tmp_path / "db.sqlite")
    synth.make_db(("ecoli", "saureus"), alleles_per_locus=10, n_profiles=400, seed=5).write_sqlite(path)
    conn = sqlite3.connect(path)
    odb = orc.OracleDB(path)
    ref = define_profile_ref(conn)
    lists = [["ecoli_adk_1"], ["ecoli_adk_1", "ecoli_fumC_2"], ["saureus_arcC_3"]] + _tie_lists(conn, random.Random(5), ("ecoli", "saureus"))
    n_ties = 0
    for labels in lists:
        want = api.define_profile(conn, labels)
        assert odb.define_profile(labels) == want, labels
        assert ref(labels) == want, labels
        n_ties += len(want) > 1
    assert n_ties >= 30


def test_oracle_merge_takes_the_statements_first_tie(tmp_path):
    """A partial line whose alleles several STs share: the merge (CPU path: SQL look-ups) and the oracle give it the same ST."""
    path = str(tmp_path / "db.sqlite")
    synth.make_db(("ecoli",), alleles_per_locus=10, n_profiles=400, seed=5).write_sqlite(path)
    folder = tmp_path / "nfo"
    folder.mkdir()
    (folder / "a.nfo").write_text("ecoli\ta\tecoli_adk_1::::99.5::0.0\r\n")
    (folder / "b.nfo").write_text("ecoli\tb\tecoli_adk_1::::98.0::0.0\tecoli_fumC_2::::97.0::0.0\r\n")
    states, _ = merge.merge_folder(str(folder), path, closest=lambda b, items: [0] * len(items), write=False)
    want = orc.merge_bacterium(orc.OracleDB(path), "ecoli", orc.parse_nfo_folder(str(folder))["ecoli"], 5)
    st = states["ecoli"]
    assert st.isolates == want["isolates"]
    assert merge.CohortMerger.st_table(st) == orc.st_table_text(want)
    assert merge.CohortMerger.report(st) == orc.report_text(want)
    assert {s: c for c, _a, s in st.isolates}["a"] == 390


# ---------------------------------------------------------------------------------------------------------------- exact match
def _exact_queries(rows, rng, n_rand=1200):
    """Exact rows and duplicates, prefixes, extensions, one substitution, flagged copies (equal and off by one byte), upper-cased
    lower-case rows, empty queries and queries longer than every row."""
    seqs = [s for _g, _v, s in rows]
    qs = [rng.choice(seqs) for _ in range(n_rand)]
    qs += qs[:200]
    for _ in range(300):
        s = rng.choice(seqs)
        qs.append(s[:-rng.randint(1, 30)])
        qs.append(s + "ACGT"[:rng.randint(1, 4)])
        p = rng.randrange(len(s))
        qs.append(s[:p] + _sub(rng, s[p].upper()) + s[p + 1:])
    flagged = [s for s in seqs if any(c not in "ACGT" for c in s)]
    for s in flagged:
        qs.append(s)
        p = rng.randrange(len(s))
        qs.append(s[:p] + ("N" if s[p] != "N" else "A") + s[p + 1:])
        qs.append(s.upper())
    qs += [""] * 5 + ["A" * 1100, seqs[0] + "C" * 800]
    rng.shuffle(qs)
    return qs


def _check_exact(idx, qs, ranges, ref_of_range):
    got = idx.exact_first(qs, ranges)
    got_gv = [None if int(r) == NO else (idx.rows[int(r)][1], idx.rows[int(r)][2]) for r in got]
    want = [ref_of_range[rg].get(q) if q else None for q, rg in zip(qs, ranges)]
    assert _first_diff(got_gv, want, "query") is None, _first_diff(got_gv, want, "query")
    return sum(w is not None for w in want)


def _first_row(rows):
    out = {}
    for g, v, s in rows:
        out.setdefault(s, (g, v))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("org", ORGS)
def test_exact_match_organism_and_locus_ranges(scale, ctx, org):
    """More than kStageQ = 64 queries in one block of exact_clean_kernel (the whole organism, thousands of queries); row_key differs
    from resident order (hazard rows appended later, interleaved by gene; one sequence under several genes), so the first row in
    table order must win.  Verbatim sequenceLocate SQL on 300 queries, every hazard among them."""
    conn = sqlite3.connect(scale.path)
    rng = random.Random(11)
    idx = api.HammingIndex.from_sqlite(ctx, conn, org)
    assert idx.W == PLANE_W[org] and idx.n_flagged_rows > 100
    rows = scale.rows[org]
    qs = _exact_queries(rows, rng)
    orng = idx.organism_range(org)
    assert _check_exact(idx, qs, [orng] * len(qs), {orng: _first_row(rows)}) > 1500
    # per-locus ranges: each query asks the locus of a random gene
    genes = [g for g, _l in synth.SCHEMES[org]]
    ranges = [idx.block[(org, rng.choice(genes))] for _ in qs]
    refs = {idx.block[(org, g)]: _first_row([r for r in rows if r[0] == g]) for g in genes}
    assert _check_exact(idx, qs, ranges, refs) > 100
    # the reference's own statement
    hz = [s for _g, o, _v, s in scale.hazards if o == org]
    sub = hz + rng.sample(qs, 300 - len(hz) if len(hz) < 300 else 0)
    got = idx.exact_first(sub, [orng] * len(sub))
    for q, r in zip(sub, got):
        row = conn.execute("SELECT alleleVariant FROM alleles WHERE sequence = ? AND bacterium = ?", (str(q), org)).fetchone()
        want = None if (row is None or q == "") else str(row[0])
        assert (None if int(r) == NO else str(idx.rows[int(r)][2])) == want, (q[:30], len(q))
    conn.close()


@pytest.mark.gpu
def test_exact_match_second_organism_starts_mid_tile(scale, ctx):
    """A two-organism index: the second organism's range does not start on a 32-row tile, so exact_clean_kernel aligns its first CTA
    down to the tile and needs the extra slack CTA (gx = ... + 1) to reach the range's end; per-locus ranges start mid-tile too."""
    conn = sqlite3.connect(scale.path)
    rng = random.Random(12)
    idx = api.HammingIndex.from_sqlite(ctx, conn)
    assert idx.W == 24
    kp = idx.organism_range("kpneumoniae")
    assert kp[0] % 32 != 0
    qs, ranges, refs = [], [], {}
    for o in ORGS:
        rows = scale.rows[o]
        q = _exact_queries(rows, rng, 800)
        orng = idx.organism_range(o)
        refs[orng] = _first_row(rows)
        for g, _l in synth.SCHEMES[o]:
            refs[idx.block[(o, g)]] = _first_row([r for r in rows if r[0] == g])
        genes = [g for g, _l in synth.SCHEMES[o]]
        for s in q:
            qs.append(s)
            ranges.append(orng if rng.random() < 0.5 else idx.block[(o, rng.choice(genes))])
    assert sum(1 for (lo, _hi) in set(ranges) if lo % 32) >= 8
    assert _check_exact(idx, qs, ranges, refs) > 1500
    conn.close()


@pytest.mark.gpu
def test_exact_match_more_than_65535_blocks(scale, ctx):
    """More than 65535 distinct ranges of 1-4 rows in one call: more blocks than gridDim.y holds (65535), so mmlst_exact_match sends
    them in slices.  Some ranges cross a (organism, gene) boundary, where the row of lowest table position is not the first row."""
    conn = sqlite3.connect(scale.path)
    idx = api.HammingIndex.from_sqlite(ctx, conn)
    n = len(idx.rows)
    qs, ranges, want = [], [], []
    for i in range(80000):
        r = (i // 4 * 7919) % n
        hi = min(n, r + 1 + i % 4)
        s = idx.rows[(r + i % 5) % n][3]
        hit = [x for x in range(r, hi) if idx.rows[x][3] == s]
        qs.append(s)
        ranges.append((r, hi))
        want.append(min(hit, key=lambda x: idx.table_pos[x]) if hit else NO)
    assert len(set(ranges)) > 65535
    got = [int(x) for x in idx.exact_first(qs, ranges)]
    assert _first_diff(got, want, "query") is None, _first_diff(got, want, "query")
    assert 30000 < sum(w != NO for w in want) < 50000
    conn.close()


# ---------------------------------------------------------------------------------------------------------------- closest allele
COUNTS = (1, 63, 64, 65, 129, 2047, 2048, 2049, 4161)


def _mutant(rng, s, W32, p_flag=0.15):
    """0-12 substitutions, shortened or lengthened ends (now and then past W*32), a shifted start, and flagged letters."""
    b = list(s)
    for p in rng.sample(range(len(b)), rng.randint(0, 12)):
        b[p] = _sub(rng, b[p].upper())
    e = rng.random()
    if e < 0.2:
        b = b[:len(b) - rng.randint(1, 60)]
    elif e < 0.35:
        b += [rng.choice("ACGT") for _ in range(rng.randint(1, 40))]
    elif e < 0.4:
        b = b[rng.randint(1, 4):]
    elif e < 0.42:
        b += ["A"] * (W32 + 7 - len(b))
    f = rng.random()
    if f < p_flag * 0.5:
        b[rng.randrange(len(b))] = "N"
    elif f < p_flag * 0.8:
        b[rng.randrange(len(b))] = rng.choice(IUPAC)
    elif f < p_flag:
        p = rng.randrange(len(b))
        b[p:p + 15] = [c.lower() for c in b[p:p + 15]]
    return "".join(b)


def _check_search(idx, qs, ranges):
    d, a = idx.search(qs, ranges)
    flat = np.frombuffer(b"".join(r[3].encode("latin-1") for r in idx.rows), np.uint8)
    off = np.zeros(len(idx.rows) + 1, np.int64)
    off[1:] = np.cumsum([len(r[3]) for r in idx.rows])
    wd, wa = corc.hamming_min([q.encode("latin-1") for q in qs], flat, off, ranges)
    got = list(zip(d.tolist(), a.tolist()))
    want = list(zip(wd.tolist(), wa.tolist()))
    assert _first_diff(got, want, "query") is None, _first_diff(got, want, "query")
    return wd


@pytest.mark.gpu
@pytest.mark.parametrize("org", ORGS)
def test_closest_allele_query_chunks_and_splits(scale, ctx, org):
    """One call whose per-locus blocks hold 1, 63, 64, 65, 129, 2047, 2048, 2049 and 4161 queries, at 24- and 16-word planes: more
    than kQChunk = 64 queries go through the cp.async double buffer, an odd last chunk gets the phantom partner (65, 129, 2047, 2049,
    4161), and more than kQSplit = 2048 queries on one locus split over gridDim.z (2049: two slices, 4161: three).  The largest
    counts go to the smallest loci; two blocks are sub-ranges that start mid-tile."""
    conn = sqlite3.connect(scale.path)
    rng = random.Random(13)
    idx = api.HammingIndex.from_sqlite(ctx, conn, org)
    assert idx.W == PLANE_W[org]
    loci = sorted(((b[1] - b[0], g) for (o, g), b in idx.block.items() if o == org))
    qs, ranges = [], []
    for j, c in enumerate(sorted(COUNTS, reverse=True)):
        lo, hi = idx.block[(org, loci[j % len(loci)][1])]
        if j >= len(loci):
            lo, hi = lo + 13, hi - 5
        for _ in range(c):
            qs.append(_mutant(rng, idx.rows[rng.randrange(lo, hi)][3], idx.W * 32))
            ranges.append((lo, hi))
    qs[0], qs[1] = "", "N" * 40
    wd = _check_search(idx, qs, ranges)
    assert sum(ranges.count(r) for r in set(ranges) if ranges.count(r) > 2048) >= 2049 + 4161
    assert (wd == 0).sum() > 100 and (wd > 12).sum() > 100 and (wd <= 5).sum() > 1000
    conn.close()


@pytest.mark.gpu
def test_closest_allele_more_than_65535_blocks(scale, ctx):
    """More than 65535 distinct row ranges in one call: mmlst_hamming_min_x and mmlst_hamming_min_dev2 send them in slices of
    gridDim.y = 65535, and the flagged-sequence kernels take the same slices.  Two-organism index, ranges of 1-4 rows anywhere."""
    conn = sqlite3.connect(scale.path)
    rng = random.Random(14)
    idx = api.HammingIndex.from_sqlite(ctx, conn)
    n = len(idx.rows)
    qs, ranges = [], []
    for i in range(80000):
        r = (i // 4 * 7919) % n
        hi = min(n, r + 1 + i % 4)
        qs.append(_mutant(rng, idx.rows[rng.randrange(r, hi)][3], idx.W * 32, p_flag=0.01))
        ranges.append((r, hi))
    assert len(set(ranges)) > 65535
    _check_search(idx, qs, ranges)
    conn.close()


@pytest.mark.gpu
def test_closest_allele_empty_row_ranges(scale, ctx):
    """Calls whose every block has an empty row range answer "no row" (0xFFFFFFFF, 0xFFFFFFFF), at both plane widths and for the
    tiled kernel's grid (sized from the largest block: 0 rows) as well as for the flagged paths; and so does exact_first."""
    conn = sqlite3.connect(scale.path)
    for org in ORGS:
        idx = api.HammingIndex.from_sqlite(ctx, conn, org)
        s = idx.rows[5][3]
        qs = [s, s[:100] + "N" + s[101:], "", s.lower()]
        for ranges in ([(7, 7)] * 4, [(7, 7), (7, 7), (40, 40), (len(idx.rows), len(idx.rows))]):
            d, a = idx.search(qs, ranges)
            assert d.tolist() == [NO] * 4 and a.tolist() == [NO] * 4, (org, ranges)
            assert idx.exact_first(qs, ranges).tolist() == [NO] * 4
        # an empty block next to a full one: the full one still answers
        d, a = idx.search([s, s], [(3, 3), (5, 6)])
        assert d.tolist() == [NO, 0] and a.tolist() == [NO, 5]
    conn.close()


# ---------------------------------------------------------------------------------------------------------------- ST assignment
def _profile_lists(scale, conn, rng):
    lists = []
    genes = {o: [g for g, _l in synth.SCHEMES[o]] for o in ORGS}
    for o in ORGS:
        p = scale.db.profiles[o]
        lab = lambda g, v: "%s_%s_%d" % (o, g, int(v))
        other = ORGS[1 - ORGS.index(o)]
        for _ in range(1500):
            labels = [lab(g, v) for g, v in zip(genes[o], p[rng.randrange(p.shape[0])])]
            k = rng.random()
            if k < 0.25:
                labels[rng.randrange(7)] = lab(rng.choice(genes[o]), rng.randint(1, 800))        # near miss
            elif k < 0.32:
                labels.insert(rng.randint(1, 6), "%s_nogene_1" % o)                               # unknown in the middle
            elif k < 0.38:
                labels[-1] = "%s_%s_99999" % (o, genes[o][-1])                                    # unknown last: [(0, 0)]
            elif k < 0.44:
                labels.insert(rng.randint(0, 7), labels[rng.randrange(7)])                        # a label twice
            elif k < 0.5:
                labels[rng.randrange(7)] = "%s_%s_%d" % (other, genes[other][rng.randrange(7)], rng.randint(1, 800))   # another organism
            lists.append(labels)
        sh = [scale.shared[(o, n)] for n in SHARED_N]
        pair = scale.shared[(o, "pair")]
        for s in sh:                                                                              # 1 .. 1100 ties at 100 %
            lists += [[s], [s, s], [s, "%s_nogene_1" % o], ["%s_nogene_1" % o, s], [s, "%s_nogene_1" % o, s]]
        lists += [pair, pair[::-1], pair + [pair[0]]]                                             # 700 ties
        for _ in range(100):                                                                      # partial lists of 1-4 labels
            n = rng.randint(1, 4)
            labels = rng.sample(sh + [pair[1]], min(n, 2)) + [lab(g, rng.randint(1, 30)) for g in rng.sample(genes[o][1:], n - min(n, 2))]
            rng.shuffle(labels)
            lists.append(labels)
    lists.append(["ecoli_adk_1", "kpneumoniae_gapA_1"])
    return lists


@pytest.mark.gpu
def test_define_profiles_ties_past_256_and_more_than_32768_lists(scale, ctx):
    """Thousands of lists, then the same lists repeated past 32768 in one call (mmlst_st_match cuts them in chunks of 32768).
    Ties of 64, 65, 255, 256, 257, 700 and 1100 profiles: more than max_out = 64 tied profiles make define_profiles retry with room
    for all of them (api.py), and more than 256 ties (st_emit_kernel's blockDim) carry s_base across its loop iterations.  The
    reference is an inverted-index count on every list; the verbatim defineProfile SQL checks every distinct tie-heavy list and 150 more."""
    conn = sqlite3.connect(scale.path)
    rng = random.Random(15)
    pidx = api.ProfileIndex(ctx, conn)
    ref = define_profile_ref(conn)
    lists = _profile_lists(scale, conn, rng)
    want = [ref(l) for l in lists]
    got = pidx.define_profiles(lists)
    assert _first_diff(got, want, "list") is None, _first_diff(got, want, "list")
    n_ties = Counter(len(w) for w in want if w and w[0][1] == 100)
    for n in SHARED_N[1:] + (PAIR_N,):
        assert n_ties[n] >= 2, n
    assert any(w == [(0, 0)] for w in want) and any(w == [] or (w and w[0][1] < 100) for w in want)
    # the reference's statement on every tie-heavy list and a random sample
    sub = {tuple(lists[i]): want[i] for i in [i for i, w in enumerate(want) if len(w) > 64] + rng.sample(range(len(lists)), 150)}
    for labels, w in sub.items():
        assert api.define_profile(conn, list(labels)) == w, labels
    many = lists * (32768 // len(lists) + 2)
    assert len(many) > 32768
    order = list(range(len(many)))
    rng.shuffle(order)
    many = [many[i] for i in order]
    got = pidx.define_profiles(many)
    wmany = [want[i % len(lists)] for i in order]
    assert _first_diff(got, wmany, "list") is None, _first_diff(got, wmany, "list")
    conn.close()


# ---------------------------------------------------------------------------------------------------------------- merge
def _write_cohort(scale, folder, rng, n_samples=700):
    """Full lines of DB alleles (empty or exact sequences), partial lines on the shared alleles, and lines with novel sequences whose
    distances straddle z = 5 (1-12 substitutions, some with N / IUPAC letters, some recurring), plus hazard sequences."""
    genes = {o: [g for g, _l in synth.SCHEMES[o]] for o in ORGS}
    by_gene = {o: defaultdict(list) for o in ORGS}
    seq_of = {}
    for o in ORGS:
        for g, v, s in scale.rows[o]:
            by_gene[o][g].append((v, s))
            seq_of[(o, g, v)] = s
    hazards = defaultdict(list)
    for g, o, _v, s in scale.hazards:
        hazards[(o, g)].append(s)
    pool = {o: defaultdict(list) for o in ORGS}

    def item(o, g, v, s):
        return "%s_%s_%s::%s::%.1f::%.2f" % (o, g, v, s, rng.uniform(90, 100), rng.uniform(0, 3))

    def novel(o, g):
        if pool[o][g] and rng.random() < 0.3:
            return rng.choice(pool[o][g])
        b = list(rng.choice(by_gene[o][g])[1].upper())
        for p in rng.sample(range(len(b)), rng.choice((1, 2, 4, 5, 5, 6, 6, 8, 12))):
            b[p] = _sub(rng, b[p])
        if rng.random() < 0.15:
            b[rng.randrange(len(b))] = rng.choice("N" + IUPAC)
        s = "".join(b)
        pool[o][g].append(s)
        return s

    def line(o, smp):
        p = scale.db.profiles[o]
        k = rng.random()
        if k < 0.25:                                       # partial line on shared alleles
            labs = rng.sample([scale.shared[(o, n)] for n in SHARED_N] + [scale.shared[(o, "pair")][1]], rng.randint(1, 3))
            items = [item(o, l.split("_")[1], l.split("_")[2], "") for l in labs]
        else:
            st = p[rng.randrange(p.shape[0])]
            items = []
            n_new = 0 if k < 0.55 else rng.randint(1, 3)
            new = set(rng.sample(genes[o], n_new))
            for g, v in zip(genes[o], st):
                if g in new:
                    items.append(item(o, g, v, novel(o, g)))
                elif rng.random() < 0.5:
                    items.append(item(o, g, v, ""))
                else:
                    s = rng.choice(hazards[(o, g)]) if rng.random() < 0.1 else seq_of[(o, g, int(v))]
                    items.append(item(o, g, v, s))
        return "%s\t%s\t%s\r\n" % (o, smp, "\t".join(items))

    for i in range(n_samples):
        smp = "s%04d" % i + (".fna" if i % 50 == 0 else "")
        orgs = ORGS if i % 9 == 0 else (ORGS[i % 2],)
        with open(os.path.join(folder, "s%04d.nfo" % i), "w", newline="") as fh:
            fh.write("".join(line(o, smp) for o in orgs))


def _same_state(a, b):
    assert a.isolates == b.isolates
    assert a.new_profiles == b.new_profiles
    assert a.old_profiles == b.old_profiles
    assert a.new_sequences == b.new_sequences
    assert merge.CohortMerger.st_table(a) == merge.CohortMerger.st_table(b)
    assert merge.CohortMerger.report(a) == merge.CohortMerger.report(b)


@pytest.mark.gpu
def test_merge_cohort_gpu_equals_cpu_path_and_oracle(scale, ctx, tmp_path):
    """700 samples through merge_folder on the GPU (exact match, closest allele and ST assignment on the device) and on the CPU path
    (exact_table, defineProfile SQL, stringDiff from the C oracle): identical ST tables, reports, isolates, new profiles and new
    sequences; the oracle's merge_bacterium agrees on the first 80 files."""
    rng = random.Random(16)
    folder = tmp_path / "nfo"
    folder.mkdir()
    _write_cohort(scale, str(folder), rng)
    closest = corc_closest(scale.path)
    gpu, gscreen = merge.merge_folder(str(folder), scale.path, ctx=ctx)
    cpu, cscreen = merge.merge_folder(str(folder), scale.path, closest=closest, write=False)
    assert gscreen == cscreen
    for o in ORGS:
        _same_state(gpu[o], cpu[o])
        assert open(folder / "merged" / ("%s_ST.txt" % o), newline="").read() == merge.CohortMerger.st_table(cpu[o])
        cats = Counter(c for prof, _h, c in gpu[o].new_profiles.values())
        assert cats[1] > 10 and cats[2] > 5 and cats[3] > 10, cats
        assert gpu[o].n_searched > 100
        assert sum(1 for code, _a, _s in gpu[o].isolates if code <= N_PROFILES) > 100
    sub = tmp_path / "sub"
    sub.mkdir()
    for f in sorted(os.listdir(folder))[:80]:
        if f.endswith(".nfo"):
            shutil.copy(folder / f, sub / f)
    gsub = merge.merge_folder(str(sub), scale.path, ctx=ctx, write=False)[0]
    odb = orc.OracleDB(scale.path)
    cl = lambda b, g, s: (closest(b, [(g, s)])[0], None)
    for o, recs in orc.parse_nfo_folder(str(sub)).items():
        want = orc.merge_bacterium(odb, o, recs, 5, closest=cl)
        assert gsub[o].isolates == want["isolates"]
        assert gsub[o].new_profiles == want["encounteredProfiles"]
        assert merge.CohortMerger.st_table(gsub[o]) == orc.st_table_text(want)
        assert merge.CohortMerger.report(gsub[o]) == orc.report_text(want)
